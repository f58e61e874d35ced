#!/usr/bin/env python
"""Cost of the travel-time gradient next to the forward on the bench.py shapes (DESIGN.md section 11).

    python profiles/grad_bench.py --out profiles/grad_bench_b200.json [--reps N]

For config 2 (1M models x 10 interfaces x 64 sources), the config-3 shape (4096 trans-dimensional
states, k = 1..30, 256 sources, kmode) and the config-5 slice (16384 models x 50 interfaces x 1024
near-critical sources), all from the seeds bench.py uses (raytracerfortran_b200.workloads):
  forward_ms    dff_batch_device with timeP and p, what the gradient needs
  grad_ms       dff_grad_device, the gradient kernel alone (with the per-ray dT/dR, dT/dd)
  loglhood_ms   grad.loglhood forward + backward (gradients for vels and depths)
Each figure is the median of N passes timed with CUDA events after a warm-up; before every timed
pass a 256 MB buffer is overwritten, so no pass finds its inputs in the 126 MB L2.  The card's name
and power limit are read in the same run.  Each invocation appends one run to --out.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracerfortran_b200 import device, grad, workloads  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, limit = (q[0].split(", ") + ["?"])[:2] if q else (torch.cuda.get_device_name(0), "unknown")
    return {"name": name, "power_limit": limit, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, reps, flush):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return {"median_ms": statistics.median(out), "min_ms": min(out), "max_ms": max(out), "reps": reps}


def shapes():
    c2, c3, c5 = (workloads.CONFIGS[k] for k in ("config2", "config3", "config5"))
    v, z, n = workloads.make_models(c2["B"], c2["nlayers"], c2["seed"])
    so, sd = workloads.make_sources(c2["nsrc"], c2["seed"])
    yield "config2", dict(v=v, z=z, n=n, so=so, sd=sd, kmode=False)
    k, vp, zi = workloads.make_transd_models(c3["B"], c3["kmax"], c3["seed"], uniform_k=True)
    so, sd = workloads.make_sources(c3["nsrc"], c3["seed"])
    yield "config3_uniform_k", dict(v=vp, z=zi, n=k, so=so, sd=sd, kmode=True)
    v, z, n = workloads.make_models(16384, c5["nlayers"], c5["seed"])
    so, sd = workloads.make_sources(c5["nsrc"], c5["seed"], near_critical=True)
    yield "config5_slice", dict(v=v, z=z, n=n, so=so, sd=sd, kmode=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("grad_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(32 << 20, dtype=torch.float64, device=dev)       # 256 MB
    run = {"card": card(), "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "shapes": {}}
    for name, s in shapes():
        t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
        v, z, n, so, sd = t(s["v"]), t(s["z"]), t(s["n"], torch.int32), t(s["so"]), t(s["sd"])
        B, S = v.shape[0], so.numel()
        fw = device.dff_batch_device(v, z, n, so, sd, want_times=True, want_p=True, kmode=s["kmode"])
        w = torch.ones_like(fw["timeP"])
        tobs = fw["timeP"][0].clone()
        sigma = torch.full((B,), 0.02, dtype=torch.float64, device=dev)
        vr, zr = v.clone().requires_grad_(True), z.clone().requires_grad_(True)

        def forward():
            device.dff_batch_device(v, z, n, so, sd, timeP=fw["timeP"], p_out=fw["p"], kmode=s["kmode"])

        def gradient():
            device.dff_grad_device(v, z, n, so, sd, fw["timeP"], fw["p"], w, want_src=True, kmode=s["kmode"])

        def loglhood():
            L = grad.loglhood(vr, zr, n, so, sd, tobs, sigma, kmode=s["kmode"])
            torch.autograd.grad(L.sum(), (vr, zr))

        e = {"models": B, "sources": S, "ldv": v.shape[1], "kmode": s["kmode"]}
        e["forward"] = timed(forward, args.reps, flush)
        e["grad"] = timed(gradient, args.reps, flush)
        e["loglhood_fwd_bwd"] = timed(loglhood, args.reps, flush)
        e["grad_over_forward"] = e["grad"]["median_ms"] / e["forward"]["median_ms"]
        run["shapes"][name] = e
        print(name, json.dumps({k: (x["median_ms"] if isinstance(x, dict) else x) for k, x in e.items()}),
              flush=True)
        del fw, w, v, z, vr, zr
        torch.cuda.empty_cache()
    runs = json.load(open(args.out)) if os.path.exists(args.out) else []
    runs.append(run)
    with open(args.out, "w") as fh:
        json.dump(runs, fh, indent=1)


if __name__ == "__main__":
    main()
