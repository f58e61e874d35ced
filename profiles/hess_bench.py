#!/usr/bin/env python
"""Cost of the per-model second derivatives next to the forward and the normal equations
(DESIGN.md section 14), on the shapes of grad_bench.py.

    python profiles/hess_bench.py --out profiles/hess_bench_b200.json [--reps N]

For config 2 (1M models x 10 interfaces x 64 sources), the config-3 shape (4096 trans-dimensional
states, k = 1..30, 256 sources, kmode) and the config-5 slice (16384 models x 50 interfaces x 1024
near-critical sources), all from the seeds bench.py uses (raytracerfortran_b200.workloads):
  forward_ms        dff_batch_device with timeP and p
  normal_ms         dff_normal_device with tobs: JtJ [B, P, P] and Jtr [B, P], P = ldv + ldz
  hess_ms           dff_hess_device with w = tobs - timeP: H [B, P, P]
  newton_ms         grad.newton_equations end to end: forward, both kernels, A = JtJ - H
  hess_bytes        what the Hessian kernel writes, from the shapes: B P^2 8
  write_bound_ms    hess_bytes over the data sheet's 7.7 TB/s
  hess_over_normal  hess_ms / normal_ms
  *_peak_bytes      torch.cuda.max_memory_allocated over one call, inputs included
Each figure is the median of N passes timed with CUDA events after a warm-up; before every timed
pass a 256 MB buffer is overwritten, so no pass finds its inputs in the 126 MB L2.  The card's
name and power limit are read in the same run.  Each invocation appends one run to --out.
"""
import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from grad_bench import card, shapes, timed  # noqa: E402
from normal_bench import HBM_BYTES_PER_S, peak  # noqa: E402
from raytracerfortran_b200 import device, grad  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("hess_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(32 << 20, dtype=torch.float64, device=dev)       # 256 MB
    run = {"card": card(), "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "shapes": {}}
    for name, s in shapes():
        t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
        v, z, n, so, sd = t(s["v"]), t(s["z"]), t(s["n"], torch.int32), t(s["so"]), t(s["sd"])
        B, S, ldv, ldz = v.shape[0], so.numel(), v.shape[1], z.shape[1]
        P = ldv + ldz
        km = s["kmode"]
        fw = device.dff_batch_device(v, z, n, so, sd, want_times=True, want_p=True, kmode=km)
        tobs = fw["timeP"][0].clone()
        tobs += 0.01
        w = (tobs[None, :] - fw["timeP"]).contiguous()
        e = {"models": B, "sources": S, "ldv": ldv, "ldz": ldz, "kmode": km}

        def forward():
            device.dff_batch_device(v, z, n, so, sd, timeP=fw["timeP"], p_out=fw["p"], kmode=km)

        e["forward"] = timed(forward, args.reps, flush)

        N = {}
        e["normal_peak_bytes"] = peak(lambda: N.update(device.dff_normal_device(
            v, z, n, so, sd, fw["timeP"], fw["p"], tobs=tobs, kmode=km)))

        def normal():
            device.dff_normal_device(v, z, n, so, sd, fw["timeP"], fw["p"], tobs=tobs, JtJ=N["JtJ"], Jtr=N["Jtr"],
                                     kmode=km)

        e["normal"] = timed(normal, args.reps, flush)
        del N
        torch.cuda.empty_cache()

        Hd = {}
        e["hess_peak_bytes"] = peak(lambda: Hd.update(device.dff_hess_device(
            v, z, n, so, sd, fw["timeP"], fw["p"], w, kmode=km)))

        def hess():
            device.dff_hess_device(v, z, n, so, sd, fw["timeP"], fw["p"], w, H=Hd["H"], kmode=km)

        e["hess"] = timed(hess, args.reps, flush)
        e["hess_symmetric"] = bool(torch.equal(Hd["H"], Hd["H"].transpose(1, 2)))
        del Hd
        torch.cuda.empty_cache()
        e["hess_bytes"] = B * P * P * 8
        e["write_bound_ms"] = e["hess_bytes"] / HBM_BYTES_PER_S * 1e3
        e["hess_over_normal"] = e["hess"]["median_ms"] / e["normal"]["median_ms"]

        def newton():
            grad.newton_equations(v, z, n, so, sd, tobs, kmode=km)

        e["newton_peak_bytes"] = peak(newton)
        e["newton"] = timed(newton, args.reps, flush)
        run["shapes"][name] = e
        print(name, json.dumps({k: (x["median_ms"] if isinstance(x, dict) else x) for k, x in e.items()}),
              flush=True)
        del fw, w, v, z
        torch.cuda.empty_cache()
    runs = json.load(open(args.out)) if os.path.exists(args.out) else []
    runs.append(run)
    with open(args.out, "w") as fh:
        json.dump(runs, fh, indent=1)


if __name__ == "__main__":
    main()
