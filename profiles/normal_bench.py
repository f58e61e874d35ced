#!/usr/bin/env python
"""Cost of the per-model normal equations next to the forward and to the route through the stored
Jacobian (DESIGN.md section 13), on the shapes of grad_bench.py.

    python profiles/normal_bench.py --out profiles/normal_bench_b200.json [--reps N]

For config 2 (1M models x 10 interfaces x 64 sources), the config-3 shape (4096 trans-dimensional
states, k = 1..30, 256 sources, kmode) and the config-5 slice (16384 models x 50 interfaces x 1024
near-critical sources), all from the seeds bench.py uses (raytracerfortran_b200.workloads):
  forward_ms        dff_batch_device with timeP and p, what both routes need
  normal_ms         dff_normal_device with tobs: JtJ [B, P, P] and Jtr [B, P], P = ldv + ldz
  normal_bytes      what that kernel writes, from the shapes: B (P^2 + P) 8
  write_bound_ms    normal_bytes over the data sheet's 7.7 TB/s; write_bound_fraction = it / normal_ms
  jac_ms            dff_jac_device alone, writing the rows [B, NSrc, ldv] + [B, NSrc, ldz]
  jac_route_ms      dff_jac_device, then torch: J = [jvels | jdepths], J^T J and J^T r by bmm
  *_peak_bytes      torch.cuda.max_memory_allocated over one call of the route, inputs included
The route's JtJ / Jtr are checked once against the kernel's within the reordering bound
2 NSrc u (|J|^T |J|).  Each figure is the median of N passes timed with CUDA events after a
warm-up; before every timed pass a 256 MB buffer is overwritten, so no pass finds its inputs in
the 126 MB L2.  The card's name and power limit are read in the same run.  Each invocation appends
one run to --out.
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
from raytracerfortran_b200 import device  # noqa: E402

HBM_BYTES_PER_S = 7.7e12      # B200 data sheet
U = 2.0 ** -53


def peak(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("normal_bench needs a CUDA device")
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
        e = {"models": B, "sources": S, "ldv": ldv, "ldz": ldz, "kmode": km}

        def forward():
            device.dff_batch_device(v, z, n, so, sd, timeP=fw["timeP"], p_out=fw["p"], kmode=km)

        e["forward"] = timed(forward, args.reps, flush)

        # ---- the normal-equations kernel
        N = {}
        e["normal_peak_bytes"] = peak(lambda: N.update(device.dff_normal_device(
            v, z, n, so, sd, fw["timeP"], fw["p"], tobs=tobs, kmode=km)))

        def normal():
            device.dff_normal_device(v, z, n, so, sd, fw["timeP"], fw["p"], tobs=tobs, JtJ=N["JtJ"], Jtr=N["Jtr"],
                                     kmode=km)

        e["normal"] = timed(normal, args.reps, flush)
        e["normal_bytes"] = B * (P * P + P) * 8
        e["write_bound_ms"] = e["normal_bytes"] / HBM_BYTES_PER_S * 1e3
        e["write_bound_fraction"] = e["write_bound_ms"] / e["normal"]["median_ms"]
        JtJ, Jtr = N["JtJ"].clone(), N["Jtr"].clone()
        del N
        torch.cuda.empty_cache()

        # ---- the route through the stored Jacobian
        R = {}

        def jac_route():
            J = device.dff_jac_device(v, z, n, so, sd, fw["timeP"], fw["p"], kmode=km)
            Jc = torch.cat([J["jvels"], J["jdepths"]], 2)
            del J
            r = tobs[None, :] - fw["timeP"]
            R["JtJ"] = torch.bmm(Jc.transpose(1, 2), Jc)
            R["Jtr"] = torch.bmm(Jc.transpose(1, 2), r[:, :, None])[:, :, 0]
            R["J"] = Jc

        e["jac_route_peak_bytes"] = peak(jac_route)
        Jc = R.pop("J")
        Ja = Jc.abs()
        ok = (JtJ - R["JtJ"]).abs() <= 2 * S * U * torch.bmm(Ja.transpose(1, 2), Ja) + 1e-300
        ra = (tobs[None, :] - fw["timeP"]).abs()
        ok2 = (Jtr - R["Jtr"]).abs() <= 2 * (S + 1) * U * torch.bmm(Ja.transpose(1, 2), ra[:, :, None])[:, :, 0] + 1e-300
        e["jac_route_within_bound"] = bool(ok.all().item() and ok2.all().item())
        del Ja, ok, ok2, ra
        jv, jz = Jc[:, :, :ldv].contiguous(), Jc[:, :, ldv:].contiguous()
        del Jc
        R.clear()           # jac_route_timed fills it again: deleting the name would unbind jac_route's R
        torch.cuda.empty_cache()

        def jac():
            device.dff_jac_device(v, z, n, so, sd, fw["timeP"], fw["p"], jvels=jv, jdepths=jz, kmode=km)

        e["jac"] = timed(jac, args.reps, flush)
        del jv, jz
        torch.cuda.empty_cache()

        def jac_route_timed():
            jac_route()
            R.clear()

        e["jac_route"] = timed(jac_route_timed, args.reps, flush)
        e["jac_over_normal"] = e["jac"]["median_ms"] / e["normal"]["median_ms"]
        e["jac_route_over_normal"] = e["jac_route"]["median_ms"] / e["normal"]["median_ms"]
        run["shapes"][name] = e
        print(name, json.dumps({k: (x["median_ms"] if isinstance(x, dict) else x) for k, x in e.items()}),
              flush=True)
        del fw, JtJ, Jtr, v, z
        torch.cuda.empty_cache()
    runs = json.load(open(args.out)) if os.path.exists(args.out) else []
    runs.append(run)
    with open(args.out, "w") as fh:
        json.dump(runs, fh, indent=1)


if __name__ == "__main__":
    main()
