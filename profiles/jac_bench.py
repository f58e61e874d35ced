#!/usr/bin/env python
"""Cost of the per-ray Jacobian next to the forward and to the one-VJP-per-source route
(DESIGN.md section 12), on the shapes of grad_bench.py.

    python profiles/jac_bench.py --out profiles/jac_bench_b200.json [--reps N] [--vjp-reps N]

For config 2 (1M models x 10 interfaces x 64 sources), the config-3 shape (4096 trans-dimensional
states, k = 1..30, 256 sources, kmode) and the config-5 slice (16384 models x 50 interfaces x 1024
near-critical sources), all from the seeds bench.py uses (raytracerfortran_b200.workloads):
  forward_ms      dff_batch_device with timeP and p, what the Jacobian needs
  jac_ms          dff_jac_device, the Jacobian kernel alone, with dT/dR and dT/dd
  jac_bytes       what that kernel writes, from the shapes: B NSrc (ldv + ldz + 2) 8
  write_bound_ms  jac_bytes over the data sheet's 7.7 TB/s; write_bound_fraction = it / jac_ms
  vjp_route_ms    the route without this kernel: NSrc launches of dff_grad_device, each with a
                  one-hot weight buffer refilled in place and its rows written to their slice of
                  an [NSrc, B, ldv] / [NSrc, B, ldz] result
Each figure is the median of N passes timed with CUDA events after a warm-up; before every timed
pass a 256 MB buffer is overwritten, so no pass finds its inputs in the 126 MB L2.  The VJP route
on the config-5 slice (1024 launches a pass) takes --vjp-reps passes.  The card's name and power
limit are read in the same run.  Each invocation appends one run to --out.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--vjp-reps", type=int, default=3, help="passes of the VJP route on the config-5 slice")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("jac_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(32 << 20, dtype=torch.float64, device=dev)       # 256 MB
    run = {"card": card(), "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "shapes": {}}
    for name, s in shapes():
        t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
        v, z, n, so, sd = t(s["v"]), t(s["z"]), t(s["n"], torch.int32), t(s["so"]), t(s["sd"])
        B, S, ldv, ldz = v.shape[0], so.numel(), v.shape[1], z.shape[1]
        km = s["kmode"]
        fw = device.dff_batch_device(v, z, n, so, sd, want_times=True, want_p=True, kmode=km)
        J = device.dff_jac_device(v, z, n, so, sd, fw["timeP"], fw["p"], want_src=True, kmode=km)
        w = torch.zeros_like(fw["timeP"])
        gv = torch.empty((S, B, ldv), dtype=torch.float64, device=dev)
        gz = torch.empty((S, B, ldz), dtype=torch.float64, device=dev)

        def forward():
            device.dff_batch_device(v, z, n, so, sd, timeP=fw["timeP"], p_out=fw["p"], kmode=km)

        def jac():
            device.dff_jac_device(v, z, n, so, sd, fw["timeP"], fw["p"], jvels=J["jvels"], jdepths=J["jdepths"],
                                  dtdr=J["dtdr"], dtdd=J["dtdd"], kmode=km)

        def vjp_route():
            for k in range(S):
                w.zero_()
                w[:, k] = 1.0
                device.dff_grad_device(v, z, n, so, sd, fw["timeP"], fw["p"], w, gvels=gv[k], gdepths=gz[k],
                                       kmode=km)

        e = {"models": B, "sources": S, "ldv": ldv, "ldz": ldz, "kmode": km}
        e["forward"] = timed(forward, args.reps, flush)
        e["jac"] = timed(jac, args.reps, flush)
        e["jac_bytes"] = B * S * (ldv + ldz + 2) * 8
        e["write_bound_ms"] = e["jac_bytes"] / HBM_BYTES_PER_S * 1e3
        e["write_bound_fraction"] = e["write_bound_ms"] / e["jac"]["median_ms"]
        e["vjp_route"] = timed(vjp_route, args.vjp_reps if name == "config5_slice" else args.reps, flush)
        # the route gives the same rows: check them once
        torch.cuda.synchronize()
        e["vjp_route_rows_equal"] = bool(torch.equal(gv.transpose(0, 1), J["jvels"])
                                         and torch.equal(gz.transpose(0, 1), J["jdepths"]))
        e["vjp_route_over_jac"] = e["vjp_route"]["median_ms"] / e["jac"]["median_ms"]
        run["shapes"][name] = e
        print(name, json.dumps({k: (x["median_ms"] if isinstance(x, dict) else x) for k, x in e.items()}),
              flush=True)
        del fw, J, w, gv, gz, v, z
        torch.cuda.empty_cache()
    runs = json.load(open(args.out)) if os.path.exists(args.out) else []
    runs.append(run)
    with open(args.out, "w") as fh:
        json.dump(runs, fh, indent=1)


if __name__ == "__main__":
    main()
