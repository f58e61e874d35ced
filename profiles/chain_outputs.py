#!/usr/bin/env python
"""Seeded chain states after the two config-4 sampler paths of config4_chains.py (8 replicas x 1024
chains, k ~ Poisson(3.01) in 1..30, 256 sources), for comparing two builds bit for bit:

    python profiles/chain_outputs.py OUT_DIR [--sweeps K]

writes OUT_DIR/graph.npz (McmcGraph: k, voro, logL, sigma, tally) and OUT_DIR/eager.npz
(bd_step_device + mh_moves_device: k, voro, logL, sigma, accepted moves per chain)."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--sweeps", type=int, default=5)
    args = ap.parse_args()
    import torch
    from raytracerfortran_b200 import chains, device, tempering, workloads

    B, ldk, nsrc, M = 8 * 1024, 30, 256, 20
    rng = np.random.default_rng(40)
    k = np.clip(rng.poisson(3.01, B), 1, ldk).astype(np.int32)
    voro = np.zeros((B, 2, ldk))
    for b in range(B):
        n = int(k[b])
        voro[b, 0, 1:n] = np.cumsum(100.1 + rng.random(n - 1) * (9000.0 / n))
        voro[b, 1, :n] = rng.uniform(1500.0, 10000.0, n)
    so, sd = workloads.make_sources(nsrc, 4)
    tobs, sigma = workloads.make_observations(np.full(nsrc, 1.3), B, 4)
    beta = np.repeat(tempering.temperature_ladder(8, 1.4), 1024)
    prior, sd_prior, pk = chains.prior_array(), chains.sd_prior_array(), chains.poisson_pk(3.01, 1, ldk)
    os.makedirs(args.out, exist_ok=True)
    for mode in ("graph", "eager"):
        f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        tk, tv, tg, tb, ts, td, to = f(k), f(voro), f(sigma), f(beta), f(so), f(sd), f(tobs)
        tl = device.dff_batch_device(tv[:, 1, :].contiguous(), tv[:, 0, 1:].contiguous(), tk, ts, td,
                                     tobs=to, sigma=tg, kmode=True)["logL"]
        if mode == "graph":
            g = chains.McmcGraph(tk, tv, tl, tg, tb, M, prior, sd_prior, pk, 1, ldk, ts, td, to, seed=2026)
            g.run(args.sweeps)
            counts = g.tally
        else:
            gen = torch.Generator(device="cuda").manual_seed(100)
            pos = torch.zeros(B, dtype=torch.int32, device="cuda")
            counts = torch.zeros(B, dtype=torch.int64, device="cuda")
            for _ in range(args.sweeps):
                u = torch.rand((5, B), dtype=torch.float64, device="cuda", generator=gen)
                idel = (2 + torch.floor(u[4] * (tk - 1).clamp(min=1))).to(torch.int32)
                chains.bd_step_device(tk, tv, tl, u[0].contiguous(), idel, u[1].contiguous(), u[2].contiguous(),
                                      u[3].contiguous(), tb, tg, prior, pk, 1, ldk, ts, td, to)
                counts += chains.mh_moves_device(tk, tv, tl, pos, M, tb, tg, prior, ts, td, to, generator=gen)
        torch.cuda.synchronize()
        np.savez(os.path.join(args.out, f"{mode}.npz"), k=tk.cpu().numpy(), voro=tv.cpu().numpy(),
                 logL=tl.cpu().numpy(), sigma=tg.cpu().numpy(), counts=counts.cpu().numpy())


if __name__ == "__main__":
    main()
