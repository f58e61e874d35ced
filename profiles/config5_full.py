#!/usr/bin/env python
"""BASELINE.json config 5 at FULL size: 16M models x 50 interfaces x 1024 near-critical sources
(1.7e10 rays), generated on the device, logL fused (no travel-time store: that would be 131 GB).
On one GPU, or under torchrun with the model axis sharded over the ranks (no collective on the
data path; the timed region is bracketed by barriers and the time is the max over ranks):

    python profiles/config5_full.py [models] [--stable-norm]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port P profiles/config5_full.py

Checks on every rank: a sample of models re-evaluated alone gives the same bits (batch invariance)
and matches the CPU oracle bit for bit in travel time.  --stable-norm switches on the opt-in
overflow-free normaliser -(N/2) log(2 pi) (the reference's (2 pi)^(N/2) overflows for N >= 773 and
every logL is -inf, loglhood.f90:194; default: reproduce that)."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import oracle
    import raytracerfortran_b200 as rt
    from raytracerfortran_b200 import device, workloads

    import torch.distributed as dist
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    stable = "--stable-norm" in sys.argv
    B_all = int(args[0]) if args else 16_000_000
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ["RTB200_DEVICE"] = str(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lo_, hi_ = rt.shard_range(B_all, rank, world)
    B = hi_ - lo_
    if stable:
        rt.set_option("stable_lognorm", 1)
    L, S = 50, 1024
    g = torch.Generator(device=dev).manual_seed(5 + 1000 * rank)
    v = 1500.0 + 8500.0 * torch.rand((B, L + 1), dtype=torch.float64, device=dev, generator=g)
    z = torch.empty((B, L), dtype=torch.float64, device=dev)
    step = 2_000_000
    for lo in range(0, B, step):           # sort in slices to bound the temporary memory
        u = torch.rand((min(step, B - lo), L), dtype=torch.float64, device=dev, generator=g)
        z[lo:lo + step] = 50.0 + 9950.0 * torch.sort(u, dim=1).values
    nl = torch.full((B,), L, dtype=torch.int32, device=dev)
    so, sd = workloads.make_sources(S, 5, near_critical=True)
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ts, td = f(so), f(sd)
    tobs, sigma = f(np.full(S, 2.0)), torch.full((B,), 0.02, dtype=torch.float64, device=dev)
    ll = torch.empty(B, dtype=torch.float64, device=dev)
    device.dff_batch_device(v[:4096], z[:4096], nl[:4096], ts, td, tobs=tobs, sigma=sigma[:4096], logL=ll[:4096])   # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    device.dff_batch_device(v, z, nl, ts, td, tobs=tobs, sigma=sigma, logL=ll)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    # batch invariance + oracle on a sample (travel times of 12 models spread over the batch)
    pick = torch.linspace(0, B - 1, 12, device=dev).long()
    out = device.dff_batch_device(v[pick].contiguous(), z[pick].contiguous(), nl[pick].contiguous(),
                                  ts, td, tobs=tobs, sigma=sigma[pick].contiguous(), want_times=True)
    torch.cuda.synchronize()
    same_ll = bool(torch.equal(out["logL"], ll[pick]))
    ref = oracle.dff_batch(v[pick].cpu().numpy(), z[pick].cpu().numpy(), nl[pick].cpu().numpy(), so, sd)
    same_t = bool(np.array_equal(out["timeP"].cpu().numpy().view(np.uint64), ref["timeP"].view(np.uint64)))
    flags = torch.tensor([ms, float(same_ll), float(same_t), float(torch.isneginf(ll).all()),
                          float(torch.isfinite(ll).all())], dtype=torch.float64, device=dev)
    if world > 1:
        mx = flags.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        ms = float(mx[0])
    if rank == 0:
        print(json.dumps({"workload": f"config5 full: {B_all} models x {L} interfaces x {S} near-critical sources "
                                      f"on {world} GPU(s), model axis sharded",
                          "n_gpus": world, "rays": B_all * S, "seconds": ms / 1e3, "evals_per_s": B_all * S / (ms / 1e3),
                          "stable_lognorm": stable,
                          "logL_all_minus_inf_like_reference": bool(flags[3]), "logL_all_finite": bool(flags[4]),
                          "batch_invariant_logL": bool(flags[1]),
                          "sample_travel_times_bit_identical_to_oracle": bool(flags[2]),
                          "variant": int(rt.get_stat("variant")), "tile_models": int(rt.get_stat("tile_models")),
                          "grid": int(rt.get_stat("grid"))}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
