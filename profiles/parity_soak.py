#!/usr/bin/env python
"""Parity soak: random batches of every kind of shape the tests use (1-50 interfaces, ordinary and
near-critical sources, ragged layer counts, trans-dimensional k-mode states), travel times and ray
parameters compared bit for bit with the CPU oracle for as long as --seconds allows.  The oracle is
the slow side (all host cores)."""
import argparse, json, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import workloads

ap = argparse.ArgumentParser()
ap.add_argument("--seconds", type=float, default=120.0)
ap.add_argument("--seed", type=int, default=2026)
args = ap.parse_args()
rng = np.random.default_rng(args.seed)
t0 = time.time()
rays = mism = batches = 0
kinds = {}
while time.time() - t0 < args.seconds:
    kind = ["shallow", "deep-critical", "ragged", "kmode", "one-model"][batches % 5]
    # the batches rotate over the default choice (variant 1, 3 or 5 by shape), variant 5 (one list
    # segment per warp), variant 3 (the deep-model kernel, on every depth) and variant 1; a kind of
    # its own for the one-model latency kernel
    rt.set_option("variant", [-1, 5, 3, 1][batches % 4])
    seed = int(rng.integers(1, 2**31))
    if kind == "shallow":
        L, S, B = int(rng.integers(1, 13)), int(rng.integers(8, 129)), 60000
        v, z, nl = workloads.make_models(B, L, seed)
        so, sd = workloads.make_sources(S, seed)
    elif kind == "deep-critical":
        L, S, B = int(rng.integers(20, 51)), int(rng.integers(64, 300)), 1500
        v, z, nl = workloads.make_models(B, L, seed, min_thickness=False)
        so, sd = workloads.make_sources(S, seed, near_critical=True)
    elif kind == "ragged":
        L, S, B = int(rng.integers(2, 30)), int(rng.integers(1, 200)), 20000
        v, z, nl = workloads.make_models(B, L, seed)
        nl = rng.integers(0, L + 1, B).astype(np.int32)
        so, sd = workloads.make_sources(S, seed, near_critical=bool(seed & 1))
    elif kind == "one-model":
        rt.set_option("variant", -1)
        bad = n = 0
        for _ in range(200):
            L, S = int(rng.integers(0, 60)), int(rng.integers(1, 400))
            v, z, nl = workloads.make_models(1, max(L, 1), int(rng.integers(1, 2**31)), min_thickness=L < 40)
            nl[:] = L
            so, sd = workloads.make_sources(S, int(rng.integers(1, 2**31)), near_critical=bool(L & 1))
            ref = oracle.dff_batch(v, z, nl, so, sd, want_p=True)
            got = rt.dff_batch(v, z, nl, so, sd, want_p=True)
            assert rt.get_stat("variant") == 9
            bad += int((got["timeP"].view(np.uint64) != ref["timeP"].view(np.uint64)).sum()) \
                + int((got["p"].view(np.uint64) != ref["p"].view(np.uint64)).sum())
            n += S
        rays += n; mism += bad; batches += 1
        kinds[kind] = kinds.get(kind, 0) + n
        continue
    else:
        S, B = int(rng.integers(16, 257)), 30000
        k, vp, zi = workloads.make_transd_models(B, 30, seed)
        so, sd = workloads.make_sources(S, seed)
        tobs, sigma = workloads.make_observations(np.full(S, 1.3), B, seed)
        ll, pred = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma, want_pred=True)
        nlr = np.where(k > 1, k - 1, 1).astype(np.int32)
        vv, zz = vp.copy(), np.zeros((B, 29))
        zz[:, :] = zi[:, :29]
        one = k <= 1
        vv[one, 1] = vv[one, 0]
        zz[one, 0] = 9999.9
        ref = oracle.dff_batch(vv, zz, nlr, so, sd)
        bad = int((pred.view(np.uint64) != ref["timeP"].view(np.uint64)).sum())
        rays += B * S; mism += bad; batches += 1
        tag = kind + " (variant %d)" % int(rt.get_stat("variant"))
        kinds[tag] = kinds.get(tag, 0) + B * S
        continue
    ref = oracle.dff_batch(v, z, nl, so, sd, want_p=True)
    got = rt.dff_batch(v, z, nl, so, sd, want_p=True)
    bad = int((got["timeP"].view(np.uint64) != ref["timeP"].view(np.uint64)).sum()) \
        + int((got["p"].view(np.uint64) != ref["p"].view(np.uint64)).sum())
    rays += B * S; mism += bad; batches += 1
    tag = kind + " (variant %d)" % int(rt.get_stat("variant"))
    kinds[tag] = kinds.get(tag, 0) + B * S
print(json.dumps({"seconds": time.time() - t0, "batches": batches, "rays_compared": rays,
                  "bit_mismatches": mism, "rays_by_kind": kinds, "seed": args.seed}))
