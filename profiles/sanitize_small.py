#!/usr/bin/env python
"""A small pass through every kernel the library has, sized for compute-sanitizer
(memcheck / racecheck): batch kernel variants 1, 3, 5 (incl. a tile with an insane model), the
one-model latency kernel, the chain moves, the whole-iteration graph, the swap kernels, the pinned
ring.  Results are checked against the oracle so a clean sanitizer run is also a correct run."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import chains, tempering, workloads

def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    nan = np.isnan(b)
    return np.array_equal(np.isnan(a), nan) and np.array_equal(a[~nan].view(np.uint64), b[~nan].view(np.uint64))

B, S = 300, 40
v, z, nl = workloads.make_models(B, 10, 1)
so, sd = workloads.make_sources(S, 1)
v[7, 2] = np.nan                     # one insane model: its rays take the built-in sqrt / divide
tobs, sigma = workloads.make_observations(np.ones(S), B, 1)
with np.errstate(all="ignore"):
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
for variant in (1, 5):
    rt.set_option("variant", variant)
    got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    assert same(got["timeP"], ref["timeP"]) and same(got["p"], ref["p"]), variant
rt.set_option("variant", -1)
rt.set_option("stage_pageable", 1); rt.set_option("chunk_models", 64)
got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
assert same(got["timeP"], ref["timeP"])
rt.set_option("stage_pageable", -1); rt.set_option("chunk_models", 0)
vd, zd, nld = workloads.make_models(24, 50, 2, min_thickness=False)
sod, sdd = workloads.make_sources(70, 2, near_critical=True)
assert same(rt.dff_batch(vd, zd, nld, sod, sdd)["timeP"], oracle.dff_batch(vd, zd, nld, sod, sdd)["timeP"])   # variant 3
t1 = rt.dff(v[0], z[0], so, sd)                                                                      # latency kernel
assert same(t1, ref["timeP"][0])
# chains: one move of each kind, then one iteration of the graph, then a swap round
dev = torch.device("cuda", 0)
f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
Bc, ldk = 256, 8
rng = np.random.default_rng(3)
k = rng.integers(1, ldk + 1, Bc).astype(np.int32)
voro = np.zeros((Bc, 2, ldk))
for b in range(Bc):
    n = int(k[b])
    voro[b, 0, 1:n] = np.cumsum(150.0 + rng.random(n - 1) * 900.0)
    voro[b, 1, :n] = rng.uniform(1500.0, 10000.0, n)
tobs2, sig2 = workloads.make_observations(np.full(S, 1.3), Bc, 3)
ll = np.array([oracle.loglhood_rt(voro[b, 1, :k[b]], voro[b, 0, 1:k[b]], so, sd, tobs2, sig2[b])[0] for b in range(Bc)])
beta = 1.0 / 1.3 ** rng.integers(0, 5, Bc)
tk, tv, tl, tg, tb, ts, td, to = f(k), f(voro), f(ll), f(sig2), f(beta), f(so), f(sd), f(tobs2)
prior, sdp, pk = chains.prior_array(), chains.sd_prior_array(), chains.poisson_pk(3.01, 1, ldk)
g = chains.McmcGraph(tk, tv, tl, tg, tb, 3, prior, sdp, pk, 1, ldk, ts, td, to, seed=4, enos=True)
g.run(2)
nb, info = tempering.tempering_swap_round_device(tl, tb, 5, 0)
torch.cuda.synchronize()
assert int(g.counter.item()) == 2 and sorted(nb.cpu().tolist()) == sorted(beta.tolist())
print("sanitize_small ok")
