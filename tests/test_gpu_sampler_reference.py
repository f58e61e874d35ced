"""The device sampler (chains.McmcGraph, rtb200_mcmc_iterations_device) against the independent
sampler reference (tests/sampler_reference.py).

* Deviates: every iteration's workspace against the numpy Philox restatement, bit for bit for the
  uniforms, idel, ivo, iwhich and the ENOS depth deviates; gauss, gauss_ar and the Cauchy steps
  within their bounds against mpmath (a sample plus the extremes) and numpy (all of them).
* Stationarity: under ISMPPRIOR = 1, chains started at the exact fixed-k prior still sample it
  after 64 full sweeps with the data-error move.
"""
import numpy as np
import pytest

import sampler_reference as sr
from raytracerfortran_b200 import chains, workloads

pytestmark = pytest.mark.gpu

P_PASS = 1e-4
COUNTER0 = (0, (1 << 32) - 2, (1 << 40) + 3)
SEEDS = (1, (1 << 32) + 5, (1 << 64) - 1)
MS = (1, 11, 506)
_worst = {}


def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _chains(B, ldk, prior, sd_prior, rng):
    """B chains with k spread over 1..ldk, each an exact draw of the ENOS = 0 fixed-k prior."""
    k = rng.integers(1, ldk + 1, B).astype(np.int32)
    voro, sigma = np.zeros((B, 2, ldk)), np.empty(B)
    for kv in np.unique(k):
        idx = np.flatnonzero(k == kv)
        depth, vp, sigma[idx] = sr.FixedKPrior(kv, 0, prior, sd_prior).sample(idx.size, rng)
        voro[idx, 0, 1:kv], voro[idx, 1, :kv] = depth, vp
    return k, voro, sigma


def _sources():
    so, sd = workloads.make_sources(4, 7)
    return so, sd, np.ones(4)


@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("B", [1, 129, 70_001])
def test_device_deviates_match_the_reference(B, M, record_property):
    """For each (B, M), three graphs: each counter start (0; 2^32 - 2, run three iterations so the
    counter's low word wraps into the high word; 2^40 + 3) with a seed of {1, 2^32 + 5, 2^64 - 1}
    and ENOS 0 or 1, rotated with M so that every B sees every (counter, seed) pair.  k per chain
    spans 1..ldk (birth/death runs, so it changes) and the sweep positions start at random."""
    import torch
    import raytracerfortran_b200 as rt
    ldk = 12
    j = MS.index(M)
    rng = np.random.default_rng(1000 * B + M)
    prior, sd_prior, pk = chains.prior_array(), chains.sd_prior_array(), chains.poisson_pk(3.01, 1, ldk)
    so, sd, tobs = _sources()
    worst = {"gauss": [0.0, 0.0], "gauss_ar": [0.0, 0.0], "dev": [0.0, 0.0]}
    n_checked = 0
    rt.set_option("ismpprior", 1)            # the deviates do not depend on the likelihood
    try:
        for i, counter0 in enumerate(COUNTER0):
            seed, enos = SEEDS[(i + j) % 3], (i + j) % 2
            k, voro, sigma = _chains(B, ldk, prior, sd_prior, rng)
            tk, tv, tl, tg, tb, ts, td, to = _dev(k, voro, np.ones(B), sigma, np.ones(B), so, sd, tobs)
            g = chains.McmcGraph(tk, tv, tl, tg, tb, M, prior, sd_prior, pk, 1, ldk, ts, td, to, seed=seed,
                                 enos=bool(enos), counter0=counter0)
            g.pos.copy_(torch.from_numpy(rng.integers(0, 2 * k.astype(np.int64) - 1).astype(np.int32)).cuda())
            for it in range(3 if counter0 == COUNTER0[1] else 1):
                k_before, pos_before = tk.cpu().numpy().copy(), g.pos.cpu().numpy().copy()
                g.run(1)
                torch.cuda.synchronize()
                w = {n: t.cpu().numpy() for n, t in g.views.items()}
                want = sr.draws(seed, counter0 + it, k_before, pos_before, M, enos, k_sweep=tk.cpu().numpy())
                rep = sr.compare_draws(w, want, enos, n_sample=2000, rng=rng)
                assert rep["ok"], (counter0 + it, seed, enos, rep)
                for n, (a, b) in rep["ratio"].items():
                    worst[n] = [max(worst[n][0], a), max(worst[n][1], b)]
                n_checked += 1
            assert int(g.counter.item()) == counter0 + (3 if counter0 == COUNTER0[1] else 1)
    finally:
        rt.set_option("ismpprior", 0)
    print(f"\nB = {B}, M = {M}: {n_checked} iterations, worst error/bound (mpmath, numpy/2):",
          {n: f"{a:.3f}, {b:.3f}" for n, (a, b) in worst.items()})
    for n, (a, b) in worst.items():
        record_property(f"worst_{n}", f"{a:.3f} / {b:.3f}")


STATIONARY = [(1, 2), (1, 6), (1, 20), (0, 2), (0, 6)]


@pytest.mark.parametrize("enos,k", STATIONARY, ids=[f"enos{e}-k{k}" for e, k in STATIONARY])
def test_device_moves_keep_the_prior(enos, k, record_property):
    """ISMPPRIOR = 1, kmin = kmax = k: 65 536 chains started at the exact fixed-k prior, 64
    iterations of one full sweep (M = 2k - 1) and the data-error move.  Every marginal keeps KS
    p >= 1e-4, except the ENOS = 0 depths at k = 6: the re-sort drift of the reference's algorithm
    (DESIGN.md section 2), recorded, not asserted."""
    import torch
    import raytracerfortran_b200 as rt
    B, iters, M = 65_536, 64, 2 * k - 1
    rng = np.random.default_rng(500 + 10 * k + enos)
    prior, sd_prior = (chains.prior_array(hmin=0.0) if enos else chains.prior_array()), chains.sd_prior_array()
    target = sr.FixedKPrior(k, enos, prior, sd_prior)
    depth, vp, sigma = target.sample(B, rng)
    voro = np.zeros((B, 2, k))
    voro[:, 0, 1:], voro[:, 1, :] = depth, vp
    so, sd, tobs = _sources()
    tk, tv, tl, tg, tb, ts, td, to = _dev(np.full(B, k, np.int32), voro, np.ones(B), sigma, np.ones(B), so, sd, tobs)
    rt.set_option("ismpprior", 1)
    try:
        g = chains.McmcGraph(tk, tv, tl, tg, tb, M, prior, sd_prior, None, k, k, ts, td, to, seed=77 + k,
                             enos=bool(enos))
        g.run(iters)
        torch.cuda.synchronize()
    finally:
        rt.set_option("ismpprior", 0)
    d, v = sr.states_of(tv.cpu().numpy(), k)
    p = sr.check_stationary({"depth": d, "vp": v, "sigma": tg.cpu().numpy()}, target)
    print(f"\nENOS = {enos}, k = {k}: min p {min(p.values()):.3g}",
          {n: f"{x:.2g}" for n, x in p.items()})
    asserted = {n: x for n, x in p.items() if not (enos == 0 and k > 2 and n.startswith("depth"))}
    if len(asserted) < len(p):
        pd = min(x for n, x in p.items() if n.startswith("depth"))
        record_property("enos0_depth_min_p", f"{pd:.3g}")
    assert min(asserted.values()) >= P_PASS, asserted
    assert (tk.cpu().numpy() == k).all() and (tl.cpu().numpy() == 1.0).all()
    tally = g.tally.cpu().numpy()
    proposed = iters * M * B
    assert 0 < tally[0].sum() <= tally[1].sum() < proposed      # accepted, and rejected outside the bounds
    assert tally[3].sum() > 0                                   # data-error moves accepted
