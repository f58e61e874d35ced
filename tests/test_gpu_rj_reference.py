"""The device's birth/death, AR(1) and swap moves against their exact stationary laws
(tests/rj_reference.py).

* Birth/death: chains.bd_step_device under ISMPPRIOR = 1 (ENOS = 0), 65 536 chains started at the
  law, deviates drawn by torch on the device; one case fills the kmax = ldk = 64 boundary.
* The whole iteration (chains.McmcGraph) under ENOS = 1, hmin = 0: at hmx = 5, where the law
  spreads over k, and at the default hmx, where it collapses to kmin.
* McmcGraph with the AR(1) move under ISMPPRIOR = 1: the law, and a bit-for-bit oracle replay.
* The swap round (tempering_swap_round_device) on n = 2..5 replicas with fixed logL: one-round
  transitions against the exact row given the round's matching, and a thinned long run against
  the stationary law.
"""
import numpy as np
import pytest
from scipy import stats

import oracle
import rj_reference as rj
from raytracerfortran_b200 import chains, workloads

pytestmark = pytest.mark.gpu

P_PASS = 1e-4
P_REJECT = 1e-6
B = 65_536


def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _sources():
    so, sd = workloads.make_sources(4, 7)
    return so, sd, np.ones(4)


def _show(name, p):
    print(f"\n{name}", {a: f"{b:.3g}" for a, b in p.items()})
    return p


class _PriorSampling:
    """ISMPPRIOR = 1 on the device (and in the oracle) for the duration of a block."""

    def __enter__(self):
        import raytracerfortran_b200 as rt
        rt.set_option("ismpprior", 1)
        oracle.set_ismpprior(1)

    def __exit__(self, *exc):
        import raytracerfortran_b200 as rt
        rt.set_option("ismpprior", 0)
        oracle.set_ismpprior(0)


# ---- births and deaths only, ENOS = 0 -----------------------------------------------------------

BD_CASES = {"hmin100.1-poisson": (100.1, 3.01, 12), "hmin100.1-flat": (100.1, None, 12),
            "hmin1000-poisson": (1000.0, 3.01, 12), "hmin1-lam60-kmax64": (1.0, 60.0, 64)}


@pytest.mark.parametrize("case", list(BD_CASES))
def test_device_bd_keeps_the_enos0_law(case, record_property):
    """300 birth/death moves of 65 536 chains started at the law (kmin = 1, ldk = kmax): k by chi^2,
    the pooled depth and vp transforms by KS.  At hmin = 100.1 the same counts reject pk itself."""
    import torch
    hmin, lam, kmax = BD_CASES[case]
    law = rj.BdLaw(0, chains.prior_array(hmin=hmin), chains.sd_prior_array(), 1, kmax, lam)
    rng = np.random.default_rng(600 + kmax + int(hmin))
    k, voro, sigma = law.sample(B, rng, kmax)
    pk = None if lam is None else chains.poisson_pk(lam, 1, kmax)
    so, sd, tobs = _sources()
    tk, tv, tl, tg, tb, ts, td, to = _dev(k, voro, np.ones(B), sigma, np.ones(B), so, sd, tobs)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(700 + kmax)
    accepted = 0
    with _PriorSampling():
        for _ in range(300):
            u = torch.rand((5, B), dtype=torch.float64, device="cuda", generator=gen)
            idel = (2 + torch.floor(u[4] * (tk - 1).clamp(min=1))).to(torch.int32)
            acc = chains.bd_step_device(tk, tv, tl, u[0].contiguous(), idel, u[1].contiguous(), u[2].contiguous(),
                                        u[3].contiguous(), tb, tg, law.prior, pk, 1, kmax, ts, td, to)
            accepted += int((acc == 1).sum())
        torch.cuda.synchronize()
    k, voro = tk.cpu().numpy(), tv.cpu().numpy()
    p = _show(f"device birth/death, {case}:", law.pvalues(k, voro, rng))
    record_property("min_p", f"{min(p.values()):.3g}")
    assert min(p.values()) >= P_PASS, p
    assert accepted > 300 * B // 20 and (tl.cpu().numpy() == 1.0).all() and voro[:, 0, :].max() <= law.L
    if kmax == 64:
        at_kmax = int((k == 64).sum())
        print(f"chains at k = kmax = 64: {at_kmax} (law {law.pi[-1] * B:.0f})")
        assert at_kmax > 1000
    if hmin == 100.1:
        p_pk = rj.chi2_pvalue(np.bincount(k - 1, minlength=kmax), law.intended)
        print(f"chi^2 p against pk itself: {p_pk:.3g}")
        assert p_pk < P_REJECT


# ---- the whole iteration, ENOS = 1 --------------------------------------------------------------

def _graph_run(law, k, voro, sigma, n_moves, iters, seed, ar=None):
    import torch
    so, sd, tobs = _sources()
    tk, tv, tl, tg, tb, ts, td, to = _dev(k, voro, np.ones(k.size), sigma, np.ones(k.size), so, sd, tobs)
    pk = None if law.lam is None else chains.poisson_pk(law.lam, law.kmin, law.kmax)
    g = chains.McmcGraph(tk, tv, tl, tg, tb, n_moves, law.prior, law.sd_prior, pk, law.kmin, law.kmax, ts, td, to,
                         seed=seed, enos=law.enos, ar=ar)
    with _PriorSampling():
        g.run(iters)
        torch.cuda.synchronize()
    return g, tk.cpu().numpy(), tv.cpu().numpy(), tg.cpu().numpy()


def test_mcmc_graph_keeps_the_enos1_law(record_property):
    """hmx = 5: pi spreads over k = 1..12.  65 536 chains started at the law, 40 iterations of
    birth/death, 23 sweep moves (a full sweep at k = 12) and the data-error move: k, the pooled
    depths, vp and sigma keep the law, and the counts reject the intended pk."""
    law = rj.BdLaw(1, chains.prior_array(hmin=0.0, hmx=5.0), chains.sd_prior_array(), 1, 12, 3.01)
    rng = np.random.default_rng(801)
    k, voro, sigma = law.sample(B, rng, 12)
    g, k, voro, sigma = _graph_run(law, k, voro, sigma, 23, 40, seed=802)
    p = _show("McmcGraph ENOS = 1, hmx = 5:", law.pvalues(k, voro, rng, sigma))
    record_property("min_p", f"{min(p.values()):.3g}")
    assert min(p.values()) >= P_PASS, p
    assert rj.chi2_pvalue(np.bincount(k - 1, minlength=12), law.intended) < P_REJECT
    assert g.tally[2].sum().item() > 40 * B // 20


def test_mcmc_graph_enos1_collapses_at_the_default_hmx(record_property):
    """hmx = 10000.1: the law has pi(2)/pi(1) = 5.0e-4 (pk(2)/pk(1) = 1.5).  65 536 chains started
    at the law, 100 iterations: the k = 2 count is binomial with pi(2), and k >= 3 (pi(3) = 2e-7)
    holds at most one chain."""
    law = rj.BdLaw(1, chains.prior_array(hmin=0.0), chains.sd_prior_array(), 1, 12, 3.01)
    rng = np.random.default_rng(811)
    k, voro, sigma = law.sample(B, rng, 12)
    _, k, _, _ = _graph_run(law, k, voro, sigma, 3, 100, seed=812)
    n1, n2 = int((k == 1).sum()), int((k == 2).sum())
    p = stats.binomtest(n2, B, law.pi[1]).pvalue
    print(f"\nENOS = 1, default hmx: pi(2)/pi(1) = {n2 / n1:.4g} on the device ({n2} of {B} chains at k = 2, "
          f"law {law.ratio(1):.4g}, binomial p = {p:.3g})")
    record_property("pi2_over_pi1", f"{n2 / n1:.4g}")
    record_property("binomial_p", f"{p:.3g}")
    assert p >= P_PASS and int((k >= 3).sum()) <= 1


# ---- McmcGraph with the AR(1) move under ISMPPRIOR = 1 -----------------------------------------

def test_mcmc_graph_ar_move_keeps_its_law(record_property):
    """65 536 chains, the birth/death law (ENOS = 0, hmin = 0) and the AR law at the start, 40
    iterations with the AR move: idxar ~ Bernoulli(1/2), arpar | idxar = 1 uniform, and k and vp
    keep their law.  With hmin = 0 no birth is refused for its spacing, so k does not depend on the
    depths, which the ENOS = 0 sweep does not keep uniform (DESIGN.md section 2)."""
    law = rj.BdLaw(0, chains.prior_array(hmin=0.0), chains.sd_prior_array(), 1, 12, 3.01)
    rng = np.random.default_rng(821)
    k, voro, sigma = law.sample(B, rng, 12)
    ap = chains.ar_prior_array()
    ti, ta = _dev(*rj.ar_sample(B, ap, rng))
    g, k, voro, _ = _graph_run(law, k, voro, sigma, 1, 40, seed=822, ar=(ti, ta, ap))
    p = rj.ar_pvalues(ti.cpu().numpy(), ta.cpu().numpy(), ap)
    p.update({"k": law.k_pvalue(k), "vp": rj.ks_uniform(law.vp_pit(k, voro))})
    _show("McmcGraph with AR under ISMPPRIOR = 1:", p)
    record_property("min_p", f"{min(p.values()):.3g}")
    assert min(p.values()) >= P_PASS, p
    assert g.tally[4].sum().item() > 40 * B // 10


def test_mcmc_graph_ar_under_ismpprior_matches_oracle():
    """ISMPPRIOR = 1 with IAR = 1, the combination no other test runs: two iterations of the graph
    replayed by the oracle from the workspace's deviates give the same outcome of every move and
    bit-identical states, and AR births are accepted (the oracle used to evaluate them on the real
    likelihood and reject them)."""
    import torch
    n, ldk, M = 1200, 8, 5
    law = rj.BdLaw(0, chains.prior_array(), chains.sd_prior_array(), 1, ldk, 3.01)
    rng = np.random.default_rng(831)
    k, voro, sigma = law.sample(n, rng, ldk)
    ap = chains.ar_prior_array()
    idxar, arpar = rj.ar_sample(n, ap, rng)
    so, sd, tobs = _sources()
    beta = 1.0 / 1.4 ** rng.integers(0, 4, n)
    ll = np.ones(n)
    pk = chains.poisson_pk(3.01, 1, ldk)
    tk, tv, tl, tg, ti, ta, tb, ts, td, to = _dev(k, voro, ll, sigma, idxar, arpar, beta, so, sd, tobs)
    ck, cv, cl, cs, ci, ca = k.copy(), voro, ll, sigma.copy(), idxar, arpar
    births = 0
    with _PriorSampling():
        g = chains.McmcGraph(tk, tv, tl, tg, tb, M, law.prior, law.sd_prior, pk, 1, ldk, ts, td, to, seed=832,
                             ar=(ti, ta, ap))
        try:
            for it in range(2):
                g.run(1)
                torch.cuda.synchronize()
                w = {name: t.cpu().numpy().copy() for name, t in g.views.items()}
                oracle.set_chain_ar(ci, ca, float(ap[3]))
                r = oracle.bd_step_batch(ck, cv, cl, w["u_k"], w["idel"], w["u_z"], w["u_v"], w["u_acc_bd"], beta, cs,
                                         law.prior, pk, 1, ldk, so, sd, tobs)
                assert np.array_equal(w["acc_bd"], r["accept"]), f"bd {it}"
                ck, cv, cl = r["k"], r["voro"], r["logL"]
                for m in range(M):
                    r = oracle.mh_step_batch(ck, cv, cl, w["ivo"][m], w["iwhich"][m], w["dev"][m], w["u_acc"][m], beta,
                                             cs, law.prior, so, sd, tobs)
                    assert np.array_equal(w["acc_mh"][m], r["accept"]), f"move {m}, iteration {it}"
                    cv, cl = r["voro"], r["logL"]
                r = oracle.sd_step_batch(ck, cv, cl, cs, w["u_gate"], w["gauss"], w["u_acc_sd"], beta, law.sd_prior,
                                         so, sd, tobs)
                assert np.array_equal(w["acc_sd"], r["accept"]), f"sd {it}"
                cl, cs = r["logL"], r["sigma"]
                r = oracle.ar_step_batch(ck, cv, cl, cs, ci, ca, w["u_choice"], w["u_prop_ar"], w["gauss_ar"],
                                         w["u_acc_ar"], beta, ap, so, sd, tobs)
                assert np.array_equal(w["acc_ar"], r["accept"]), f"ar {it}"
                births += int(((ci == 0) & (r["accept"] == 1)).sum())
                cl, ci, ca = r["logL"], r["idxar"], r["arpar"]
                assert np.array_equal(tk.cpu().numpy(), ck)
                assert np.array_equal(tv.cpu().numpy().view(np.uint64), cv.view(np.uint64)), f"iteration {it}"
                assert np.array_equal(tg.cpu().numpy().view(np.uint64), cs.view(np.uint64))
                assert np.array_equal(ti.cpu().numpy(), ci)
                assert np.array_equal(ta.cpu().numpy().view(np.uint64), ca.view(np.uint64))
                assert (tl.cpu().numpy() == 1.0).all() and (cl == 1.0).all()
        finally:
            oracle.set_chain_ar()
    print(f"\nAR births accepted in the replay: {births}")
    assert births > 200


# ---- the swap round -----------------------------------------------------------------------------

def _swap_setup(n):
    return np.linspace(-2.0, 4.0, n), 1.0 / 1.4 ** np.arange(n)


def _matching_of(partner):
    """The round's pairs from rtb200_swap_round_device's partner array (j accepted, -1 - j
    rejected, -1 unpaired; -1 is also 'rejected with replica 0', told apart by replica 0's entry)."""
    n = partner.size
    dec = [int(v) if v >= 0 else -1 - int(v) for v in partner]      # -1 reads as replica 0
    mate0 = dec[0] if dec[0] != 0 else None
    pairs = set()
    for i in range(1, n):
        if dec[i] == 0 and mate0 != i:
            continue                                                 # unpaired
        pairs.add((min(i, dec[i]), max(i, dec[i])))
    return tuple(sorted(pairs))


def _swap_rounds(logL, beta0, seed, rounds, round0, feed_back=False, keep_every=1):
    """Run `rounds` device swap rounds with distinct round indices; returns (betas [S, n], partner [S, n])
    of every `keep_every`-th round, starting from beta0 each time or (feed_back) from the last."""
    import torch
    from raytracerfortran_b200 import tempering
    tl, tb0 = _dev(logL, beta0)
    S = rounds // keep_every
    betas = torch.empty((S, logL.size), dtype=torch.float64, device="cuda")
    partners = torch.empty((S, logL.size), dtype=torch.int32, device="cuda")
    beta = tb0
    for r in range(rounds):
        out, info = tempering.tempering_swap_round_device(tl, beta, seed, round0 + r)
        if feed_back:
            beta = out
        if (r + 1) % keep_every == 0:
            betas[(r + 1) // keep_every - 1].copy_(out)
            partners[(r + 1) // keep_every - 1].copy_(info["partner"])
    torch.cuda.synchronize()
    return betas.cpu().numpy(), partners.cpu().numpy()


def _assignment_index(betas, ladder):
    """Assignment a (a[r] = ladder index of replica r's beta) of each row, as an index into rj.assignments."""
    n = ladder.size
    A = {a: i for i, a in enumerate(rj.assignments(n))}
    pos = np.argmin(np.abs(betas[:, :, None] - ladder[None, None, :]), axis=2)
    assert np.array_equal(ladder[pos], betas), "a beta left the ladder"
    return np.array([A[tuple(int(x) for x in row)] for row in pos])


SWAP_N = [2, 3, 4, 5]


@pytest.mark.parametrize("n", SWAP_N)
def test_swap_round_transition_rows(n, record_property):
    """From each of several starting assignments (the identity, where every swap is accepted, the
    reverse and a random one), 20 000 rounds with distinct round indices.  The outcome counts
    against the exact row given each round's matching (read back from the partner array): the
    pairing is not a uniform matching (test_swap_pairing_is_not_a_uniform_matching), so the
    unconditional uniform-matching row is printed, not asserted."""
    logL, ladder = _swap_setup(n)
    A = rj.assignments(n)
    M = rj.matchings(n)
    mindex = {tuple(sorted(tuple(sorted(p)) for p in m)): i for i, m in enumerate(M)}
    rng = np.random.default_rng(900 + n)
    starts = [tuple(range(n)), tuple(range(n))[::-1]]
    others = [a for a in A if a not in starts]
    starts += [others[rng.integers(len(others))]] if others else []
    worst = 1.0
    for s_i, start in enumerate(starts):
        betas, partners = _swap_rounds(logL, ladder[list(start)], seed=77 + n, rounds=20_000,
                                       round0=(1 << 33) + 100_000 * s_i)
        out = _assignment_index(betas, ladder)
        mt = np.array([mindex[_matching_of(p)] for p in partners])
        counts = np.bincount(out, minlength=len(A))
        expected = np.zeros(len(A))
        for mi in np.unique(mt):
            w = [1.0 if j == mi else 0.0 for j in range(len(M))]
            _, Pm = rj.swap_transition(logL, ladder, weights=w)
            expected += (mt == mi).sum() * Pm[A.index(start)]
        p = rj.chi2_pvalue(counts, expected / expected.sum())
        _, P = rj.swap_transition(logL, ladder)
        p_uniform = rj.chi2_pvalue(counts, P[A.index(start)])
        print(f"\nn = {n}, start {start}: chi^2 p given the matchings {p:.3g}; "
              f"against a uniform matching {p_uniform:.3g}; matchings seen {np.bincount(mt).tolist()}")
        assert p >= P_PASS, (start, p)
        worst = min(worst, p)
    record_property("min_p", f"{worst:.3g}")


def test_swap_round_long_run_keeps_the_stationary_law(record_property):
    """n = 4: one chain of 160 000 rounds fed back into each other, every 20th assignment kept
    (|lambda_2| = 0.67 for a uniform matching, so 20 rounds leave a correlation below 1e-3): the
    8000 kept assignments against pi ∝ exp(sum beta L)."""
    n = 4
    logL, ladder = _swap_setup(n)
    betas, _ = _swap_rounds(logL, ladder, seed=91, rounds=160_000, round0=5, feed_back=True, keep_every=20)
    _, pi = rj.swap_stationary(logL, ladder)
    counts = np.bincount(_assignment_index(betas, ladder), minlength=pi.size)
    p = rj.chi2_pvalue(counts, pi)
    print(f"\nn = 4 long run: chi^2 p against the stationary law {p:.3g}")
    record_property("p", f"{p:.3g}")
    assert p >= P_PASS
