"""The exact laws of tests/rj_reference.py checked without a GPU.

* The laws against the oracle: oracle chains under ISMPPRIOR = 1 started at the exact law of the
  birth/death move (ENOS = 0) or of the whole iteration (ENOS = 1, hmin = 0) still follow it; one
  state per chain, so the p-values are exact.
* Power: plain numpy models of the birth/death, AR and swap moves follow the laws, and each of
  the mutants a kernel could plausibly carry is rejected.
* Two recorded properties of the moves as the reference defines them (DESIGN.md section 2): the
  ENOS = 0 k-marginal is tilted away from pk by the hmin spacing, and under ENOS = 1 the chain
  collapses to kmin at the default hmx.
* The oracle's AR move under ISMPPRIOR = 1 evaluates LOGLHOOD2's constant, like its other moves.
"""
import math

import numpy as np
import pytest
from scipy import stats

import oracle
import rj_reference as rj
from oracle.tempering_ref import swap_perm
from raytracerfortran_b200 import chains

P_PASS = 1e-4        # a true null fails this with probability 1e-4 per check; seeds are fixed
P_REJECT = 1e-6
SRC = (np.array([1000.0]), np.array([10.0]), np.array([1.0]))      # unused: logL = 1


def _show(name, p):
    print(name, {a: f"{b:.3g}" for a, b in p.items()})
    return p


# ---- the laws on their own ----------------------------------------------------------------------

def test_laws_are_consistent():
    """hmin = 0 gives pk back (up to q_b/q_d = 0.3333/0.3334 per step); the volume factor is exactly
    0 once k - 1 interfaces no longer fit; the ENOS = 1 ratio is the closed form; the exact samplers
    follow their own laws; every swap transition matrix is stochastic and keeps its stationary law."""
    sp = chains.sd_prior_array()
    law = rj.BdLaw(0, chains.prior_array(hmin=0.0), sp, 1, 12, 3.01)
    tilt = law.pi / law.intended / (law.pi[0] / law.intended[0])
    assert ((tilt <= 1.0 + 1e-12) & (tilt >= (0.3333 / 0.3334) ** 11 - 1e-12)).all()
    law = rj.BdLaw(0, chains.prior_array(hmin=1000.0), sp, 1, 12, None)
    assert (law.pi[10:] == 0.0).all() and law.pi[9] > 0.0          # (k - 1) hmin >= L_b = 9000.1 at k = 11
    law = rj.BdLaw(1, chains.prior_array(hmin=0.0), sp, 1, 12, 3.01)
    hmx = 10000.1
    assert math.isclose(law.ratio(1), 3.01 / 2 * (4 * 5) / (2 * 3) / hmx * 0.3333 / 0.3334, rel_tol=1e-12)
    assert math.isclose(law.ratio(2), 3.01 / 3 * (6 * 7) / (4 * 5) * 2 / hmx * 0.3333 / 0.3334, rel_tol=1e-12)
    rng = np.random.default_rng(1)
    for law in (rj.BdLaw(0, chains.prior_array(), sp, 1, 12, 3.01),
                rj.BdLaw(1, chains.prior_array(hmin=0.0, hmx=5.0), sp, 1, 12, 3.01)):
        k, voro, sigma = law.sample(40_000, rng, 12)
        p = _show("exact sampler:", law.pvalues(k, voro, rng, sigma))
        assert min(p.values()) >= P_PASS
    for n in range(2, 7):
        logL, ladder = np.linspace(-2.0, 4.0, n), 1.0 / 1.4 ** np.arange(n)
        A, P = rj.swap_transition(logL, ladder)
        _, pi = rj.swap_stationary(logL, ladder)
        assert len(A) == math.factorial(n) and len(rj.matchings(n)) == (1, 3, 3, 15, 15)[n - 2]
        assert np.allclose(P.sum(axis=1), 1.0, atol=1e-14) and np.allclose(pi @ P, pi, atol=1e-14)


def test_chi2_merging():
    """Cells expecting fewer than 5 are merged with their neighbours; a count where the law puts
    no mass fails outright."""
    p = np.array([0.5, 0.49, 0.006, 0.004, 0.0])
    assert rj.chi2_pvalue([500, 490, 6, 4, 0], p) > 0.9
    assert rj.chi2_pvalue([500, 489, 6, 4, 1], p) == 0.0
    assert rj.chi2_pvalue([500, 460, 40, 0, 0], p) < 1e-6


# ---- the oracle's birth/death move against the ENOS = 0 law -------------------------------------

def _oracle_bd(law, n, steps, seed):
    rng = np.random.default_rng(seed)
    k, voro, sigma = law.sample(n, rng, law.kmax)
    pk = None if law.lam is None else chains.poisson_pk(law.lam, law.kmin, law.kmax)
    ll, beta = np.ones(n), np.ones(n)
    oracle.set_ismpprior(1)
    try:
        for _ in range(steps):
            u = rng.random((5, n))
            idel = (2 + np.floor(u[4] * np.maximum(k - 1, 1))).astype(np.int32)
            r = oracle.bd_step_batch(k, voro, ll, u[0], idel, u[1], u[2], u[3], beta, sigma, law.prior, pk,
                                     law.kmin, law.kmax, *SRC)
            k, voro = r["k"], r["voro"]
    finally:
        oracle.set_ismpprior(0)
    return k, voro, rng


BD0 = [(100.1, 3.01), (100.1, None), (1000.0, 3.01), (1000.0, None)]


@pytest.fixture(scope="module")
def bd0_runs():
    out = {}
    for hmin, lam in BD0:
        law = rj.BdLaw(0, chains.prior_array(hmin=hmin), chains.sd_prior_array(), 1, 12, lam)
        out[(hmin, lam)] = (law,) + _oracle_bd(law, 20_000, 200, seed=int(hmin) + (0 if lam is None else 7))
    return out


@pytest.mark.parametrize("hmin,lam", BD0, ids=[f"hmin{h}-{'poisson' if l else 'flat'}" for h, l in BD0])
def test_oracle_bd_keeps_the_enos0_law(bd0_runs, hmin, lam):
    """20 000 oracle chains, ENOS = 0, kmin = 1, kmax = 12, started at the exact law and run 200
    birth/death moves: k by chi^2, the pooled depth and vp transforms by KS."""
    law, k, voro, rng = bd0_runs[(hmin, lam)]
    p = _show(f"oracle ENOS = 0, hmin = {hmin}, lam = {lam}:", law.pvalues(k, voro, rng))
    assert min(p.values()) >= P_PASS, p
    assert voro[:, 0, :].max() <= law.L


def test_enos0_k_marginal_is_tilted_by_hmin(bd0_runs):
    """Recorded property: with hmin > 0 the ENOS = 0 k-marginal is not pk but pk times the volume
    factor (1 - (k-1) hmin / L_b)^(k-1).  The oracle's counts reject pk (and the flat prior) at
    hmin = 100.1 and follow the law."""
    for lam in (3.01, None):
        law, k, _, _ = bd0_runs[(100.1, lam)]
        counts = np.bincount(k - 1, minlength=12)
        p_law, p_pk = rj.chi2_pvalue(counts, law.pi), rj.chi2_pvalue(counts, law.intended)
        print(f"lam = {lam}: chi^2 p against the law {p_law:.3g}, against pk {p_pk:.3g};",
              "pi(1), pk(1):", round(counts[0] / k.size, 4), round(law.intended[0], 4))
        assert p_law >= P_PASS and p_pk < P_REJECT


# ---- the whole iteration under ENOS = 1 ---------------------------------------------------------

def _oracle_iteration_enos1(law, n, iters, seed):
    """Oracle chains under ISMPPRIOR = 1, ENOS = 1, started at the law: per iteration the
    birth/death move, one full sweep of every chain (chains with fewer nodes sit a move out) and
    the data-error move, as chains.mcmc_step_device strings them."""
    rng = np.random.default_rng(seed)
    k, voro, sigma = law.sample(n, rng, law.kmax)
    pk = chains.poisson_pk(law.lam, law.kmin, law.kmax)
    ll, beta = np.ones(n), np.ones(n)
    oracle.set_ismpprior(1)
    oracle.set_enos(1)
    try:
        for _ in range(iters):
            u = rng.random((5, n))
            idel = (2 + np.floor(u[4] * np.maximum(k - 1, 1))).astype(np.int32)
            r = oracle.bd_step_batch(k, voro, ll, u[0], idel, u[1], u[2], u[3], beta, sigma, law.prior, pk,
                                     law.kmin, law.kmax, *SRC)
            k, voro = r["k"], r["voro"]
            for ivo in range(1, int(k.max()) + 1):
                for iw in ((2,) if ivo == 1 else (1, 2)):
                    u = rng.random((2, n))
                    dev = u[0] if iw == 1 else np.tan(np.pi * (u[0] - 0.5))
                    voro = oracle.mh_step_batch(k, voro, ll, np.full(n, ivo, np.int32), np.full(n, iw, np.int32),
                                                dev, u[1], beta, sigma, law.prior, *SRC)["voro"]
            u = rng.random((2, n))
            sigma = oracle.sd_step_batch(k, voro, ll, sigma, u[0], rng.standard_normal(n), u[1], beta,
                                         law.sd_prior, *SRC)["sigma"]
    finally:
        oracle.set_ismpprior(0)
        oracle.set_enos(0)
    return k, voro, sigma, rng


def test_oracle_iteration_keeps_the_enos1_law():
    """hmx = 5 (a few units), so pi spreads over k = 1..12: 20 000 chains, 40 iterations; k, the
    pooled depths (odd order statistics restored), vp and sigma keep the law, and the counts reject
    the intended pk."""
    law = rj.BdLaw(1, chains.prior_array(hmin=0.0, hmx=5.0), chains.sd_prior_array(), 1, 12, 3.01)
    k, voro, sigma, rng = _oracle_iteration_enos1(law, 20_000, 40, seed=11)
    p = _show("oracle ENOS = 1, hmx = 5:", law.pvalues(k, voro, rng, sigma))
    assert min(p.values()) >= P_PASS, p
    assert rj.chi2_pvalue(np.bincount(k - 1, minlength=12), law.intended) < P_REJECT


def test_enos1_collapses_to_kmin_at_the_default_hmx():
    """Recorded property: the coded ENOS = 1 ratio has no proposal term, so at hmx = 10000.1 the
    law puts pi(2)/pi(1) = 3.01/2 * 20/6 * 1/hmx * 0.3333/0.3334 = 5.0e-4 where the intended prior
    has pk(2)/pk(1) = 1.5.  40 000 oracle chains started at k = 1 (births and deaths only, 300
    moves): the k = 2 count is binomial with that probability, k >= 3 (pi(3) = 2e-7) stays empty."""
    law = rj.BdLaw(1, chains.prior_array(hmin=0.0), chains.sd_prior_array(), 1, 12, 3.01)
    n, rng = 40_000, np.random.default_rng(12)
    k, voro = np.ones(n, np.int32), np.zeros((n, 2, 12))
    voro[:, 1, 0] = rng.uniform(1500.0, 10000.0, n)
    ll, beta, sigma = np.ones(n), np.ones(n), np.full(n, 0.01)
    pk = chains.poisson_pk(3.01, 1, 12)
    oracle.set_ismpprior(1)
    oracle.set_enos(1)
    try:
        for _ in range(300):
            u = rng.random((5, n))
            idel = (2 + np.floor(u[4] * np.maximum(k - 1, 1))).astype(np.int32)
            r = oracle.bd_step_batch(k, voro, ll, u[0], idel, u[1], u[2], u[3], beta, sigma, law.prior, pk, 1, 12,
                                     *SRC)
            k, voro = r["k"], r["voro"]
    finally:
        oracle.set_ismpprior(0)
        oracle.set_enos(0)
    n2 = int((k == 2).sum())
    p = stats.binomtest(n2, n, law.pi[1]).pvalue
    print(f"ENOS = 1, hmx = {law.hmx}: pi(2)/pi(1) = {law.ratio(1):.4g} (law), "
          f"{n2 / max(int((k == 1).sum()), 1):.4g} (oracle, {n2} of {n} chains at k = 2, p = {p:.3g})")
    assert math.isclose(law.ratio(1), 5.0e-4, rel_tol=0.01)
    assert p >= P_PASS and (k >= 3).sum() == 0


# ---- a numpy model of the ENOS = 0 birth/death move, and its mutants -----------------------------

def _np_bd(law, n, steps, seed, mutant=None):
    """The ENOS = 0 move from its definition: ran_unik picks birth / death (q_b, q_d), a birth draws
    depth L_b u_z and vp uniformly, a death removes node idel = 2 + floor(u (k - 1)), nodes are
    re-sorted, CHECKBOUNDS refuses what violates the hmin spacing, and the pk ratio decides.
    Mutants: "idel 1..k" (the top node can die: its vp goes and node 2 becomes the top node),
    "idel 2..k+1" (idel = k + 1 is refused, like an out-of-range idel in the oracle), "pk ratio
    dropped", "pk ratio inverted", "q = 0.5 inside" (birth iff u <= 0.5 inside (kmin, kmax), the
    boundaries unchanged; q_b = q_d = 0.5 everywhere would shift pi by (0.3334/0.3333)^k only)."""
    rng = np.random.default_rng(seed)
    kmin, kmax, ldk = law.kmin, law.kmax, law.kmax + 1
    k, voro, _ = law.sample(n, rng, ldk)
    cols = np.arange(ldk)[None, :]
    d = np.where(cols < k[:, None], voro[:, 0, :], np.inf)
    v = voro[:, 1, :].copy()
    vmin, vmax, hmin, hmx = law.prior[3], law.prior[5], law.hmin, law.hmx
    lpk = np.array([rj.log_pk(i, law.lam) for i in range(ldk + 1)])
    rows = np.arange(n)
    for _ in range(steps):
        u = rng.random((5, n))
        lo, hi = (0.5, 0.5) if mutant == "q = 0.5 inside" else (rj.Q_LO, rj.Q_HI)
        birth = np.where(k == kmax, False, np.where(k == kmin, u[0] <= rj.Q_LO, u[0] <= lo))
        death = np.where(k == kmax, u[0] <= rj.Q_LO, np.where(k == kmin, False, u[0] > hi))
        if mutant == "idel 1..k":
            idel = 1 + np.floor(u[4] * k).astype(np.int64)
        elif mutant == "idel 2..k+1":
            idel = 2 + np.floor(u[4] * k).astype(np.int64)
        else:
            idel = 2 + np.floor(u[4] * np.maximum(k - 1, 1)).astype(np.int64)
        dn, vn = d.copy(), v.copy()
        b = rows[birth]
        dn[b, k[b]] = law.L * u[1][b]
        vn[b, k[b]] = vmin + (vmax - vmin) * u[2][b]
        dd = rows[death]
        dn[dd, np.minimum(idel[dd], ldk) - 1] = np.inf
        order = np.argsort(dn, axis=1, kind="stable")
        dn, vn = np.take_along_axis(dn, order, axis=1), np.take_along_axis(vn, order, axis=1)
        dn[:, 0] = 0.0                                           # the top node sits at depth 0
        kn = np.where(birth, k + 1, np.where(death, k - 1, k))
        with np.errstate(invalid="ignore"):                      # inf - inf past the last node
            gaps = np.diff(dn, axis=1)                           # h_1 = z_2, h_i = z_{i+1} - z_i
        live = cols[:, 1:] < kn[:, None]
        ok = ~(live & ((gaps < hmin) | (dn[:, 1:] > hmx))).any(axis=1)
        ok &= ~(death & ((idel < 2) & (mutant != "idel 1..k") | (idel > k)))
        logr = lpk[kn] - lpk[k]
        if mutant == "pk ratio dropped":
            logr = 0.0 * logr
        elif mutant == "pk ratio inverted":
            logr = -logr
        acc = (birth | death) & ok & ~(u[3] >= np.exp(logr))
        d = np.where(acc[:, None], dn, d)
        v = np.where(acc[:, None], vn, v)
        k = np.where(acc, kn, k)
    voro = np.zeros((n, 2, ldk))
    voro[:, 0, :] = np.where(cols < k[:, None], d, 0.0)
    voro[:, 1, :] = np.where(cols < k[:, None], v, 0.0)
    return law.pvalues(k, voro, rng)


BD_MUTANTS = ["idel 1..k", "idel 2..k+1", "pk ratio dropped", "pk ratio inverted", "q = 0.5 inside"]


@pytest.fixture(scope="module")
def bd_model_law():
    return rj.BdLaw(0, chains.prior_array(hmin=100.1), chains.sd_prior_array(), 1, 12, 3.01)


def test_numpy_bd_model_keeps_the_law(bd_model_law):
    p = _show("numpy birth/death model:", _np_bd(bd_model_law, 40_000, 150, seed=21))
    assert min(p.values()) >= P_PASS, p


@pytest.mark.parametrize("mutant", BD_MUTANTS)
def test_bd_mutant_is_rejected(bd_model_law, mutant):
    p = _show(f"mutant {mutant}:", _np_bd(bd_model_law, 40_000, 150, seed=22, mutant=mutant))
    assert min(p.values()) < P_REJECT, p


# ---- the AR(1) move -----------------------------------------------------------------------------

def _np_ar(ar_prior, n, steps, seed, swapped=False):
    """The AR move from its definition under a flat likelihood: birth with log-ratio log 1/2, death
    (u_choice >= 1/2) with log 2, otherwise a Gaussian step kept inside the bounds."""
    rng = np.random.default_rng(seed)
    pert, lo, hi = float(ar_prior[0]), float(ar_prior[1]), float(ar_prior[2])
    lb, ld = (math.log(2.0), math.log(0.5)) if swapped else (math.log(0.5), math.log(2.0))
    idx, ar = rj.ar_sample(n, ar_prior, rng)
    for _ in range(steps):
        u = rng.random((3, n))
        g = rng.standard_normal(n)
        birth, death = idx == 0, (idx == 1) & (u[0] >= 0.5)
        new = np.where(birth, lo + (hi - lo) * u[1], np.where(death, lo - 1.0, ar + pert * g))
        inside = death | ((new >= lo) & (new <= hi))
        logr = np.where(birth, lb, np.where(death, ld, 0.0))
        acc = inside & ~(u[2] >= np.exp(logr))
        idx = np.where(acc, np.where(birth, 1, np.where(death, 0, idx)), idx)
        ar = np.where(acc, new, ar)
    return rj.ar_pvalues(idx, ar, ar_prior)


def test_numpy_ar_model_and_its_mutant():
    ap = chains.ar_prior_array()
    p = _show("numpy AR model:", _np_ar(ap, 40_000, 30, seed=31))
    assert min(p.values()) >= P_PASS
    p = _show("AR log-ratios swapped:", _np_ar(ap, 40_000, 30, seed=32, swapped=True))
    assert min(p.values()) < P_REJECT


def _oracle_ar(n, steps, seed, start_at_law=True):
    rng = np.random.default_rng(seed)
    ap = chains.ar_prior_array()
    k, voro = np.full(n, 2, np.int32), np.zeros((n, 2, 2))
    voro[:, 0, 1], voro[:, 1] = 500.0, [2000.0, 3000.0]
    ll, sigma, beta = np.ones(n), np.full(n, 0.05), np.ones(n)
    idx, ar = rj.ar_sample(n, ap, rng) if start_at_law else (np.zeros(n, np.int32), np.full(n, ap[1] - 1.0))
    first = None
    oracle.set_ismpprior(1)
    try:
        for _ in range(steps):
            u = rng.random((3, n))
            r = oracle.ar_step_batch(k, voro, ll, sigma, idx, ar, u[0], u[1], rng.standard_normal(n), u[2], beta, ap,
                                     *SRC)
            ll, idx, ar = r["logL"], r["idxar"], r["arpar"]
            first = r if first is None else first
    finally:
        oracle.set_ismpprior(0)
    return idx, ar, ap, first


def test_oracle_ar_move_honours_ismpprior():
    """Under ISMPPRIOR = 1 the oracle's AR move evaluates LOGLHOOD2's constant like its other three
    moves (the device does, through its shared move evaluation), so its law is Bernoulli(1/2) x
    uniform: from the law and from idxar = 0 everywhere.  Before, it evaluated the real likelihood,
    rejected every birth on these data and left every chain at idxar = 0."""
    idx, ar, ap, first = _oracle_ar(20_000, 40, seed=41)
    evaluated = first["accept"] >= 0
    assert evaluated.sum() > 15_000 and (first["accept"] == 1).sum() > 5_000
    assert (first["logL_prop"][evaluated] == 1.0).all() and (first["logL"] == 1.0).all()
    p = _show("oracle AR from the law:", rj.ar_pvalues(idx, ar, ap))
    assert min(p.values()) >= P_PASS
    idx, ar, ap, _ = _oracle_ar(20_000, 40, seed=42, start_at_law=False)
    p = _show("oracle AR from idxar = 0:", rj.ar_pvalues(idx, ar, ap))
    assert min(p.values()) >= P_PASS


# ---- the swap round -----------------------------------------------------------------------------

SWAP_LOGL = {n: np.linspace(-2.0, 4.0, n) for n in range(2, 7)}
SWAP_LADDER = {n: 1.0 / 1.4 ** np.arange(n) for n in range(2, 7)}


def _np_swap(n, start, n_chains, rounds, rng, rule="exact"):
    """n_chains independent copies of the swap round on n replicas: a uniformly random matching,
    then pair (i, j) exchanges betas iff u <= exp(x), x = (b_j - b_i)(L_i - L_j).  Mutants: "sign"
    uses -x, "abs" uses |x|.  Returns the final assignments [n_chains, n]."""
    L, lad = SWAP_LOGL[n], SWAP_LADDER[n]
    M = rj.matchings(n)
    a = np.broadcast_to(np.asarray(start, dtype=np.int64), (n_chains, n)).copy()
    idx = np.arange(a.shape[0])
    for _ in range(rounds):
        m = np.array(M)[rng.integers(0, len(M), a.shape[0])]           # [N, n//2, 2]
        for t in range(m.shape[1]):
            i, j = m[:, t, 0], m[:, t, 1]
            bi, bj = lad[a[idx, i]], lad[a[idx, j]]
            x = (bj - bi) * (L[i] - L[j])
            x = {"exact": x, "sign": -x, "abs": np.abs(x)}[rule]
            acc = rng.random(a.shape[0]) <= np.exp(x)
            ai, aj = a[idx, i].copy(), a[idx, j].copy()
            a[idx, i], a[idx, j] = np.where(acc, aj, ai), np.where(acc, ai, aj)
    return a


def _counts(a, A):
    index = {s: r for r, s in enumerate(A)}
    return np.bincount([index[tuple(s)] for s in a], minlength=len(A))


def _swap_pvalues(n, rule, rng):
    """{"row": chi^2 of 20 000 one-round transitions from the identity against the exact row,
    "stationary": chi^2 of 20 000 chains started at the stationary law after 5 rounds}."""
    A, P = rj.swap_transition(SWAP_LOGL[n], SWAP_LADDER[n])
    _, pi = rj.swap_stationary(SWAP_LOGL[n], SWAP_LADDER[n])
    row = _counts(_np_swap(n, tuple(range(n)), 20_000, 1, rng, rule), A)
    start = np.array(A)[rng.choice(len(A), 20_000, p=pi)]
    stat = _counts(_np_swap(n, start, 20_000, 5, rng, rule), A)
    return {"row": rj.chi2_pvalue(row, P[0]), "stationary": rj.chi2_pvalue(stat, pi)}


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6])
def test_numpy_swap_model_and_its_mutants(n):
    rng = np.random.default_rng(50 + n)
    p = _show(f"swap n = {n}:", _swap_pvalues(n, "exact", rng))
    assert min(p.values()) >= P_PASS
    for rule in ("sign", "abs"):
        p = _show(f"swap n = {n}, rule {rule}:", _swap_pvalues(n, rule, rng))
        assert min(p.values()) < P_REJECT, (rule, p)


def test_swap_pairing_is_not_a_uniform_matching():
    """Recorded property of the device's pairing (restated in oracle/tempering_ref.py: a 4-round
    Feistel bijection of [0, 4^bits), cycle-walked into [0, n)): over 6000 rounds its matchings
    are not uniform for n = 4 and 5.  Each matching's round keeps the stationary law on its own,
    so the law of the chain is unaffected; only the one-round transition differs from a uniformly
    drawn matching's, and the device test conditions on the matching it reads back."""
    for n in (4, 5):
        M = {frozenset(map(frozenset, m)): r for r, m in enumerate(rj.matchings(n))}
        counts = np.zeros(len(M), np.int64)
        for r in range(6000):
            p = swap_perm(n, 12345, r)
            counts[M[frozenset(frozenset((int(p[2 * t]), int(p[2 * t + 1]))) for t in range(n // 2))]] += 1
        p_uniform = rj.chi2_pvalue(counts, np.full(len(M), 1.0 / len(M)))
        print(f"n = {n}: matching counts {counts.tolist()}, chi^2 p against uniform {p_uniform:.3g}")
        assert p_uniform < P_REJECT
        A, _ = rj.swap_transition(SWAP_LOGL[n], SWAP_LADDER[n])
        _, pi = rj.swap_stationary(SWAP_LOGL[n], SWAP_LADDER[n])
        for m in rj.matchings(n):
            _, Pm = rj.swap_transition(SWAP_LOGL[n], SWAP_LADDER[n], weights=[1.0 if x == m else 0.0
                                                                            for x in rj.matchings(n)])
            assert np.allclose(pi @ Pm, pi, atol=1e-14)
