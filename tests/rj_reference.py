"""Exact stationary laws of the sampler's birth/death, AR(1) and tempering-swap moves.

Written from the move definitions (the comments of orc_bd_step_chain / orc_ar_step in
oracle/raymod_oracle.c and of raytracerfortran_b200/tempering.py), not from the kernels, so a
mistake that the device and the oracle share in these moves shows up as a law the chains do not
keep.  Every law comes with an exact sampler, so chains can start at the target, and with exact
goodness-of-fit checks on one state per chain.

Notation.  L_b = hmx - hmin is the birth range (BIRTH_FULL: znew = (maxlim1 - minlim1) u_z);
q_b(k), q_d(k) are the probabilities of proposing a birth / death from k nodes (ran_unik):
0.3333 / 0.3334 inside (kmin, kmax), 0.3333 / 0 at kmin, 0 / 0.3333 at kmax.  Under ISMPPRIOR = 1
(logL = 1) the birth of a node is accepted with min(1, A), the death with min(1, 1/A); a birth
draws the new depth with density 1/L_b and its vp with density 1/(vmax - vmin), a death removes one
of the k - 1 interfaces (idel = 2..k).  Detailed balance between k and k + 1 nodes then gives

    pi(k+1) g_{k+1}(y) / (pi(k) g_k(x)) = A * k / L_b * q_b(k) / q_d(k+1)

for the depth density g_k of k-node models (vp and sigma stay uniform).

* ENOS = 0, A = pk(k+1)/pk(k) (1 with pk = None).  g_k is uniform on the interfaces allowed by
  CHECKBOUNDS inside [0, L_b]: z_{i+1} = i hmin + y_i with y the order statistics of k - 1
  uniforms on [0, L_b - (k - 1) hmin].  Its volume is (L_b - (k-1) hmin)^(k-1) / (k-1)!, so

      pi(k) ∝ p~(k) (1 - (k - 1) hmin / L_b)_+^(k-1),  p~(k+1)/p~(k) = pk(k+1)/pk(k) q_b(k)/q_d(k+1),

  which is pk only when hmin = 0.  Chains that start inside z <= L_b stay there: a node in
  (L_b, hmx] passes CHECKBOUNDS and can be killed, but no birth can put one there.
* ENOS = 1, hmin = 0, A = pk(k+1)/pk(k) (2k+2)(2k+3)/L_b^2 (z*-z_j)(z_{j+1}-z*)/(z_{j+1}-z_j)
  as coded (BIRTH_FULL :1090-1098; DEATH_FULL is its inverse).  g_k = the intended
  Dirichlet(2, ..., 2) gaps on [0, hmx] satisfies the balance, since its density ratio
  g_{k+1}/g_k = 2k(2k+1)/hmx^2 times the same gap factor, and

      pi(k+1)/pi(k) = pk(k+1)/pk(k) (2k+2)(2k+3)/(2k(2k+1)) k hmx^2/L_b^3 q_b(k)/q_d(k+1).

  The ratio has no proposal term, so it carries 1/length: at the default hmx = 10000.1 the chain
  sits at kmin (pi(2)/pi(1) = 5.0e-4 for Poisson lambda = 3.01), where the intended prior is pk.
* AR(1) move, flat likelihood: idxar ~ Bernoulli(1/2); given idxar = 1, arpar ~ U[minlimar, maxlimar].
* Swap round on n replicas with fixed logL L_r: `swap_transition` enumerates the perfect matchings
  (one replica left out when n is odd) and the accept rule min(1, exp((b_j - b_i)(L_i - L_j))) over
  the n! assignments of the betas; its stationary law is ∝ exp(sum_r beta_sigma(r) L_r).
"""
import itertools
import math

import numpy as np
from scipy import stats

from sampler_reference import FixedKPrior

Q_LO, Q_HI = 0.3333, 0.6666          # ran_unik thresholds: birth iff u <= Q_LO, death iff u > Q_HI


def move_probs(k, kmin, kmax):
    """(q_b, q_d) of a chain with k nodes."""
    if kmin == kmax:
        return 0.0, 0.0
    if k == kmax:
        return 0.0, Q_LO
    if k == kmin:
        return Q_LO, 0.0
    return Q_LO, 1.0 - Q_HI


def log_pk(k, lam):
    """log of the Poisson prior pk(k) = e^-lam lam^k / k! (0 for lam = None: IPOIPR = 0)."""
    return 0.0 if lam is None else -lam + k * math.log(lam) - math.lgamma(k + 1.0)


def _normalise(logw):
    logw = np.asarray(logw, dtype=np.float64)
    w = np.exp(logw - logw[np.isfinite(logw)].max())
    return w / w.sum()


class BdLaw:
    """The stationary law of the birth/death move (ENOS = 0), or of the whole iteration (ENOS = 1,
    hmin = 0), under ISMPPRIOR = 1 for the priors of chains.prior_array / sd_prior_array.

    `pi` [kmax - kmin + 1] is the k-marginal (index k - kmin), `intended` the Poisson pk (or the
    flat prior) it should have been.  Given k, vp and sigma are uniform and the depths follow
    `fixed_k(k)` (a sampler_reference.FixedKPrior; for ENOS = 0 with L_b in place of hmx)."""

    def __init__(self, enos, prior, sd_prior, kmin, kmax, lam=None):
        self.enos, self.kmin, self.kmax, self.lam = bool(enos), int(kmin), int(kmax), lam
        self.prior, self.sd_prior = np.asarray(prior, dtype=np.float64), np.asarray(sd_prior, dtype=np.float64)
        self.hmin, self.hmx = float(prior[6]), float(prior[4])
        self.L = self.hmx - float(prior[2])                      # maxlim1 - minlim1
        if self.enos and self.hmin != 0.0:
            raise ValueError("the ENOS = 1 law is written for hmin = 0")
        self.ks = np.arange(self.kmin, self.kmax + 1)
        logw = [0.0]
        for k in self.ks[:-1]:
            qb, _ = move_probs(k, kmin, kmax)
            _, qd = move_probs(k + 1, kmin, kmax)
            step = log_pk(k + 1, lam) - log_pk(k, lam) + math.log(qb) - math.log(qd)
            if self.enos:
                step += (math.log((2 * k + 2) * (2 * k + 3) / (2 * k * (2 * k + 1))) + math.log(k)
                         + 2 * math.log(self.hmx) - 3 * math.log(self.L))
            logw.append(logw[-1] + step)
        logw = np.array(logw)
        if not self.enos:
            logw = logw + np.array([self.log_volume(k) for k in self.ks])
        self.log_pi = logw
        self.pi = _normalise(logw)
        self.intended = _normalise([log_pk(k, lam) for k in self.ks])

    def log_volume(self, k):
        """log (1 - (k - 1) hmin / L_b)_+^(k-1): -inf when k - 1 interfaces no longer fit."""
        if k == 1:
            return 0.0
        x = 1.0 - (k - 1) * self.hmin / self.L
        return (k - 1) * math.log(x) if x > 0.0 else -math.inf

    def ratio(self, k):
        """pi(k + 1) / pi(k)."""
        return math.exp(self.log_pi[k + 1 - self.kmin] - self.log_pi[k - self.kmin])

    def fixed_k(self, k):
        prior = self.prior.copy()
        if not self.enos:
            prior[4] = self.L                                    # births fill [0, L_b], not [0, hmx]
        return FixedKPrior(k, self.enos, prior, self.sd_prior)

    def sample(self, n, rng, ldk):
        """n exact draws: k [n] i32, voro [n, 2, ldk] (node 1 at depth 0, slots past k zero), sigma [n]."""
        k = rng.choice(self.ks, size=n, p=self.pi).astype(np.int32)
        voro, sigma = np.zeros((n, 2, ldk)), np.empty(n)
        for kv in np.unique(k):
            idx = np.flatnonzero(k == kv)
            depth, vp, sigma[idx] = self.fixed_k(int(kv)).sample(idx.size, rng)
            voro[idx, 0, 1:kv], voro[idx, 1, :kv] = depth, vp
        return k, voro, sigma

    def k_pvalue(self, k):
        """chi^2 p-value of the node counts k [N] against pi."""
        return chi2_pvalue(np.bincount(np.asarray(k) - self.kmin, minlength=self.ks.size), self.pi)

    def depth_pit(self, k, voro, rng):
        """Probability-integral transforms of every chain's depths, pooled: i.i.d. U(0, 1) exactly
        when each chain's depths follow the law given its k.  ENOS = 0: the order statistics
        y_i / (L_b - (k-1) hmin), which are a sorted sample of k - 1 i.i.d. uniforms.  ENOS = 1: the
        k - 1 interfaces are the even order statistics of 2k - 1 uniforms on [0, hmx]; given them
        the odd ones are independent uniforms within the k gaps, so drawing those restores the
        whole sorted sample of 2k - 1 uniforms."""
        k, voro = np.asarray(k), np.asarray(voro)
        out = []
        for kv in np.unique(k):
            z = voro[k == kv, 0, 1:kv]
            if self.enos:
                edges = np.concatenate([np.zeros((z.shape[0], 1)), z, np.full((z.shape[0], 1), self.hmx)], axis=1)
                odd = edges[:, :-1] + rng.random((z.shape[0], kv)) * np.diff(edges, axis=1)
                out += [z.ravel() / self.hmx, odd.ravel() / self.hmx]
            elif kv > 1:
                span = self.L - (kv - 1) * self.hmin
                out.append(((z - self.hmin * np.arange(1, kv)) / span).ravel())
        return np.concatenate(out) if out else np.empty(0)

    def vp_pit(self, k, voro):
        """(vp - vmin) / (vmax - vmin) of every node of every chain: i.i.d. U(0, 1) under the law."""
        k, voro = np.asarray(k), np.asarray(voro)
        vmin, vmax = float(self.prior[3]), float(self.prior[5])
        mask = np.arange(voro.shape[2])[None, :] < k[:, None]
        return (voro[:, 1, :][mask] - vmin) / (vmax - vmin)

    def pvalues(self, k, voro, rng, sigma=None):
        """{"k": chi^2, "depth", "vp" (and "sigma"): KS of the pooled transforms}."""
        p = {"k": self.k_pvalue(k), "depth": ks_uniform(self.depth_pit(k, voro, rng)),
             "vp": ks_uniform(self.vp_pit(k, voro))}
        if sigma is not None:
            p["sigma"] = ks_uniform((np.asarray(sigma) - self.sd_prior[1]) / (self.sd_prior[2] - self.sd_prior[1]))
        return p


def ks_uniform(x):
    """KS p-value of x against U(0, 1); 0 when any value lies outside [0, 1]."""
    x = np.asarray(x, dtype=np.float64)
    if x.size == 0:
        return 1.0
    if (x < 0.0).any() or (x > 1.0).any():
        return 0.0
    return float(stats.kstest(x, "uniform").pvalue)


def chi2_pvalue(counts, probs, min_expected=5.0):
    """Pearson chi^2 p-value of counts against cell probabilities, adjacent cells merged (in order)
    until each group expects at least `min_expected`.  A count in a cell of probability 0 gives 0."""
    counts, probs = np.asarray(counts, dtype=np.float64), np.asarray(probs, dtype=np.float64)
    if (counts[probs <= 0.0] > 0).any():
        return 0.0
    n = counts.sum()
    obs, exp, o, e = [], [], 0.0, 0.0
    for c, p in zip(counts, probs):
        o, e = o + c, e + n * p
        if e >= min_expected:
            obs.append(o)
            exp.append(e)
            o = e = 0.0
    if exp:
        obs[-1] += o
        exp[-1] += e
    if len(exp) < 2:
        return 1.0
    exp = np.array(exp)
    return float(stats.chisquare(obs, exp * (n / exp.sum())).pvalue)


# ---- the AR(1) move -----------------------------------------------------------------------------

def ar_pvalues(idxar, arpar, ar_prior):
    """{"idxar": two-sided binomial p of idxar against Bernoulli(1/2), "arpar": KS p of arpar given
    idxar = 1 against U[minlimar, maxlimar]}: the law of the AR move under a flat likelihood."""
    idxar, arpar = np.asarray(idxar), np.asarray(arpar)
    lo, hi = float(ar_prior[1]), float(ar_prior[2])
    if not np.isin(idxar, (0, 1)).all():
        return {"idxar": 0.0, "arpar": 0.0}
    return {"idxar": float(stats.binomtest(int(idxar.sum()), idxar.size, 0.5).pvalue),
            "arpar": ks_uniform((arpar[idxar == 1] - lo) / (hi - lo))}


def ar_sample(n, ar_prior, rng):
    """n exact draws (idxar i32, arpar) of the AR law; arpar = minlimar - 1 where idxar = 0, as the
    death move leaves it."""
    lo, hi = float(ar_prior[1]), float(ar_prior[2])
    idx = rng.integers(0, 2, n).astype(np.int32)
    return idx, np.where(idx == 1, rng.uniform(lo, hi, n), lo - 1.0)


# ---- the tempering swap round -------------------------------------------------------------------

def matchings(n):
    """Every perfect matching of 0..n-1 (one element left out when n is odd), as tuples of pairs."""
    def rec(rest):
        if len(rest) < 2:
            yield ()
            return
        a = rest[0]
        for i in range(1, len(rest)):
            for m in rec(rest[1:i] + rest[i + 1:]):
                yield ((a, rest[i]),) + m
    out = []
    for left in (range(n) if n % 2 else [None]):
        out += list(rec(tuple(r for r in range(n) if r != left)))
    return out


def assignments(n):
    """The n! assignments: a[r] = index into the ladder of the beta replica r holds."""
    return list(itertools.permutations(range(n)))


def swap_row(a, logL, ladder, matching):
    """Probabilities of the assignments after one round from assignment `a` with a given matching:
    {assignment: probability}; pair (i, j) exchanges its betas with min(1, exp((b_j - b_i)(L_i - L_j)))."""
    out = {tuple(a): 1.0}
    for i, j in matching:
        nxt = {}
        for s, p in out.items():
            bi, bj = ladder[s[i]], ladder[s[j]]
            acc = min(1.0, math.exp(min((bj - bi) * (logL[i] - logL[j]), 0.0)))
            t = list(s)
            t[i], t[j] = s[j], s[i]
            for state, q in ((tuple(t), acc), (s, 1.0 - acc)):
                if q > 0.0:
                    nxt[state] = nxt.get(state, 0.0) + p * q
        out = nxt
    return out


def swap_transition(logL, ladder, weights=None):
    """(assignments, P [n!, n!]): the one-round transition matrix over assignments, the matching
    drawn with `weights` (default: uniformly)."""
    n = len(logL)
    A, M = assignments(n), matchings(n)
    w = np.full(len(M), 1.0 / len(M)) if weights is None else np.asarray(weights, dtype=np.float64)
    index = {a: i for i, a in enumerate(A)}
    P = np.zeros((len(A), len(A)))
    for r, a in enumerate(A):
        for wm, m in zip(w, M):
            if wm == 0.0:
                continue
            for s, p in swap_row(a, logL, ladder, m).items():
                P[r, index[s]] += wm * p
    return A, P


def swap_stationary(logL, ladder):
    """(assignments, pi): pi(a) ∝ exp(sum_r ladder[a[r]] logL[r])."""
    A = assignments(len(logL))
    logw = np.array([sum(ladder[a[r]] * logL[r] for r in range(len(logL))) for a in A])
    return A, _normalise(logw)
