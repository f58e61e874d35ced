"""An independent reference of the device sampler's random deviates and of the fixed-k prior.

Two things about `chains.McmcGraph` (rtb200_mcmc_iterations_device) are checked with it:

* The deviates.  `draws` restates an iteration's draws in numpy from the counter layout that
  DESIGN.md section 2 and rt_kernels.cu document, on `oracle/tempering_ref.py`'s Philox4x32-10 and
  u01 (pinned by the Random123 known answers), not by porting the draw kernels:

      words      = Philox4x32-10(counter = (b, it & 0xffffffff, it >> 32, purpose),
                                 key = (seed & 0xffffffff, seed >> 32))
      u0, u1     = u01(r0, r1), u01(r2, r3)
      purpose    1: u_k, idel   2: u_z, u_v   3: u_acc_bd, u_gate   4: gauss (d0, d1)
                 5: u_acc_sd, u_choice   6: u_prop_ar, u_acc_ar   7: gauss_ar (g0, g1)
                 16 + m: sweep move m (dev from u0, u_acc = u1)

  Uniforms, idel, ivo, iwhich and the ENOS = 1 depth deviate are exact and compared bit for bit.
  The Box-Muller normals and the Cauchy steps go through the device's log, cospi and tan, so
  `gauss_exact` and `cauchy_exact` give their values in mpmath with a first-order bound on the
  error of a binary64 evaluation, computed from the exact values at the same point.
* The target.  Under ISMPPRIOR = 1 (logL = 1) a correct fixed-dimension move leaves the prior
  invariant.  `FixedKPrior` samples the fixed-k prior exactly and gives its marginal CDFs, and
  `check_stationary` returns one KS p-value per marginal from one state per chain, so the samples
  are independent and the p-values exact.

The maximum ulp errors are those the CUDA C++ Programming Guide lists in its table of
double-precision mathematical standard library functions (appendix "Mathematical Functions"):
log 1, cospi 2, tan 2; sqrt is correctly rounded.  One ulp of x is at most 2u|x|, u = 2^-53.
"""
import math

import mpmath
import numpy as np
from mpmath import mp, mpf
from scipy import stats

from oracle.tempering_ref import philox4x32_10, u01

DPS = 50
U = 2.0 ** -53
PI_HAT = 3.141592653589793          # the binary64 pi of the sweep draw kernel and chains.cauchy_deviates
ULP_LOG, ULP_COSPI, ULP_TAN = 1, 2, 2
SWEEP_PURPOSE0 = 16
_MASK = 0xFFFFFFFF
_SWEEP_ROWS = 64                    # sweep moves per Philox batch: bounds the temporaries at large B


def words(seed, it, chain, purpose):
    """The four Philox4x32-10 output words of (chain, iteration, purpose) under `seed`; chain and
    purpose may be arrays (broadcast), seed and it Python integers below 2^64."""
    seed, it = int(seed), int(it)
    return philox4x32_10((np.asarray(chain, dtype=np.uint64), it & _MASK, (it >> 32) & _MASK,
                          np.asarray(purpose, dtype=np.uint64)), (seed & _MASK, (seed >> 32) & _MASK))


def uniforms(r):
    """(u0, u1) from the four words of one Philox call."""
    return u01(r[0], r[1]), u01(r[2], r[3])


def cospi(x):
    """cos(pi x) in float64 for x in [0, 2), with the reduction done exactly (2 - x, 1 - r and
    0.5 - r are exact by Sterbenz), so only the final argument pi*r is rounded and the result is
    accurate relative to itself also next to the zeros at x = 1/2 and 3/2."""
    x = np.asarray(x, dtype=np.float64)
    r = np.where(x > 1.0, 2.0 - x, x)
    sign = np.where(r > 0.5, -1.0, 1.0)
    r = np.where(r > 0.5, 1.0 - r, r)
    return sign * np.where(r <= 0.25, np.cos(np.pi * r), np.sin(np.pi * (0.5 - r)))


def box_muller(d0, d1):
    """The normal deviate of a uniform pair in float64: sqrt(-2 ln(1 - d0)) cos(pi * 2 d1)."""
    return np.sqrt(-2.0 * np.log(1.0 - d0)) * cospi(2.0 * d1)


def cauchy(u0):
    """The Cauchy step of PROPOSAL in float64: tan(pi_hat (u0 - 1/2))."""
    return np.tan(PI_HAT * (u0 - 0.5))


def idel_of(a1, k):
    """The node a death removes, 2 + floor(a1 * max(k - 1, 1)) with the product rounded to binary64.

    With n = max(k - 1, 1) and a1 <= 1 - 2^-53, the exact product is n - n 2^-53 or less.  Below n
    the doubles are spaced s = 2^(e-52) for 2^e < n < 2^(e+1) (n a multiple of s), and that product
    is more than s/2 below n, so it rounds to n - s at most; for n = 2^e the product is itself a
    double.  So the rounded product never reaches n and idel never exceeds k.

    It is not always the exact floor, though: the product can lie within half an ulp below a
    smaller integer and round up to it.  At k = 4, a1 = 6004799503160661 * 2^-53 gives the exact
    product 2 - 2^-53, a tie that rounds to 2, so idel is 4 where the exact floor gives 3.  This
    happens for fewer than n of the 2^53 values of a1 and is what the device computes, so the
    restatement keeps the rounded product."""
    n = np.maximum(np.asarray(k, dtype=np.int64) - 1, 1).astype(np.float64)
    return (2 + np.floor(a1 * n)).astype(np.int32)


def draws(seed, it, k, pos, M, enos, k_sweep=None):
    """The deviates of iteration `it` (the counter's value when it starts) for chains b = 0..B-1:
    a dict with the keys of chains.mcmc_workspace_views (u_k, idel, u_z, u_v, u_acc_bd, u_gate,
    gauss, u_acc_sd, u_choice, u_prop_ar, u_acc_ar, gauss_ar [B]; ivo, iwhich, dev, u_acc [M, B]),
    plus the uniform pairs the two normals came from (d0, d1, g0, g1) and the sweep's u0.

    k [B] is the node count the iteration starts with (idel); the sweep's schedule uses the counts
    after the birth/death move, `k_sweep` (default k).  pos [B] is each chain's sweep position:
    move m of chain b is step j = (pos + m) mod max(2 k - 1, 1) + 1 of its sweep, ivo = j // 2 + 1,
    iwhich = j mod 2 + 1.  With ENOS = 1 a depth move (iwhich = 1) takes u0 itself."""
    k = np.asarray(k, dtype=np.int64)
    ks = k if k_sweep is None else np.asarray(k_sweep, dtype=np.int64)
    pos = np.asarray(pos, dtype=np.int64)
    B, M = k.size, int(M)
    b = np.arange(B, dtype=np.uint64)
    (a0, a1), (b0, b1), (c0, c1), (d0, d1), (e0, e1), (f0, f1), (g0, g1) = (
        uniforms(words(seed, it, b, p)) for p in range(1, 8))
    out = {"u_k": a0, "idel": idel_of(a1, k), "u_z": b0, "u_v": b1, "u_acc_bd": c0, "u_gate": c1,
           "gauss": box_muller(d0, d1), "u_acc_sd": e0, "u_choice": e1, "u_prop_ar": f0, "u_acc_ar": f1,
           "gauss_ar": box_muller(g0, g1), "d0": d0, "d1": d1, "g0": g0, "g1": g1}
    period = np.maximum(2 * ks - 1, 1)
    m = np.arange(M, dtype=np.int64)[:, None]
    j = (pos[None, :] + m) % period[None, :] + 1
    out["ivo"] = (j // 2 + 1).astype(np.int32)
    out["iwhich"] = (j % 2 + 1).astype(np.int32)
    u0 = np.empty((M, B))
    u1 = np.empty((M, B))
    for m0 in range(0, M, _SWEEP_ROWS):
        rows = np.arange(m0, min(M, m0 + _SWEEP_ROWS), dtype=np.uint64)[:, None]
        u0[m0:m0 + rows.size], u1[m0:m0 + rows.size] = uniforms(words(seed, it, b[None, :], SWEEP_PURPOSE0 + rows))
    out["u0"], out["u_acc"] = u0, u1
    out["dev"] = np.where((out["iwhich"] == 1) & bool(enos), u0, cauchy(u0))
    return out


# ---- exact transforms with bounds ---------------------------------------------------------------

def gauss_exact(d0, d1):
    """(value, bound) of sqrt(-2 ln(1 - d0)) cospi(2 d1) at 50 digits.  1 - d0 and 2 d1 are exact
    in binary64.  A correct evaluation errs by at most: log's ULP_LOG ulps, which the square root
    halves, ULP_LOG u |g|; the square root's rounding, u |g|; cospi's ULP_COSPI ulps, 2 ULP_COSPI u |g|
    plus ULP_COSPI subnormal ulps where cospi is 0; the product's rounding, u |g|."""
    with mp.workdps(DPS):
        rad = mpmath.sqrt(-2 * mpmath.log(1 - mpf(float(d0))))
        c = mpmath.cospi(2 * mpf(float(d1)))
        g = rad * c
        bound = (ULP_LOG + 1 + 2 * ULP_COSPI + 1) * U * abs(g) + ULP_COSPI * 2.0 ** -1074 * rad
        return float(g), float(bound)


def cauchy_exact(u0):
    """(value, bound) of tan(pi_hat (u0 - 1/2)) at 50 digits, pi_hat the binary64 constant.
    u0 - 1/2 is exact; the rounded product y moves tan by (1 + t^2) |y| u, and tan itself errs by
    ULP_TAN ulps, 2 ULP_TAN u |t|.  The first term grows without bound toward u0 -> 0 and 1, where
    tan is ill-conditioned."""
    with mp.workdps(DPS):
        y = mpf(PI_HAT) * (mpf(float(u0)) - mpf(0.5))
        t = mpmath.tan(y)
        bound = (1 + t * t) * abs(y) * U + 2 * ULP_TAN * U * abs(t)
        return float(t), float(bound)


def gauss_bound64(g, rad):
    """gauss_exact's bound from float64 values (for checking every deviate, not just a sample)."""
    return (ULP_LOG + 1 + 2 * ULP_COSPI + 1) * U * np.abs(g) + ULP_COSPI * 2.0 ** -1074 * rad


def cauchy_bound64(u0):
    """cauchy_exact's bound from float64 values."""
    y = PI_HAT * (u0 - 0.5)
    t = np.tan(y)
    return (1.0 + t * t) * np.abs(y) * U + 2 * ULP_TAN * U * np.abs(t)


def extremes(d0=None, d1=None, u0=None):
    """Indices of the draws where the transforms are hardest: the largest d0 (deepest log), d1
    nearest 1/4 and 3/4 (cospi's zeros), u0 nearest 0 and 1 (tan's poles)."""
    idx = []
    if d0 is not None:
        idx += [int(np.argmax(d0))]
    if d1 is not None:
        idx += [int(np.argmin(np.abs(d1 - 0.25))), int(np.argmin(np.abs(d1 - 0.75)))]
    if u0 is not None:
        idx += [int(np.argmin(u0)), int(np.argmax(u0))]
    return idx


def check_normals(got, d0, d1, n_sample, rng):
    """The worst error/bound ratios of normal deviates `got` made from the pairs (d0, d1): against
    mpmath on n_sample of them plus the extremes, against numpy float64 on all of them (where the
    allowance is twice the bound).  Returns (ratio_mpmath, ratio_numpy)."""
    got, d0, d1 = (np.asarray(a, dtype=np.float64).ravel() for a in (got, d0, d1))
    idx = np.unique(np.concatenate([rng.choice(got.size, min(n_sample, got.size), replace=False),
                                    extremes(d0=d0, d1=d1)]))
    worst = 0.0
    for i in idx:
        v, bnd = gauss_exact(d0[i], d1[i])
        err = abs(got[i] - v)
        worst = max(worst, err / bnd if bnd > 0 else (0.0 if err == 0 else math.inf))
    ref = box_muller(d0, d1)
    bnd = gauss_bound64(ref, np.sqrt(-2.0 * np.log(1.0 - d0)))
    err = np.abs(got - ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bnd > 0, err / (2 * bnd), np.where(err == 0, 0.0, np.inf))
    return worst, float(r.max(initial=0.0))


def check_cauchy(got, u0, n_sample, rng):
    """check_normals for Cauchy steps `got` made from u0."""
    got, u0 = (np.asarray(a, dtype=np.float64).ravel() for a in (got, u0))
    if got.size == 0:
        return 0.0, 0.0
    idx = np.unique(np.concatenate([rng.choice(got.size, min(n_sample, got.size), replace=False),
                                    extremes(u0=u0)]))
    worst = 0.0
    for i in idx:
        v, bnd = cauchy_exact(u0[i])
        err = abs(got[i] - v)
        worst = max(worst, err / bnd if bnd > 0 else (0.0 if err == 0 else math.inf))
    ref = cauchy(u0)
    bnd = cauchy_bound64(u0)
    err = np.abs(got - ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bnd > 0, err / (2 * bnd), np.where(err == 0, 0.0, np.inf))
    return worst, float(r.max(initial=0.0))


EXACT_KEYS = ("u_k", "idel", "u_z", "u_v", "u_acc_bd", "u_gate", "u_acc_sd", "u_choice", "u_prop_ar",
              "u_acc_ar", "ivo", "iwhich", "u_acc")


def compare_draws(got, want, enos, n_sample=2000, rng=None):
    """Compare an iteration's deviates `got` (workspace views as numpy, or a mutant stream) with
    `want = draws(...)`.  Returns a report: `mismatch` lists the keys that differ in any bit
    (the exact keys and the ENOS depth deviates), `ratio` the worst error/bound of gauss, gauss_ar
    and the Cauchy dev against mpmath and against numpy.  ok iff nothing mismatches and every ratio
    is at most 1."""
    rng = np.random.default_rng(0) if rng is None else rng
    mismatch = [n for n in EXACT_KEYS
                if not np.array_equal(np.asarray(got[n]).view(np.uint8), np.asarray(want[n]).view(np.uint8))]
    enos_dev = (want["iwhich"] == 1) & bool(enos)
    if not np.array_equal(np.asarray(got["dev"])[enos_dev].view(np.uint64), want["dev"][enos_dev].view(np.uint64)):
        mismatch.append("dev (ENOS)")
    ratio = {"gauss": check_normals(got["gauss"], want["d0"], want["d1"], n_sample, rng),
             "gauss_ar": check_normals(got["gauss_ar"], want["g0"], want["g1"], n_sample, rng),
             "dev": check_cauchy(np.asarray(got["dev"])[~enos_dev], want["u0"][~enos_dev], n_sample, rng)}
    ok = not mismatch and all(r <= 1.0 for pair in ratio.values() for r in pair)
    return {"ok": ok, "mismatch": mismatch, "ratio": ratio}


# ---- the fixed-k prior --------------------------------------------------------------------------

class FixedKPrior:
    """The prior of k-node models under chains.prior_array / sd_prior_array, for fixed k.

    Node 1 sits at depth 0; the k - 1 interface depths z_2 < ... < z_k lie in [0, hmx].
    ENOS = 0: every interface at least hmin below the one above (CHECKBOUNDS2), otherwise uniform,
    so y_j = z_{j+1} - j hmin are the order statistics of k - 1 uniforms on [0, hmx - (k - 1) hmin]
    and y_j / (hmx - (k - 1) hmin) ~ Beta(j, k - j).
    ENOS = 1 (even-numbered order statistics, needs hmin = 0): z_{j+1} is the 2j-th of 2k - 1
    uniforms on [0, hmx], so the k gaps / hmx are Dirichlet(2, ..., 2) and z_{j+1} / hmx ~
    Beta(2j, 2(k - j)).
    vp is uniform on [vmin, vmax] for every node, sigma on [sdmn, sdmx]."""

    def __init__(self, k, enos, prior, sd_prior):
        self.k, self.enos = int(k), bool(enos)
        self.hmx, self.vmin, self.vmax, self.hmin = float(prior[4]), float(prior[3]), float(prior[5]), float(prior[6])
        self.sdmn, self.sdmx = float(sd_prior[1]), float(sd_prior[2])
        if self.enos and self.hmin != 0.0:
            raise ValueError("the ENOS = 1 target is written for hmin = 0")

    def sample(self, n, rng):
        """n exact draws: (depth [n, k-1] = z_2..z_k, vp [n, k], sigma [n])."""
        k = self.k
        if self.enos:
            gaps = rng.gamma(2.0, size=(n, k))
            depth = self.hmx * np.cumsum(gaps, axis=1)[:, :k - 1] / gaps.sum(axis=1, keepdims=True)
        else:
            span = self.hmx - (k - 1) * self.hmin
            depth = np.sort(rng.uniform(0.0, span, (n, k - 1)), axis=1) + self.hmin * np.arange(1, k)
        return depth, rng.uniform(self.vmin, self.vmax, (n, k)), rng.uniform(self.sdmn, self.sdmx, n)

    def depth_cdf(self, j):
        """CDF of z_{j+1}, j = 1..k-1."""
        k = self.k
        if self.enos:
            return stats.beta(2 * j, 2 * (k - j), scale=self.hmx).cdf
        span = self.hmx - (k - 1) * self.hmin
        return stats.beta(j, k - j, loc=j * self.hmin, scale=span).cdf

    def vp_cdf(self):
        return stats.uniform(self.vmin, self.vmax - self.vmin).cdf

    def sigma_cdf(self):
        return stats.uniform(self.sdmn, self.sdmx - self.sdmn).cdf


def states_of(voro, k):
    """(depth [B, k-1], vp [B, k]) of the chains' sorted nodes: voro [B, 2, ldk]."""
    voro = np.asarray(voro)
    return voro[:, 0, 1:k], voro[:, 1, :k]


def check_stationary(states, target):
    """Per-marginal KS p-values of one state per chain against `target` (a FixedKPrior).
    states: a dict with any of depth [N, k-1], vp [N, k], sigma [N].  Keys of the result: depth2 ..
    depthk (node numbers), vp1 .. vpk, sigma."""
    p = {}
    if "depth" in states:
        for j in range(1, target.k):
            p[f"depth{j + 1}"] = stats.kstest(states["depth"][:, j - 1], target.depth_cdf(j)).pvalue
    if "vp" in states:
        for i in range(target.k):
            p[f"vp{i + 1}"] = stats.kstest(states["vp"][:, i], target.vp_cdf()).pvalue
    if "sigma" in states:
        p["sigma"] = stats.kstest(states["sigma"], target.sigma_cdf()).pvalue
    return p
