"""An independent high-precision reference of the forward, the likelihood and the derivatives.

The physics of DESIGN.md sections 2, 11 and 12, evaluated in mpmath at DPS = 50 significant digits
from the reference's formulas (SURVEY.md): whichLayer (sq:9-32), InsertLayer (sq:38-69) with the
LOGLHOOD_RT model mapping (ll:127-146), the offset and the travel time (sq:184-202, sq:165-166),
and logL (ll:171-182, ll:194-196).  It imports nothing from the C oracle, grad_reference or
jac_reference and shares no rounding order with them or with the kernels:

* X(p), X'(p) and T(p) are evaluated in closed form; p* solves X(p) = R to the working precision;
* derivatives are mpmath.diff of G(theta; p) = p R + sum_i H_i(theta) eta_i(theta; p) at fixed p,
  eta_i = sqrt(1 - p^2 V_i^2) / V_i, theta = (velocities, interfaces, R, d): not the closed forms of
  rt_kernels.cu.  At p = p* the derivatives of G are those of the converged travel time T*(theta)
  (Fermat); mpmath.diff of T* itself checks that.

Every value comes with a first-order bound on the error a correct binary64 evaluation of it may
make, computed from the exact values at the same point.  One constant, C = 8, stands for "a few
roundings per quantity": a layer quantity such as H / (V cos) carries at most C u (1 + 1/cos^2)
relative error (u = 2^-53), because the rounding of 1 - p^2 V^2 is amplified by 1/cos^2 in a layer
close to critical; a sum of S terms adds S u times the sum of their magnitudes; logL over N
residuals carries (N + C) u (|log c| + ss / (2 sigma^2) + N |log sigma|).  Near-critical rays thus
get the looser bound they need and no other ray does.
"""
import functools
import math

import mpmath
from mpmath import mp, mpf

DPS = 50
U = 2.0 ** -53
C = 8
FAKE_IFACE = 9999.9      # ll:141
TOL = 0.1                # sq:234: the solver stops once |X(p) - R| < 0.1 m
NOT_CONVERGED = -999.0   # sq:167-169
DBL_MAX = 1.7976931348623157e308


def _hp(f):
    """Run f at DPS digits at least (mpmath.diff raises the precision further inside)."""
    @functools.wraps(f)
    def g(*a, **k):
        with mp.workdps(max(mp.dps, DPS)):
            return f(*a, **k)
    return g


def which_layer(depths, d):
    """sq:9-32: the number of layers above a source at depth d.  A source exactly on an interface
    counts as below it, except on the deepest interface; 1 for a bare half-space."""
    n_in, diff = 0, 0.0
    for i, z in enumerate(depths):
        n_in, diff = i + 1, z - d
        if diff > 0:
            break
    if len(depths) == 0:
        return 1
    return len(depths) + 1 if diff < 0 else n_in


def offset(p, V, H):
    """X(p) = sum H V p / sqrt(1 - p^2 V^2) (sq:184-202)."""
    return mpmath.fsum(h * v * p / mpmath.sqrt(1 - (p * v) ** 2) for v, h in zip(V, H))


def offset_slope(p, V, H):
    """X'(p) = sum H V / (1 - p^2 V^2)^(3/2) (sq:206-221)."""
    return mpmath.fsum(h * v / (1 - (p * v) ** 2) ** mpf(1.5) for v, h in zip(V, H))


def travel_time(p, V, H):
    """T(p) = sum H / (V sqrt(1 - p^2 V^2)) (sq:165-166)."""
    return mpmath.fsum(h / (v * mpmath.sqrt(1 - (p * v) ** 2)) for v, h in zip(V, H))


def solve_p(V, H, R):
    """The converged ray parameter p* on [0, 1/max V): X(p*) = R to the working precision.
    None when no ray in that interval reaches R, which happens only when every layer of the
    largest velocity has zero thickness (a source exactly on an interface above a faster layer)."""
    R = mpf(R)
    if len(V) == 1:                                  # the straight ray of the top layer (sq:94-97)
        return R / (mpmath.sqrt(H[0] ** 2 + R ** 2) * V[0])
    if R == 0:
        return mpf(0)
    vmax = max(V)
    lo, hi = mpf(0), 1 / vmax
    if all(h == 0 for v, h in zip(V, H) if v == vmax):
        lim = offset(hi, *zip(*[(v, h) for v, h in zip(V, H) if v != vmax])) if any(v != vmax for v in V) else 0
        if lim <= R:
            return None
    p = hi / 2
    eps = mpf(2) ** (-mp.prec + 4)
    for _ in range(10 * mp.prec):
        f = offset(p, V, H) - R
        if f == 0:
            return p
        if f < 0:
            lo = p
        else:
            hi = p
        q = p - f / offset_slope(p, V, H)
        if not lo < q < hi:
            q = (lo + hi) / 2
        if abs(q - p) <= eps * q or hi - lo <= eps * hi:
            return q
        p = q
    raise RuntimeError("p* did not converge")


class Ray:
    """One ray: a model row (vels, depths, nlayers; kmode: the vp nodes, ziface and k of
    LOGLHOOD_RT) and a source (R, d).  The parameters are theta = (the velocities the forward
    reads, the interfaces it reads, R, d); the layer count n is frozen at theta0, so derivatives
    at a source on an interface are one-sided (the side on which the source is below it)."""

    def __init__(self, vels, depths, nlayers, R, d, kmode=False, ldv=None, ldz=None):
        vels, depths = [float(x) for x in vels], [float(x) for x in depths]
        ldv = len(vels) if ldv is None else ldv
        ldz = len(depths) if ldz is None else ldz
        k = int(nlayers)
        self.fake = bool(kmode) and k <= 1                  # ll:138-145: vp(1) twice, z = 9999.9
        if self.fake:
            self.nv, self.nz = 1, 0
        else:
            nl = min(k - 1 if kmode else max(k, 0), ldv - 1, ldz)
            self.nv, self.nz = nl + 1, nl
        self.theta0 = vels[:self.nv] + depths[:self.nz] + [float(R), float(d)]
        self.n = which_layer(self._model(self.theta0)[1], float(d))
        self.iR, self.id = self.nv + self.nz, self.nv + self.nz + 1

    def _model(self, theta):
        if self.fake:
            return [theta[0], theta[0]], [mpf(FAKE_IFACE)]
        return list(theta[:self.nv]), list(theta[self.nv:self.nv + self.nz])

    def column(self, theta=None, n=None):
        """InsertLayer (sq:38-69): (V, H) of the n layers above the source, in mpf."""
        theta = [mpf(x) for x in (self.theta0 if theta is None else theta)]
        V, Z = self._model(theta)
        d = theta[-1]
        n = self.n if n is None else n
        if n == 1:
            return V[:1], [d]
        H = [Z[0]] + [Z[i] - Z[i - 1] for i in range(1, n - 1)] + [d - Z[n - 2]]
        return V[:n], H

    @_hp
    def X(self, p):
        return offset(mpf(p), *self.column())

    @_hp
    def T(self, p):
        return travel_time(mpf(p), *self.column())

    @_hp
    def p_star(self):
        return solve_p(*self.column(), self.theta0[-2])

    def T_star(self, theta, follow_layers=False):
        """The converged travel time as a function of theta (n re-evaluated if follow_layers)."""
        n = which_layer(self._model(theta)[1], theta[-1]) if follow_layers else None
        V, H = self.column(theta, n)
        return travel_time(solve_p(V, H, theta[-2]), V, H)

    def G(self, theta, p):
        V, H = self.column(theta)
        return p * theta[-2] + mpmath.fsum(h * mpmath.sqrt(1 - (p * v) ** 2) / v for v, h in zip(V, H))

    def _diff(self, f, col, direction=0):
        th = [mpf(x) for x in self.theta0]

        def g(x):
            t = list(th)
            t[col] = x
            return f(t)
        return mpmath.diff(g, th[col], direction=direction)

    @_hp
    def dG(self, p, cols):
        """mpmath.diff of G(theta; p) at fixed p over the parameter columns `cols`."""
        p = mpf(p)
        return [self._diff(lambda t: self.G(t, p), c) for c in cols]

    @_hp
    def dG_dp(self, p, cols):
        """d/dp of the columns of dG: how fast a derivative moves with the ray parameter."""
        p = mpf(p)
        return [mpmath.diff(lambda q: self._diff(lambda t: self.G(t, q), c), p) for c in cols]

    @_hp
    def dT_star(self, cols, follow_layers=False, directions=None):
        """mpmath.diff of the converged travel time T*(theta)."""
        dirs = directions or [0] * len(cols)
        return [self._diff(lambda t: self.T_star(t, follow_layers), c, s) for c, s in zip(cols, dirs)]

    # ---- error bounds of a binary64 evaluation, from the exact values -------------------------
    @_hp
    def _layers(self, p):
        p = mpf(p)
        V, H = self.column()
        cos = [mpmath.sqrt(1 - (p * v) ** 2) for v in V]
        return V, H, cos

    @_hp
    def t_bound(self, p):
        V, H, cos = self._layers(p)
        if self.n == 1:
            return float(C * U * travel_time(mpf(p), V, H))
        terms = [h / (v * c) for v, h, c in zip(V, H, cos)]
        return float(C * U * mpmath.fsum(t * (1 + 1 / c ** 2) for t, c in zip(terms, cos))
                     + len(terms) * U * mpmath.fsum(terms))

    @_hp
    def x_bound(self, p):
        V, H, cos = self._layers(p)
        terms = [h * v * mpf(p) / c for v, h, c in zip(V, H, cos)]
        return float(C * U * mpmath.fsum(t * (1 + 1 / c ** 2) for t, c in zip(terms, cos))
                     + len(terms) * U * mpmath.fsum(terms))

    @_hp
    def row_bounds(self, p, cols):
        """Per-column bounds of a binary64 row at p: the velocity terms H/(V^2 cos), the interface
        terms eta_j - eta_{j+1} (the two terms' bounds added), dT/dR = p (exact: the forward's p),
        dT/dd = eta_{n-1} (straight ray: d / (D V_0))."""
        V, H, cos = self._layers(p)
        n = self.n
        rel = [C * U * (1 + 1 / c ** 2) for c in cos]
        vel = [h / (v * v * c) for v, h, c in zip(V, H, cos)]
        eta = [c / v for v, c in zip(V, cos)]
        out = []
        for c in cols:
            if c < self.nv:
                layers = [0, 1][:n] if self.fake else ([c] if c < n else [])
                if n == 1:
                    b = 2 * C * U * vel[0]
                else:
                    b = mpmath.fsum(rel[i] * vel[i] for i in layers) + U * mpmath.fsum(vel[i] for i in layers)
            elif c < self.iR:
                j = c - self.nv
                b = rel[j] * eta[j] + rel[j + 1] * eta[j + 1] + U * abs(eta[j] - eta[j + 1]) if j <= n - 2 else 0
            elif c == self.iR:
                b = 0
            else:
                b = 2 * C * U * eta[0] if n == 1 else rel[n - 1] * eta[n - 1]
            out.append(float(b))
        return out


def ratio(got, exact, bound, noise=1e-30):
    """max |got - exact| / bound over the entries; the exact values' own noise (mpmath.diff at
    DPS digits) is allowed for at `noise` times the largest exact entry."""
    floor = noise * max([abs(float(e)) for e in exact] + [0.0])
    worst = 0.0
    for g, e, b in zip(got, exact, bound):
        err = abs(mpf(float(g)) - mpf(e))
        tol = b + floor
        r = float(err / tol) if tol > 0 else (0.0 if err == 0 else math.inf)
        worst = max(worst, r)
    return worst


# ---- the likelihood -------------------------------------------------------------------------
@_hp
def lognorm_overflows(n):
    """Whether (2 pi)^(N/2) rounds to +Inf in binary64 (ll:194): it does when it reaches
    DBL_MAX + ulp/2 = 2^1024 (1 - 2^-54)."""
    return (2 * mp.pi) ** (mpf(n) / 2) >= mpf(2) ** 1024 * (1 - mpf(2) ** -54)


@_hp
def loglhood(tpred, tobs, sigma, stable=False, idxar=0, arpar=0.0, armx=0.5):
    """logL of ll:194-196 (idxar = 1: the AR(1) residuals of ll:171-182) at the given times.

    Returns (logL, bound, rejected): logL exact (an mpf; -inf where the reference's constant
    LOG(1/(2 pi)^(N/2)) overflows, unless `stable`), the error bound of a binary64 evaluation, and
    whether the AR bound check rejects the state (then the reference returns -HUGE)."""
    N = len(tpred)
    res = [mpf(float(o)) - mpf(float(t)) for o, t in zip(tobs, tpred)]
    dar = [mpf(0)] * N
    if idxar == 1:
        for i in range(1, N - 1):
            dar[i] = mpf(float(arpar)) * res[i - 1]
    rejected = N > 0 and (max(dar) > mpf(float(armx)) or min(dar) < -mpf(float(armx)))
    ss = mpmath.fsum((r - a) ** 2 for r, a in zip(res, dar))
    s = mpf(float(sigma))
    logc = -(mpf(N) / 2) * mpmath.log(2 * mp.pi)
    if not stable and lognorm_overflows(N):
        return mpf("-inf"), 0.0, rejected
    val = logc - (ss / (2 * s * s) + N * mpmath.log(s))
    bound = (N + C) * U * (abs(logc) + ss / (2 * s * s) + N * abs(mpmath.log(s)))
    return val, float(bound), rejected


def as_double(x):
    """The binary64 a correctly rounded evaluation of the exact x gives (overflow: +-Inf)."""
    if mpmath.isinf(x):
        return float(x)
    return float(x) if abs(x) <= mpf(DBL_MAX) * (1 + mpf(2) ** -53) else math.copysign(math.inf, x)
