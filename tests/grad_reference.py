"""Reference of the travel-time gradient (DESIGN.md section 11) in numpy, for the tests.

grad_batch() evaluates the same expressions as the library's gradient kernel, in the same rounding
order: every numpy operation below is one correctly rounded binary64 operation, and nothing is
fused.  The sums run over the sources in order, one multiply and one add per term, so the result is
comparable bit for bit.  It takes p from the caller: the forward's p (the oracle's or the
library's), or a fully converged one (converged_ray).
"""
import numpy as np

FAKE_IFACE = 9999.9     # loglhood.f90:141
NOT_CONVERGED = -999.0  # sq:167-169


def model_columns(vels, depths, nlayers, kmode=False):
    """The layered columns the forward evaluates: V [B, LPa], Z [B, LPa], H [B, LPa], NL [B], fake [B]
    (InsertLayer, and in kmode the LOGLHOOD_RT mapping with its fake interface at k = 1)."""
    v, z = np.asarray(vels, dtype=np.float64), np.asarray(depths, dtype=np.float64)
    kk = np.asarray(nlayers, dtype=np.int64)
    B, ldv = v.shape
    ldz = z.shape[1]
    LP, LPa = max(ldv, 2) | 1, max(ldv, 2)
    if kmode:
        NL = np.where(kk > 1, kk - 1, 1)
    else:
        NL = np.maximum(kk, 0)
    NL = np.minimum(NL, LP - 1)
    fake = (kk <= 1) if kmode else np.zeros(B, bool)
    NL = np.where(fake, NL, np.minimum(NL, min(ldv - 1, ldz)))
    V, Z, H = np.ones((B, LPa)), np.zeros((B, LPa)), np.zeros((B, LPa))
    for b in range(B):
        n = int(NL[b])
        if fake[b]:
            V[b, :2] = v[b, 0]
            Z[b, 0] = FAKE_IFACE
        else:
            V[b, :n + 1] = v[b, :n + 1]
            Z[b, :n] = z[b, :n]
        H[b, 0] = Z[b, 0]
        H[b, 1:n] = Z[b, 1:n] - Z[b, :n - 1]
    return V, Z, H, NL, fake


def which_layer(Z, NL, d):
    """whichLayer (sq:9-32) for every model at source depth d: the layer count above the source."""
    col = np.arange(Z.shape[1])[None, :]
    diff = Z - d
    pos = (diff > 0.0) & (col < NL[:, None])
    first = np.argmax(pos, axis=1) + 1
    last = diff[np.arange(Z.shape[0]), np.maximum(NL - 1, 0)]
    n = np.where(pos.any(axis=1), first, np.where(last < 0.0, NL + 1, NL))
    return np.where(NL <= 0, 1, n)


def grad_batch(vels, depths, nlayers, src_offset, src_depth, timeP, p, w, kmode=False):
    """Vector-Jacobian product of the travel times.  Returns (gvels [B, ldv], gdepths [B, ldz],
    dtdr [B, S], dtdd [B, S])."""
    V, Z, H, NL, fake = model_columns(vels, depths, nlayers, kmode)
    T, P, W = (np.asarray(a, dtype=np.float64) for a in (timeP, p, w))
    so, sd = np.asarray(src_offset, np.float64), np.asarray(src_depth, np.float64)
    B, LPa = V.shape
    ldv, ldz = np.asarray(vels).shape[1], np.asarray(depths).shape[1]
    gv, gz = np.zeros((B, LPa)), np.zeros((B, LPa))
    dtdr, dtdd = np.zeros(T.shape), np.zeros(T.shape)
    rows = np.arange(B)
    VV = V * V
    with np.errstate(all="ignore"):
        for s in range(so.size):
            R, d = so[s], sd[s]
            t, q, ws = T[:, s], P[:, s], W[:, s]
            n = np.where(t == NOT_CONVERGED, 0, which_layer(Z, NL, d))
            pp = q * q
            top, deep = n == 1, n >= 2
            vl = V[rows, np.maximum(n - 1, 0)]
            dtdr[:, s] = np.where(n >= 1, q, 0.0)
            dtdd[:, s] = np.where(top, (d / np.sqrt(d * d + R * R)) / V[:, 0],
                                  np.where(deep, np.sqrt(1.0 - pp * (vl * vl)) / vl, 0.0))
            for i in range(int(n.max(initial=0))):
                act = i < n
                c = np.sqrt(1.0 - pp * VV[:, i])
                h = np.where(i == n - 1, d - Z[:, max(i - 1, 0)], H[:, i])
                term = np.where(top, -(t / V[:, 0]), -(h / (VV[:, i] * c)))
                gv[:, i] = np.where(act, gv[:, i] + ws * term, gv[:, i])
                if i + 1 < LPa:
                    c1 = np.sqrt(1.0 - pp * VV[:, i + 1])
                    dz = c / V[:, i] - c1 / V[:, i + 1]
                    gz[:, i] = np.where(i <= n - 2, gz[:, i] + ws * dz, gz[:, i])
    col = np.arange(LPa)[None, :]
    gvels = np.where(col <= NL[:, None], gv, 0.0)
    gvels[fake, 0] = gv[fake, 0] + gv[fake, 1]
    gvels[fake, 1:] = 0.0
    gdepths = np.where((col < NL[:, None]) & ~fake[:, None], gz, 0.0)
    out_v, out_z = np.zeros((B, ldv)), np.zeros((B, ldz))
    out_v[:, :min(ldv, LPa)] = gvels[:, :min(ldv, LPa)]
    out_z[:, :min(ldz, LPa)] = gdepths[:, :min(ldz, LPa)]
    return out_v, out_z, dtdr, dtdd


def column(vels, depths, nl, d):
    """InsertLayer for one model and source: (V[:n], H[:n])."""
    V, Z, H, NL, _ = model_columns(np.atleast_2d(vels), np.atleast_2d(depths), [nl])
    n = int(which_layer(Z, NL, d)[0])
    Hs = H[0, :n].copy()
    if n >= 2:
        Hs[n - 1] = d - Z[0, n - 2]
    return V[0, :n].copy(), Hs


def offset_of(p, V, H):
    """X(p) = sum H V p / sqrt(1 - p^2 V^2), the offset a ray of parameter p reaches."""
    return float(np.sum(H * V * p / np.sqrt(1.0 - p * p * V * V)))


def offset_slope(p, V, H):
    """X'(p) = sum H V / (1 - p^2 V^2)^(3/2)."""
    return float(np.sum(H * V / (1.0 - p * p * V * V) ** 1.5))


def converged_ray(vels, depths, nl, R, d):
    """An independent, fully converged solve of X(p) = R by bisection: returns (T, p)."""
    V, H = column(vels, depths, nl, d)
    if V.size == 1:
        D = np.sqrt(d * d + R * R)
        return D / V[0], (R / D) / V[0]
    lo, hi = 0.0, 1.0 / V.max()
    for _ in range(2000):
        mid = 0.5 * (lo + hi)
        if mid <= lo or mid >= hi:
            break
        if offset_of(mid, V, H) < R:
            lo = mid
        else:
            hi = mid
    p = lo if abs(offset_of(lo, V, H) - R) <= abs(offset_of(hi, V, H) - R) else hi
    return float(np.sum(H / (V * np.sqrt(1.0 - p * p * V * V)))), p
