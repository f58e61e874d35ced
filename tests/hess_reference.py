"""Reference of the per-model second derivatives of the travel times (DESIGN.md section 14), for the tests.

hess_batch() restates the library's second-derivative kernel in numpy in its rounding order: every
operation is one correctly rounded binary64 operation (nothing fused), each ray's term of entry
(x, y) is (u_x u_y) alpha + band_xy with band_xy = 0.0 off the band, and the terms are added in
source order from +0.0 over the pairs the ray reaches (normal_reference.reach_batch).  So it is
comparable with the kernel bit for bit.  It reuses grad_reference's model columns and layer
lookup, and takes p from the caller.

closed_form() evaluates the same closed form in mpmath for one hp_reference.Ray, at any p, with the
magnitudes of its terms; `mutant` switches in one plausible mistake at a time, for the tests that
show the checks would catch it.
"""
import mpmath
import numpy as np
from mpmath import mpf

from grad_reference import NOT_CONVERGED, model_columns, which_layer
from normal_reference import reach_batch


def _layer(V, Z, Hc, i, n, q, d):
    """The kernel's per-layer values of layer i at ray parameter q (arrays over the models)."""
    v = V[:, i]
    vv = v * v
    pp = q * q
    cc = 1.0 - pp * vv
    c = np.sqrt(cc)
    c3 = cc * c
    h = np.where(i == n - 1, d - Z[:, max(i - 1, 0)], Hc[:, i])
    return {"u": (q * h) / c3, "xp": (h * v) / c3, "dvv": (h * (3.0 * cc - 1.0)) / ((vv * v) * c3),
            "e": 1.0 / (vv * c), "g": v / c}


def ray_terms(V, Z, Hc, NL, fake, ldv, ldz, t, q_p, ws, d):
    """The rank-one vectors u [B, P], alpha [B] and the weighted band [B, P, P] of one source's
    rays, as the kernel builds them."""
    B, LPa = V.shape
    P = ldv + ldz
    n = np.where(t == NOT_CONVERGED, 0, which_layer(Z, NL, d))
    q = np.where(n == 1, t, q_p)
    top, deep = n == 1, n >= 2
    u, band = np.zeros((B, P)), np.zeros((B, P, P))
    L = [_layer(V, Z, Hc, i, n, q, d) for i in range(LPa)]
    xp = L[0]["xp"]
    for i in range(1, LPa):
        xp = np.where(i < n, xp + L[i]["xp"], xp)
    al = np.where(deep, ws / xp, 0.0)
    real = deep & ~fake
    for i in range(min(ldv, LPa)):
        on = real & (i < n)
        u[:, i] = np.where(on, L[i]["u"], 0.0)
        band[:, i, i] = np.where(on, ws * L[i]["dvv"], 0.0)
        be = ws * L[i]["e"]
        if 1 <= i <= ldz:                                   # (V_i, z_{i-1})
            band[:, i, ldv + i - 1] = band[:, ldv + i - 1, i] = np.where(on, be, 0.0)
        if i < ldz:                                         # (V_i, z_i), i <= n - 2
            on2 = real & (i <= n - 2)
            band[:, i, ldv + i] = band[:, ldv + i, i] = np.where(on2, -be, 0.0)
    for j in range(min(ldz, LPa - 1)):
        u[:, ldv + j] = np.where(real & (j <= n - 2), q * (L[j]["g"] - L[j + 1]["g"]), 0.0)
    # k = 1 (kmode): column 0 takes both layers, no interface
    fd = deep & fake
    u[:, 0] = np.where(fd, L[0]["u"] + L[1]["u"], u[:, 0])
    band[:, 0, 0] = np.where(fd, ws * (L[0]["dvv"] + L[1]["dvv"]), band[:, 0, 0])
    # straight top-layer ray: 2 T / V_0^2 alone
    band[:, 0, 0] = np.where(top, ws * ((2.0 * t) / (V[:, 0] * V[:, 0])), band[:, 0, 0])
    return u, al, band


def hess_batch(vels, depths, nlayers, src_offset, src_depth, timeP, p, w, kmode=False):
    """H [B, P, P] = sum_s w[b, s] d2T[b, s], P = ldv + ldz, in the kernel's rounding order."""
    V, Z, Hc, NL, fake = model_columns(vels, depths, nlayers, kmode)
    T, Pq, W = (np.asarray(a, dtype=np.float64) for a in (timeP, p, w))
    so, sd = np.asarray(src_offset, np.float64), np.asarray(src_depth, np.float64)
    ldv, ldz = np.asarray(vels).shape[1], np.asarray(depths).shape[1]
    B, P = V.shape[0], ldv + ldz
    R = reach_batch(vels, depths, nlayers, so, sd, T, kmode=kmode)
    H = np.zeros((B, P, P))
    with np.errstate(all="ignore"):
        for s in range(so.size):
            u, al, band = ray_terms(V, Z, Hc, NL, fake, ldv, ldz, T[:, s], Pq[:, s], W[:, s], sd[s])
            term = (u[:, :, None] * u[:, None, :]) * al[:, None, None] + band
            H = H + np.where(R[:, s, :, None] & R[:, s, None, :], term, 0.0)
    return H


# ---- the closed form in mpmath ---------------------------------------------------------------
MUTANTS = ("no_rank_one", "band_sign", "x_not_slope", "uz_wrong_layer")


def closed_form(ray, p, mutant=None, T=None):
    """d2T of one hp_reference.Ray at ray parameter p by the closed form, in mpmath, over the ray's
    model columns (velocities then interfaces, as Ray.theta0 without R and d).  A straight ray's
    2 T / V_0^2 takes T if given (the forward's, as the kernel does), else T(p).  Returns (D2, M):
    the matrix and the magnitudes of its terms, |u_x u_y / X'| + |band|, with 3 cos^2 + 1 for
    |3 cos^2 - 1| and p (V_j / cos_j + V_j+1 / cos_j+1) for |u_zj|, as lists of lists of mpf."""
    with mpmath.workdps(max(mpmath.mp.dps, 50)):
        p = mpf(p)
        V, H = ray.column()
        n, nv, nz = ray.n, ray.nv, ray.nz
        P = nv + nz
        D2 = [[mpf(0)] * P for _ in range(P)]
        M = [[mpf(0)] * P for _ in range(P)]
        if n == 1:
            T = ray.T(p) if T is None else mpf(T)
            D2[0][0] = M[0][0] = 2 * T / V[0] ** 2
            return D2, M
        cos = [mpmath.sqrt(1 - (p * v) ** 2) for v in V]
        u = [mpf(0)] * P
        umag = [mpf(0)] * P
        band = [[mpf(0)] * P for _ in range(P)]
        bmag = [[mpf(0)] * P for _ in range(P)]
        for i in range(n):
            col = 0 if ray.fake else i
            u[col] += p * H[i] / cos[i] ** 3
            umag[col] += abs(p * H[i] / cos[i] ** 3)
            band[col][col] += H[i] * (3 * cos[i] ** 2 - 1) / (V[i] ** 3 * cos[i] ** 3)
            bmag[col][col] += H[i] * (3 * cos[i] ** 2 + 1) / (V[i] ** 3 * cos[i] ** 3)
        if not ray.fake:
            sgn = -1 if mutant == "band_sign" else 1
            for i in range(n):
                e = 1 / (V[i] ** 2 * cos[i])
                if i >= 1:
                    band[i][nv + i - 1] = band[nv + i - 1][i] = sgn * e
                    bmag[i][nv + i - 1] = bmag[nv + i - 1][i] = e
                if i <= n - 2:
                    band[i][nv + i] = band[nv + i][i] = -sgn * e
                    bmag[i][nv + i] = bmag[nv + i][i] = e
            for j in range(n - 1):
                k = min(j + 1, n - 2) if mutant == "uz_wrong_layer" else j
                u[nv + j] = p * (V[k] / cos[k] - V[k + 1] / cos[k + 1])
                umag[nv + j] = p * (V[j] / cos[j] + V[j + 1] / cos[j + 1])
        if mutant == "x_not_slope":
            xs = mpmath.fsum(h * v * p / c for v, h, c in zip(V, H, cos))
        else:
            xs = mpmath.fsum(h * v / c ** 3 for v, h, c in zip(V, H, cos))
        r1 = 0 if mutant == "no_rank_one" else 1
        for x in range(P):
            for y in range(P):
                D2[x][y] = band[x][y] + r1 * u[x] * u[y] / xs
                M[x][y] = bmag[x][y] + umag[x] * umag[y] / xs
        return D2, M
