"""Reference of the per-ray Jacobian of the travel times (DESIGN.md section 12) in numpy, for the tests.

jacobian_batch() writes, per ray, the terms grad_reference.grad_batch() sums over the sources, with
the same correctly rounded binary64 operations in the same order (nothing fused), so it is
comparable with the library's Jacobian kernel bit for bit.  It reuses grad_reference's model columns
and layer lookup, and takes p from the caller.
"""
import numpy as np

from grad_reference import NOT_CONVERGED, model_columns, which_layer


def jacobian_batch(vels, depths, nlayers, src_offset, src_depth, timeP, p, kmode=False):
    """The terms grad_batch sums, per ray.  Returns (jvels [B, S, ldv], jdepths [B, S, ldz],
    dtdr [B, S], dtdd [B, S]); at k = 1 (kmode) jvels[b, s, 0] is the one rounded sum of both
    layers' terms."""
    V, Z, H, NL, fake = model_columns(vels, depths, nlayers, kmode)
    T, P = (np.asarray(a, dtype=np.float64) for a in (timeP, p))
    so, sd = np.asarray(src_offset, np.float64), np.asarray(src_depth, np.float64)
    B, LPa = V.shape
    S = so.size
    ldv, ldz = np.asarray(vels).shape[1], np.asarray(depths).shape[1]
    jv, jz = np.zeros((B, S, LPa)), np.zeros((B, S, LPa))
    dtdr, dtdd = np.zeros(T.shape), np.zeros(T.shape)
    rows = np.arange(B)
    VV = V * V
    with np.errstate(all="ignore"):
        for s in range(S):
            R, d = so[s], sd[s]
            t, q = T[:, s], P[:, s]
            n = np.where(t == NOT_CONVERGED, 0, which_layer(Z, NL, d))
            pp = q * q
            top, deep = n == 1, n >= 2
            vl = V[rows, np.maximum(n - 1, 0)]
            dtdr[:, s] = np.where(n >= 1, q, 0.0)
            dtdd[:, s] = np.where(top, (d / np.sqrt(d * d + R * R)) / V[:, 0],
                                  np.where(deep, np.sqrt(1.0 - pp * (vl * vl)) / vl, 0.0))
            tv, eta = np.zeros((B, LPa)), np.zeros((B, LPa))
            for i in range(LPa):
                c = np.sqrt(1.0 - pp * VV[:, i])
                h = np.where(i == n - 1, d - Z[:, max(i - 1, 0)], H[:, i])
                tv[:, i] = np.where(i < n, np.where(top, -(t / V[:, 0]), -(h / (VV[:, i] * c))), 0.0)
                eta[:, i] = c / V[:, i]
            for j in range(LPa - 1):
                jz[:, s, j] = np.where(j <= n - 2, eta[:, j] - eta[:, j + 1], 0.0)
            jv[:, s] = tv
            jv[fake, s, 0] = np.where(n[fake] >= 1, tv[fake, 0] + np.where(n[fake] >= 2, tv[fake, 1], 0.0), 0.0)
    col = np.arange(LPa)[None, None, :]
    jv = np.where(fake[:, None, None] & (col > 0), 0.0, jv)
    jz[fake] = 0.0
    out_v, out_z = np.zeros((B, S, ldv)), np.zeros((B, S, ldz))
    out_v[:, :, :min(ldv, LPa)] = jv[:, :, :min(ldv, LPa)]
    out_z[:, :, :min(ldz, LPa)] = jz[:, :, :min(ldz, LPa)]
    return out_v, out_z, dtdr, dtdd
