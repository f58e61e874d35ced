"""Reference of the per-model Gauss-Newton normal equations (DESIGN.md section 13) in numpy, for the tests.

normal_batch() contracts the rows jac_reference.jacobian_batch() writes, J_s = [jvels[b, s] |
jdepths[b, s]], in source order from +0.0 with one correctly rounded multiply and one correctly
rounded add per term, and takes only the terms whose columns the ray reaches.  Every step is one
binary64 operation, so it is comparable with the library's normal-equations kernel bit for bit.
"""
import numpy as np

from grad_reference import NOT_CONVERGED, model_columns, which_layer
from jac_reference import jacobian_batch


def reach_batch(vels, depths, nlayers, src_offset, src_depth, timeP, kmode=False):
    """[B, S, P] bool: the columns of [vels | depths] ray (b, s) reaches: velocity column i < n
    (kmode k = 1: column 0 when n >= 1), depth column j <= n - 2 (none at k = 1), none for a ray
    with timeP = -999."""
    _, Z, _, NL, fake = model_columns(vels, depths, nlayers, kmode)
    T = np.asarray(timeP, np.float64)
    sd = np.asarray(src_depth, np.float64)
    ldv, ldz = np.asarray(vels).shape[1], np.asarray(depths).shape[1]
    n = np.stack([np.where(T[:, s] == NOT_CONVERGED, 0, which_layer(Z, NL, sd[s])) for s in range(sd.size)], 1) \
        if sd.size else np.zeros(T.shape, int)
    ne = np.where(fake[:, None], np.minimum(n, 1), n)
    level = np.concatenate([np.arange(ldv) + 1, np.arange(ldz) + 2])
    return level[None, None, :] <= ne[:, :, None]


def normal_batch(vels, depths, nlayers, src_offset, src_depth, timeP, p, tobs=None, kmode=False):
    """Returns (JtJ [B, P, P], Jtr [B, P] or None), P = ldv + ldz."""
    jv, jz, _, _ = jacobian_batch(vels, depths, nlayers, src_offset, src_depth, timeP, p, kmode=kmode)
    J = np.concatenate([jv, jz], axis=2)
    R = reach_batch(vels, depths, nlayers, src_offset, src_depth, timeP, kmode=kmode)
    T = np.asarray(timeP, np.float64)
    B, S, P = J.shape
    JtJ = np.zeros((B, P, P))
    Jtr = None if tobs is None else np.zeros((B, P))
    with np.errstate(all="ignore"):
        for s in range(S):
            Js, Rs = J[:, s], R[:, s]
            JtJ = JtJ + np.where(Rs[:, :, None] & Rs[:, None, :], Js[:, :, None] * Js[:, None, :], 0.0)
            if tobs is not None:
                r = tobs[s] - T[:, s]
                Jtr = Jtr + np.where(Rs, Js * r[:, None], 0.0)
    return JtJ, Jtr
