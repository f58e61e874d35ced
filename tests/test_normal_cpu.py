"""CPU checks of the per-model normal equations (DESIGN.md section 13): the reference normal_batch
against an exactly rounded contraction of the same rows within the reordering bound, its symmetry,
its zero rows and columns, the rays it leaves out, a huge residual; and the wrappers refuse bad
arguments before anything reaches the library."""
import math

import numpy as np
import pytest
import torch

from raytracerfortran_b200 import device, grad, raymod, workloads

from jac_reference import jacobian_batch
from normal_reference import normal_batch, reach_batch
from test_jac_cpu import _bits_equal, _forward

U = 2.0 ** -53


def _exact(v, z, n, so, sd, T, P, tobs, kmode=False):
    """math.fsum of the reached terms, and the sum of their magnitudes."""
    jv, jz, _, _ = jacobian_batch(v, z, n, so, sd, T, P, kmode=kmode)
    J = np.concatenate([jv, jz], axis=2)
    R = reach_batch(v, z, n, so, sd, T, kmode=kmode)
    B, S, Pc = J.shape
    A, Aabs = np.zeros((B, Pc, Pc)), np.zeros((B, Pc, Pc))
    g, gabs = np.zeros((B, Pc)), np.zeros((B, Pc))
    for b in range(B):
        for i in range(Pc):
            ti = [J[b, s, i] * float(tobs[s] - T[b, s]) for s in range(S) if R[b, s, i]]
            g[b, i], gabs[b, i] = math.fsum(ti), math.fsum(abs(t) for t in ti)
            for j in range(Pc):
                tij = [J[b, s, i] * J[b, s, j] for s in range(S) if R[b, s, i] and R[b, s, j]]
                A[b, i, j], Aabs[b, i, j] = math.fsum(tij), math.fsum(abs(t) for t in tij)
    return A, Aabs, g, gabs


def _check_against_exact(v, z, n, so, sd, T, P, tobs, kmode=False):
    JtJ, Jtr = normal_batch(v, z, n, so, sd, T, P, tobs=tobs, kmode=kmode)
    A, Aabs, g, gabs = _exact(v, z, n, so, sd, T, P, tobs, kmode=kmode)
    S = so.size
    assert np.all(np.abs(JtJ - A) <= S * U * Aabs * 1.01 + 1e-300)
    assert np.all(np.abs(Jtr - g) <= (S + 1) * U * gabs * 1.01 + 1e-300)
    assert _bits_equal(JtJ, JtJ.transpose(0, 2, 1))
    return JtJ, Jtr


@pytest.mark.parametrize("nl", [1, 2, 5, 12])
def test_reference_within_the_reordering_bound(nl):
    v, z, n = workloads.make_models(12, nl, 500 + nl)
    so, sd = workloads.make_sources(20, nl)
    T, P = _forward(v, z, n, so, sd)
    tobs = T[0] + np.random.default_rng(nl).normal(0, 0.01, so.size)
    _check_against_exact(v, z, n, so, sd, T, P, tobs)


def test_kmode_and_the_k1_fake_interface():
    k, vp, zi = workloads.make_transd_models(30, 8, 31, uniform_k=True)
    so, sd = workloads.make_sources(16, 31)
    T, P = _forward(vp, zi, k, so, sd, kmode=True)
    tobs = T[0] * 1.01
    JtJ, Jtr = _check_against_exact(vp, zi, k, so, sd, T, P, tobs, kmode=True)
    one = k == 1
    assert one.any()
    assert np.all(JtJ[one][:, 1:, :] == 0) and np.all(JtJ[one][:, :, 1:] == 0)
    assert np.all(Jtr[one][:, 1:] == 0) and np.all(JtJ[one][:, 0, 0] > 0)


def test_padding_gives_zero_rows_and_columns():
    rng = np.random.default_rng(3)
    B, ldv, ldz = 10, 12, 11
    v, z, _ = workloads.make_models(B, 6, 3)
    vp, zp = np.zeros((B, ldv)), np.full((B, ldz), 1e30)
    vp[:, :7], zp[:, :6] = v, z
    n = rng.integers(1, 7, B).astype(np.int32)
    so, sd = workloads.make_sources(18, 3)
    T, P = _forward(vp, zp, n, so, sd)
    JtJ, Jtr = _check_against_exact(vp, zp, n, so, sd, T, P, T[0])
    for b in range(B):
        dead = np.r_[np.arange(n[b] + 1, ldv), ldv + np.arange(n[b], ldz)]
        assert np.all(JtJ[b][dead] == 0) and np.all(JtJ[b][:, dead] == 0) and np.all(Jtr[b][dead] == 0)


def test_rays_that_did_not_converge_contribute_nothing():
    v, z, n = workloads.make_models(8, 5, 7)
    so, sd = workloads.make_sources(15, 7)
    T, P = _forward(v, z, n, so, sd)
    tobs = T[1] + 0.05
    T[0, :] = -999.0                       # a whole model
    T[3, 4] = -999.0                       # one ray: as if its source were absent
    JtJ, Jtr = normal_batch(v, z, n, so, sd, T, P, tobs=tobs)
    assert np.all(JtJ[0] == 0) and np.all(Jtr[0] == 0)
    keep = np.arange(so.size) != 4
    A, g = normal_batch(v[3:4], z[3:4], n[3:4], so[keep], sd[keep], T[3:4, keep], P[3:4, keep], tobs=tobs[keep])
    assert _bits_equal(JtJ[3], A[0]) and _bits_equal(Jtr[3], g[0])


def test_a_huge_residual_stays_in_its_terms():
    v, z, n = workloads.make_models(6, 4, 11)
    so, sd = workloads.make_sources(10, 11)
    T, P = _forward(v, z, n, so, sd)
    tobs = T[0].copy()
    tobs[6] = 1e300
    JtJ, Jtr = _check_against_exact(v, z, n, so, sd, T, P, tobs)
    base, _ = normal_batch(v, z, n, so, sd, T, P)
    assert _bits_equal(JtJ, base)
    assert np.all(np.isfinite(Jtr)) and np.abs(Jtr).max() > 1e290


def test_wrappers_refuse_bad_arguments():
    v, z, n = (torch.as_tensor(a) for a in workloads.make_models(3, 2, 1))
    n = n.to(torch.int32)
    so, sd = (torch.as_tensor(a) for a in workloads.make_sources(4, 1))
    T = torch.zeros((3, 4), dtype=torch.float64)
    with pytest.raises(ValueError, match="timeP must be"):
        device.dff_normal_device(v, z, n, so, sd, T[:, :3], T)
    with pytest.raises(ValueError, match="tobs must be"):
        device.dff_normal_device(v, z, n, so, sd, T, T, tobs=so[:3])
    with pytest.raises(ValueError, match="Jtr needs tobs"):
        device.dff_normal_device(v, z, n, so, sd, T, T, Jtr=torch.empty((3, 5), dtype=torch.float64))
    with pytest.raises(ValueError, match="JtJ must be"):
        device.dff_normal_device(v, z, n, so, sd, T, T, JtJ=torch.empty((3, 5, 4), dtype=torch.float64))
    with pytest.raises(ValueError, match="CUDA tensors"):
        device.dff_normal_device(v, z, n, so, sd, T, T)
    with pytest.raises(ValueError, match="CUDA tensors"):
        grad.normal_equations(v, z, n, so, sd)
    with pytest.raises(ValueError, match="tobs must be"):
        raymod.dff_batch_normal(v.numpy(), z.numpy(), n.numpy(), so.numpy(), sd.numpy(), tobs=np.zeros(3))
    with pytest.raises(ValueError, match="ldv must be"):
        raymod.dff_batch_normal(np.zeros((3, 256)), z.numpy(), n.numpy(), so.numpy(), sd.numpy())
