"""CPU checks of the per-ray Jacobian (DESIGN.md section 12): the reference jacobian_batch,
contracted with weights in source order, is grad_batch bit for bit, which ties it to the reference
test_grad_cpu.py checks against finite differences; and the wrappers refuse bad arguments before
anything reaches the library."""
import numpy as np
import pytest
import torch

import oracle
from raytracerfortran_b200 import _lib, device, grad, raymod, workloads

from grad_reference import grad_batch
from jac_reference import jacobian_batch


def _bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _contract(jv, jz, w):
    """sum_s w[b, s] J[b, s, :], one rounded multiply and one rounded add per term, in source order."""
    gv, gz = np.zeros(jv[:, 0].shape), np.zeros(jz[:, 0].shape)
    for s in range(w.shape[1]):
        gv = gv + w[:, s, None] * jv[:, s]
        gz = gz + w[:, s, None] * jz[:, s]
    return gv, gz


def _forward(v, z, n, so, sd, kmode=False):
    """The forward's own T and p: the oracle's (bit-identical to the library's)."""
    if not kmode:
        r = oracle.dff_batch(v, z, n, so, sd, want_p=True)
        return r["timeP"], r["p"]
    T, P = np.empty((v.shape[0], so.size)), np.empty((v.shape[0], so.size))
    for b in range(v.shape[0]):
        k = int(n[b])
        vv, zz, nl = (np.array([v[b, 0], v[b, 0]]), np.array([9999.9]), 1) if k <= 1 else (v[b, :k], z[b, :k - 1], k - 1)
        r = oracle.dff_batch(vv[None], zz[None], np.array([nl], np.int32), so, sd, want_p=True)
        T[b], P[b] = r["timeP"][0], r["p"][0]
    return T, P


def _check_contraction(v, z, n, so, sd, T, P, w, kmode=False):
    jv, jz, dr, dd = jacobian_batch(v, z, n, so, sd, T, P, kmode=kmode)
    gv, gz, gdr, gdd = grad_batch(v, z, n, so, sd, T, P, w, kmode=kmode)
    cv, cz = _contract(jv, jz, w)
    assert _bits_equal(cv, gv) and _bits_equal(cz, gz)
    assert _bits_equal(dr, gdr) and _bits_equal(dd, gdd)
    return jv, jz


@pytest.mark.parametrize("nl", [1, 2, 5, 10, 25, 50])
def test_contraction_is_grad_batch(nl):
    v, z, n = workloads.make_models(40, nl, 300 + nl)
    so, sd = workloads.make_sources(24, nl)
    T, P = _forward(v, z, n, so, sd)
    T[np.random.default_rng(nl).random(T.shape) < 0.05] = -999.0       # rays that did not converge
    w = np.random.default_rng(nl).normal(size=T.shape)
    jv, jz = _check_contraction(v, z, n, so, sd, T, P, w)
    assert np.all(jv[T == -999.0] == 0) and np.all(jz[T == -999.0] == 0)


def test_contraction_padded_ragged_rows():
    rng = np.random.default_rng(21)
    B, ldv, ldz = 17, 16, 14
    v, z, _ = workloads.make_models(B, 13, 21)
    n = rng.integers(0, 14, B).astype(np.int32)
    vp = np.zeros((B, ldv))
    vp[:, :14] = v
    zp = np.full((B, ldz), 1e30)
    zp[:, :13] = z
    so, sd = workloads.make_sources(20, 21)
    T, P = _forward(vp, zp, n, so, sd)
    _check_contraction(vp, zp, n, so, sd, T, P, rng.normal(size=T.shape))


def test_contraction_kmode():
    k, vp, zi = workloads.make_transd_models(60, 12, 31, uniform_k=True)
    so, sd = workloads.make_sources(16, 31)
    T, P = _forward(vp, zi, k, so, sd, kmode=True)
    rng = np.random.default_rng(31)
    keep = k >= 2                           # random weights: k = 1 sums its two layers in a different order
    _check_contraction(vp[keep], zi[keep], k[keep], so, sd, T[keep], P[keep], rng.normal(size=T[keep].shape),
                       kmode=True)
    for s in range(so.size):                # one-hot weights: every state, k = 1 included
        w = np.zeros(T.shape)
        w[:, s] = 1.0
        _check_contraction(vp, zi, k, so, sd, T, P, w, kmode=True)


def test_half_space_row():
    """k = 1: dT/dV_0 is the sum of both layers' terms, nothing else is non-zero."""
    vp, zi, k = np.full((1, 3), 2500.0), np.zeros((1, 2)), np.array([1], np.int32)
    so, sd = np.array([100.0, 300.0]), np.array([50.0, 20000.0])
    T, P = _forward(vp, zi, k, so, sd, kmode=True)
    jv, jz, _, _ = jacobian_batch(vp, zi, k, so, sd, T, P, kmode=True)
    assert jv[0, 0, 0] == -(T[0, 0] / 2500.0) + 0.0
    assert np.all(jv[0, :, 1:] == 0) and np.all(jz == 0)
    # the deep source crosses the fake interface: two velocity terms of the same layer
    assert jv[0, 1, 0] < 0 and np.isfinite(jv[0, 1, 0])


# ---- argument checks: the wrappers refuse bad arguments before anything reaches the library ----

@pytest.fixture
def no_library(monkeypatch):
    def boom():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", boom)


def _cpu_batch(B=3, ldv=4, S=5):
    f = torch.float64
    return (torch.ones(B, ldv, dtype=f), torch.ones(B, ldv - 1, dtype=f), torch.full((B,), ldv - 1, dtype=torch.int32),
            torch.ones(S, dtype=f), torch.ones(S, dtype=f))


@pytest.mark.parametrize("bad", ["timeP", "p", "jvels", "jdepths", "dtdr", "nlayers", "src", "vels"])
def test_device_wrapper_rejects_bad_shapes(no_library, bad):
    v, z, n, so, sd = _cpu_batch()
    t = p = torch.zeros(3, 5, dtype=torch.float64)
    kw = {}
    if bad == "timeP":
        t = torch.zeros(5, 3, dtype=torch.float64)
    elif bad == "p":
        p = torch.zeros(3, 4, dtype=torch.float64)
    elif bad == "jvels":
        kw["jvels"] = torch.zeros(3, 5, 3, dtype=torch.float64)
    elif bad == "jdepths":
        kw["jdepths"] = torch.zeros(3, 4, 3, dtype=torch.float64)
    elif bad == "dtdr":
        kw["dtdr"] = torch.zeros(3, 4, dtype=torch.float64)
    elif bad == "nlayers":
        n = torch.zeros(2, dtype=torch.int32)
    elif bad == "src":
        sd = torch.zeros(4, dtype=torch.float64)
    elif bad == "vels":
        v = torch.ones(3, 300, dtype=torch.float64)
    with pytest.raises(ValueError):
        device.dff_jac_device(v, z, n, so, sd, t, p, **kw)


def test_device_wrapper_needs_cuda_tensors(no_library):
    v, z, n, so, sd = _cpu_batch()
    t = torch.zeros(3, 5, dtype=torch.float64)
    with pytest.raises(ValueError, match="CUDA"):
        device.dff_jac_device(v, z, n, so, sd, t, t)
    with pytest.raises(ValueError, match="CUDA"):
        device.dff_jac_device(v.float(), z, n, so, sd, t, t)


def test_jacobian_rejects_bad_shapes_and_dtypes(no_library):
    v, z, n, so, sd = _cpu_batch()
    with pytest.raises(ValueError):
        grad.jacobian(v, z[:2], n, so, sd)
    with pytest.raises(ValueError):
        grad.jacobian(v, z, n[:2], so, sd)
    with pytest.raises(ValueError, match="int32"):
        grad.jacobian(v, z, n.to(torch.int64), so, sd)
    with pytest.raises(ValueError, match="float64"):
        grad.jacobian(v.float(), z, n, so, sd)
    with pytest.raises(ValueError, match="float64"):
        grad.jacobian(v, z, n, so, sd.float())
    with pytest.raises(ValueError, match="CUDA"):
        grad.jacobian(v, z, n, so, sd)


def test_host_wrapper_rejects_bad_shapes(no_library):
    v, z, n = np.ones((3, 4)), np.ones((3, 3)), np.full(3, 3, np.int32)
    so = sd = np.ones(5)
    with pytest.raises(ValueError):
        raymod.dff_batch_jac(v, z, np.full(3, 4, np.int32), so, sd)
    with pytest.raises(ValueError):
        raymod.dff_batch_jac(v, z[:2], n, so, sd)
    with pytest.raises(ValueError):
        raymod.dff_batch_jac(v, z, n[:2], so, sd)
    with pytest.raises(ValueError):
        raymod.dff_batch_jac(v, z, n, so, np.ones(4))
    with pytest.raises(ValueError):
        raymod.dff_batch_jac(np.ones((3, 300)), np.ones((3, 299)), n, so, sd)
