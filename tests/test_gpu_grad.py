"""The travel-time gradient on the B200 (DESIGN.md section 11): rtb200_dff_grad_device against the
numpy reference of tests/grad_reference.py bit for bit, evaluated at the forward's own timeP and p
(which are the oracle's, checked here too); the host entry, determinism, the autograd functions and
the stream semantics."""
import numpy as np
import pytest
import torch

import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import device, grad, workloads

from grad_reference import grad_batch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _t(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=DEV)


def _bits_equal(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _run(v, z, n, so, sd, kmode=False, seed=0, not_converged=0):
    """Forward on the device, then the gradient on the device and in the reference."""
    rng = np.random.default_rng(seed)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    torch.cuda.synchronize()
    T, p = out["timeP"], out["p"]
    if not_converged:       # mark rays as the solver's failures: they must contribute nothing
        idx = rng.choice(T.numel(), not_converged, replace=False)
        T.view(-1)[torch.as_tensor(idx, device=DEV)] = -999.0
    w = rng.normal(size=tuple(T.shape))
    got = device.dff_grad_device(tv, tz, tn, tso, tsd, T, p, _t(w), want_src=True, kmode=kmode)
    torch.cuda.synchronize()
    ref = grad_batch(v, z, n, so, sd, T.cpu().numpy(), p.cpu().numpy(), w, kmode=kmode)
    for name, r in zip(("gvels", "gdepths", "dtdr", "dtdd"), ref):
        assert _bits_equal(got[name], r), name
    return T.cpu().numpy(), p.cpu().numpy()


def _check_forward_is_the_oracle(v, z, n, so, sd, T, p):
    ref = oracle.dff_batch(v, z, n, so, sd, want_p=True)
    assert _bits_equal(T, ref["timeP"]) and _bits_equal(p, ref["p"])


def test_config1(golden):
    c = golden["config1"]
    v, z = np.array(c["vels"])[None], np.array(c["depths"])[None]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    n = np.array([z.shape[1]], np.int32)
    T, p = _run(v, z, n, so, sd)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


@pytest.mark.parametrize("variant", [1, 3, 5])
@pytest.mark.parametrize("nl", [1, 2, 5, 10, 25, 50])
def test_random_batches(nl, variant):
    v, z, n = workloads.make_models(300, nl, 100 + nl)
    so, sd = workloads.make_sources(40, nl)
    rt.set_option("variant", variant)
    try:
        T, p = _run(v, z, n, so, sd, seed=nl)
    finally:
        rt.set_option("variant", -1)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_kmode_states_k_1_to_30():
    k, vp, zi = workloads.make_transd_models(600, 30, 31, uniform_k=True)
    so, sd = workloads.make_sources(64, 31)
    assert k.min() == 1 and k.max() == 30
    T, _ = _run(vp, zi, k, so, sd, kmode=True, seed=3)
    for b in range(0, 600, 37):
        _, pred = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :k[b] - 1], so, sd, np.zeros(so.size), 1.0)
        assert _bits_equal(T[b], pred)


def test_near_critical_deep_rays():
    v, z, n = workloads.make_models(64, 50, 5)
    so, sd = workloads.make_sources(128, 5, near_critical=True)
    T, p = _run(v, z, n, so, sd, seed=5)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_top_layer_and_not_converged_rays():
    v, z, n = workloads.make_models(200, 6, 9)
    so, sd = workloads.make_sources(48, 9)
    sd[:16] = z[:, 0].min() * np.linspace(0.1, 0.9, 16)          # above every first interface
    T, p = _run(v, z, n, so, sd, seed=9, not_converged=500)
    assert (T == -999.0).sum() >= 500


def test_many_sources():
    v, z, n = workloads.make_models(50, 8, 12)
    so, sd = workloads.make_sources(300, 12)
    _run(v, z, n, so, sd, seed=12)


def test_ragged_batch_with_padded_rows():
    rng = np.random.default_rng(21)
    B, ldv, ldz = 37, 16, 14
    v, z, _ = workloads.make_models(B, 13, 21)
    n = rng.integers(0, 14, B).astype(np.int32)
    vp = np.zeros((B, ldv))
    vp[:, :14] = v
    zp = np.full((B, ldz), 1e30)
    zp[:, :13] = z
    so, sd = workloads.make_sources(70, 21)
    T, p = _run(vp, zp, n, so, sd, seed=21)
    _check_forward_is_the_oracle(vp, zp, n, so, sd, T, p)


def test_config2_sample():
    c = workloads.CONFIGS["config2"]
    v, z, n = workloads.make_models(c["B"], c["nlayers"], c["seed"])
    pick = np.sort(np.random.default_rng(0).choice(c["B"], 3000, replace=False))
    so, sd = workloads.make_sources(c["nsrc"], c["seed"])
    T, p = _run(v[pick], z[pick], n[pick], so, sd, seed=2)
    _check_forward_is_the_oracle(v[pick], z[pick], n[pick], so, sd, T, p)


def test_host_entry_equals_device_entry_and_is_deterministic():
    v, z, n = workloads.make_models(500, 10, 44)
    so, sd = workloads.make_sources(64, 44)
    w = np.random.default_rng(44).normal(size=(500, 64))
    h1 = rt.dff_batch_grad(v, z, n, so, sd, w, want_times=True, want_p=True, want_src=True)
    h2 = rt.dff_batch_grad(v, z, n, so, sd, w, want_times=True, want_p=True, want_src=True)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    d1 = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], _t(w), want_src=True)
    d2 = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], _t(w), want_src=True)
    torch.cuda.synchronize()
    assert _bits_equal(h1["timeP"], out["timeP"]) and _bits_equal(h1["p"], out["p"])
    for name in ("gvels", "gdepths", "dtdr", "dtdd"):
        assert _bits_equal(h1[name], d1[name]), name
        assert _bits_equal(h1[name], h2[name]) and _bits_equal(d1[name], d2[name]), name


def _autograd_inputs(kmode):
    if kmode:
        k, vp, zi = workloads.make_transd_models(256, 12, 7)
        v, z, n = vp, zi, k
    else:
        v, z, n = workloads.make_models(256, 10, 7)
    so, sd = workloads.make_sources(64, 7)
    tobs, sigma = workloads.make_observations(np.full(64, 1.5), 256, 7)
    leaf = lambda a: _t(a).requires_grad_(True)
    return leaf(v), leaf(z), _t(n, torch.int32), leaf(so), leaf(sd), leaf(tobs), leaf(sigma)


@pytest.mark.parametrize("kmode", [False, True])
def test_autograd_travel_times(kmode):
    v, z, n, so, sd, _, _ = _autograd_inputs(kmode)
    T = grad.travel_times(v, z, n, so, sd, kmode=kmode)
    ref = device.dff_batch_device(v.detach(), z.detach(), n, so.detach(), sd.detach(), want_times=True,
                                  want_p=True, kmode=kmode)
    assert _bits_equal(T, ref["timeP"])
    w = torch.randn(T.shape, dtype=torch.float64, device=DEV)
    gv, gz, gso, gsd = torch.autograd.grad((T * w).sum(), (v, z, so, sd))
    vjp = device.dff_grad_device(v.detach(), z.detach(), n, so.detach(), sd.detach(), ref["timeP"],
                                 ref["p"], w, want_src=True, kmode=kmode)
    assert _bits_equal(gv, vjp["gvels"]) and _bits_equal(gz, vjp["gdepths"])
    assert _bits_equal(gso, (w * vjp["dtdr"]).sum(0)) and _bits_equal(gsd, (w * vjp["dtdd"]).sum(0))


@pytest.mark.parametrize("kmode", [False, True])
def test_autograd_loglhood(kmode):
    v, z, n, so, sd, tobs, sigma = _autograd_inputs(kmode)
    L = grad.loglhood(v, z, n, so, sd, tobs, sigma, kmode=kmode)
    ref = device.dff_batch_device(v.detach(), z.detach(), n, so.detach(), sd.detach(), tobs=tobs.detach(),
                                  sigma=sigma.detach(), want_times=True, want_p=True, kmode=kmode)
    assert _bits_equal(L, ref["logL"])
    g = torch.randn(L.shape, dtype=torch.float64, device=DEV)
    gv, gz, gso, gsd, gt, gs = torch.autograd.grad((L * g).sum(), (v, z, so, sd, tobs, sigma))
    T, s2 = ref["timeP"], sigma.detach() * sigma.detach()
    res = tobs.detach()[None, :] - T
    w = (g[:, None] * (res / s2[:, None])).contiguous()                  # g dlogL/dT = g res / sigma^2
    vjp = device.dff_grad_device(v.detach(), z.detach(), n, so.detach(), sd.detach(), T, ref["p"], w,
                                 want_src=True, kmode=kmode)
    assert _bits_equal(gv, vjp["gvels"]) and _bits_equal(gz, vjp["gdepths"])
    assert _bits_equal(gso, (w * vjp["dtdr"]).sum(0)) and _bits_equal(gsd, (w * vjp["dtdd"]).sum(0))
    N = T.shape[1]
    sg = sigma.detach()
    torch.testing.assert_close(gs, g * ((res * res).sum(1) / sg ** 3 - N / sg), rtol=1e-13, atol=0)
    torch.testing.assert_close(gt, -(g[:, None] * res / s2[:, None]).sum(0), rtol=1e-12, atol=1e-12)


def test_rejected_model_has_zero_gradient():
    v, z, n, so, sd, tobs, sigma = _autograd_inputs(False)
    with torch.no_grad():
        sigma[3] = -1.0                     # log(sigma) is NaN: logL = -HUGE
    L = grad.loglhood(v, z, n, so, sd, tobs, sigma)
    assert L[3].item() == -torch.finfo(torch.float64).max
    gv, gs = torch.autograd.grad(L.sum(), (v, sigma))
    assert torch.all(gv[3] == 0) and gs[3].item() == 0.0 and torch.any(gv[4] != 0)


def test_user_stream_call_does_not_synchronise_the_host():
    v, z, n = workloads.make_models(20000, 10, 3)
    so, sd = workloads.make_sources(64, 3)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    w = torch.ones_like(out["timeP"])
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))        # about a second of GPU time queued ahead of the call
        r = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], w, stream=s)
    assert not s.query(), "the call waited for the stream"
    s.synchronize()
    ref = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], w)
    torch.cuda.synchronize()
    assert _bits_equal(r["gvels"], ref["gvels"])


def test_no_sources_gives_zero_gradients():
    v, z, n = workloads.make_models(40, 5, 13)
    tv, tz, tn = _t(v), _t(z), _t(n, torch.int32)
    e = torch.empty(0, dtype=torch.float64, device=DEV)
    e2 = torch.empty((40, 0), dtype=torch.float64, device=DEV)
    r = device.dff_grad_device(tv, tz, tn, e, e, e2, e2, e2,
                               gvels=torch.full((40, 6), 7.0, dtype=torch.float64, device=DEV),
                               gdepths=torch.full((40, 5), 7.0, dtype=torch.float64, device=DEV))
    torch.cuda.synchronize()
    assert torch.all(r["gvels"] == 0) and torch.all(r["gdepths"] == 0)


def test_wide_models_up_to_254_interfaces():
    """More than 64 layer columns: the kernel's narrowest tile (8 models per CTA), its largest tables."""
    rng = np.random.default_rng(254)
    B, L = 40, 254
    v = rng.uniform(workloads.VMIN, workloads.VMAX, (B, L + 1))
    z = np.cumsum(rng.uniform(20.0, 40.0, (B, L)), axis=1)
    n = rng.integers(150, L + 1, B).astype(np.int32)
    n[0] = L
    so, sd = workloads.make_sources(48, 254)
    sd = rng.uniform(100.0, z[:, -1].min() + 500.0, sd.size)     # some below every interface
    T, p = _run(v, z, n, so, sd, seed=254)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_zero_sigma_model_has_zero_gradient():
    v, z, n, so, sd, tobs, sigma = _autograd_inputs(False)
    with torch.no_grad():
        sigma[5] = 0.0                      # log(0) = -inf, the residual term is inf: logL = -HUGE
    L = grad.loglhood(v, z, n, so, sd, tobs, sigma)
    gv, gs, gt = torch.autograd.grad(L.sum(), (v, sigma, tobs))
    assert torch.all(gv[5] == 0) and gs[5].item() == 0.0
    assert torch.isfinite(gv).all() and torch.isfinite(gs).all() and torch.isfinite(gt).all()
