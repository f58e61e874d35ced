"""The per-ray Jacobian on the B200 (DESIGN.md section 12): rtb200_dff_jac_device against the numpy
reference jacobian_batch bit for bit at the forward's own timeP and p; the gradient kernel with a
one-hot weight returns the same rows; the host entry, the autograd route, stream semantics, empty
batches, refusals and 64-bit output offsets."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import _lib, device, grad, workloads

from jac_reference import jacobian_batch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _t(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=DEV)


def _bits_equal(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _run(v, z, n, so, sd, kmode=False, seed=0, not_converged=0):
    """Forward on the device, then the Jacobian on the device and in the reference."""
    rng = np.random.default_rng(seed)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    torch.cuda.synchronize()
    T, p = out["timeP"], out["p"]
    if not_converged:       # mark rays as the solver's failures: their rows must be zero
        idx = rng.choice(T.numel(), not_converged, replace=False)
        T.view(-1)[torch.as_tensor(idx, device=DEV)] = -999.0
    got = device.dff_jac_device(tv, tz, tn, tso, tsd, T, p, want_src=True, kmode=kmode)
    torch.cuda.synchronize()
    ref = jacobian_batch(v, z, n, so, sd, T.cpu().numpy(), p.cpu().numpy(), kmode=kmode)
    for name, r in zip(("jvels", "jdepths", "dtdr", "dtdd"), ref):
        assert _bits_equal(got[name], r), name
    return T.cpu().numpy(), p.cpu().numpy(), got


def _check_forward_is_the_oracle(v, z, n, so, sd, T, p):
    ref = oracle.dff_batch(v, z, n, so, sd, want_p=True)
    assert _bits_equal(T, ref["timeP"]) and _bits_equal(p, ref["p"])


def test_config1(golden):
    c = golden["config1"]
    v, z = np.array(c["vels"])[None], np.array(c["depths"])[None]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    n = np.array([z.shape[1]], np.int32)
    T, p, _ = _run(v, z, n, so, sd)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


@pytest.mark.parametrize("variant", [1, 3, 5])
@pytest.mark.parametrize("nl", [1, 2, 5, 10, 25, 50])
def test_random_batches(nl, variant):
    v, z, n = workloads.make_models(300, nl, 100 + nl)
    so, sd = workloads.make_sources(40, nl)
    rt.set_option("variant", variant)
    try:
        T, p, _ = _run(v, z, n, so, sd, seed=nl)
    finally:
        rt.set_option("variant", -1)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_kmode_states_k_1_to_30():
    k, vp, zi = workloads.make_transd_models(600, 30, 31, uniform_k=True)
    so, sd = workloads.make_sources(64, 31)
    assert k.min() == 1 and k.max() == 30
    T, _, got = _run(vp, zi, k, so, sd, kmode=True, seed=3)
    for b in range(0, 600, 37):
        _, pred = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :k[b] - 1], so, sd, np.zeros(so.size), 1.0)
        assert _bits_equal(T[b], pred)
    half = torch.as_tensor(k == 1, device=DEV)
    assert torch.all(got["jvels"][half][:, :, 1:] == 0) and torch.all(got["jdepths"][half] == 0)


def test_near_critical_deep_rays():
    v, z, n = workloads.make_models(64, 50, 5)
    so, sd = workloads.make_sources(128, 5, near_critical=True)
    T, p, _ = _run(v, z, n, so, sd, seed=5)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_top_layer_and_not_converged_rays():
    v, z, n = workloads.make_models(200, 6, 9)
    so, sd = workloads.make_sources(48, 9)
    sd[:16] = z[:, 0].min() * np.linspace(0.1, 0.9, 16)          # above every first interface
    T, p, got = _run(v, z, n, so, sd, seed=9, not_converged=500)
    nc = torch.as_tensor(T == -999.0, device=DEV)
    assert nc.sum().item() >= 500
    assert torch.all(got["jvels"][nc] == 0) and torch.all(got["jdepths"][nc] == 0)
    assert torch.all(got["jvels"][:, :16, 1:] == 0) and torch.all(got["jdepths"][:, :16] == 0)


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
    T, p, _ = _run(vp, zp, n, so, sd, seed=21)
    _check_forward_is_the_oracle(vp, zp, n, so, sd, T, p)


def test_wide_models_up_to_254_interfaces():
    rng = np.random.default_rng(254)
    B, L = 40, 254
    v = rng.uniform(workloads.VMIN, workloads.VMAX, (B, L + 1))
    z = np.cumsum(rng.uniform(20.0, 40.0, (B, L)), axis=1)
    n = rng.integers(150, L + 1, B).astype(np.int32)
    n[0] = L
    so, sd = workloads.make_sources(48, 254)
    sd = rng.uniform(100.0, z[:, -1].min() + 500.0, sd.size)     # some below every interface
    T, p, _ = _run(v, z, n, so, sd, seed=254)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


def test_config2_sample():
    c = workloads.CONFIGS["config2"]
    v, z, n = workloads.make_models(c["B"], c["nlayers"], c["seed"])
    pick = np.sort(np.random.default_rng(0).choice(c["B"], 3000, replace=False))
    so, sd = workloads.make_sources(c["nsrc"], c["seed"])
    T, p, _ = _run(v[pick], z[pick], n[pick], so, sd, seed=2)
    _check_forward_is_the_oracle(v[pick], z[pick], n[pick], so, sd, T, p)


@pytest.mark.parametrize("kmode", [False, True])
def test_one_hot_gradient_is_the_row(kmode):
    """dff_grad_device with w = e_s returns jvels[:, s] and jdepths[:, s], k = 1 included."""
    if kmode:
        k, vp, zi = workloads.make_transd_models(500, 20, 17, uniform_k=True)
        v, z, n = vp, zi, k
        assert (k == 1).any()
    else:
        v, z, n = workloads.make_models(500, 12, 17)
    so, sd = workloads.make_sources(48, 17)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    J = device.dff_jac_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], kmode=kmode)
    w = torch.zeros_like(out["timeP"])
    for s in (0, 1, 7, 23, 47):
        w.zero_()
        w[:, s] = 1.0
        g = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], w, kmode=kmode)
        torch.cuda.synchronize()
        assert _bits_equal(g["gvels"], J["jvels"][:, s]), s
        assert _bits_equal(g["gdepths"], J["jdepths"][:, s]), s


def test_autograd_jacobian_diagonal_blocks():
    v, z, n = workloads.make_models(4, 6, 8)
    so, sd = workloads.make_sources(8, 8)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    jv, jz = torch.autograd.functional.jacobian(lambda a, b: grad.travel_times(a, b, tn, tso, tsd), (tv, tz))
    J = grad.jacobian(tv, tz, tn, tso, tsd)
    ref = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True)
    assert _bits_equal(J["timeP"], ref["timeP"])
    assert J["timeP"].grad_fn is None and J["jvels"].grad_fn is None
    for b in range(4):
        assert _bits_equal(jv[b, :, b, :], J["jvels"][b]), b
        assert _bits_equal(jz[b, :, b, :], J["jdepths"][b]), b


def test_host_entry_equals_device_entry_and_is_deterministic():
    v, z, n = workloads.make_models(500, 10, 44)
    so, sd = workloads.make_sources(64, 44)
    h1 = rt.dff_batch_jac(v, z, n, so, sd, want_times=True, want_p=True, want_src=True)
    h2 = rt.dff_batch_jac(v, z, n, so, sd, want_times=True, want_p=True, want_src=True)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    d1 = device.dff_jac_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], want_src=True)
    d2 = device.dff_jac_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], want_src=True)
    torch.cuda.synchronize()
    assert _bits_equal(h1["timeP"], out["timeP"]) and _bits_equal(h1["p"], out["p"])
    for name in ("jvels", "jdepths", "dtdr", "dtdd"):
        assert _bits_equal(h1[name], d1[name]), name
        assert _bits_equal(h1[name], h2[name]) and _bits_equal(d1[name], d2[name]), name


def test_user_stream_call_does_not_synchronise_the_host():
    v, z, n = workloads.make_models(20000, 10, 3)
    so, sd = workloads.make_sources(64, 3)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))        # about a second of GPU time queued ahead of the call
        r = device.dff_jac_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], stream=s)
    assert not s.query(), "the call waited for the stream"
    s.synchronize()
    ref = device.dff_jac_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"])
    torch.cuda.synchronize()
    assert _bits_equal(r["jvels"], ref["jvels"]) and _bits_equal(r["jdepths"], ref["jdepths"])


def test_empty_batches():
    v, z, n = workloads.make_models(40, 5, 13)
    tv, tz, tn = _t(v), _t(z), _t(n, torch.int32)
    e = torch.empty(0, dtype=torch.float64, device=DEV)
    e2 = torch.empty((40, 0), dtype=torch.float64, device=DEV)
    r = device.dff_jac_device(tv, tz, tn, e, e, e2, e2, want_src=True)
    assert r["jvels"].shape == (40, 0, 6) and r["jdepths"].shape == (40, 0, 5)
    so, sd = workloads.make_sources(8, 13)
    e3 = torch.empty((0, 8), dtype=torch.float64, device=DEV)
    r = device.dff_jac_device(tv[:0], tz[:0], tn[:0], _t(so), _t(sd), e3, e3)
    assert r["jvels"].shape == (0, 8, 6)
    h = rt.dff_batch_jac(v, z, n, so[:0], sd[:0], want_times=True)
    assert h["jvels"].shape == (40, 0, 6) and h["timeP"].shape == (40, 0)
    h = rt.dff_batch_jac(v[:0], z[:0], n[:0], so, sd)
    assert h["jvels"].shape == (0, 8, 6)
    torch.cuda.synchronize()


def test_refusals_name_the_bad_argument():
    lib = _lib.load()
    v, z, n = workloads.make_models(4, 3, 1)
    so, sd = workloads.make_sources(5, 1)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    T = torch.zeros((4, 5), dtype=torch.float64, device=DEV)
    jv = torch.empty((4, 5, 4), dtype=torch.float64, device=DEV)
    jz = torch.empty((4, 5, 3), dtype=torch.float64, device=DEV)
    P = lambda t: t.data_ptr()
    good = dict(v=P(tv), z=P(tz), n=P(tn), ldv=4, ldz=3, so=P(tso), sd=P(tsd), t=P(T), p=P(T), jv=P(jv), jz=P(jz))
    cases = [
        (dict(ldv=0), "ldv must be >= 1"),
        (dict(ldv=256), "more than 254 interfaces per model are not supported"),
        (dict(v=None), "the Jacobian needs vels, nlayers and jvels"),
        (dict(n=None), "the Jacobian needs vels, nlayers and jvels"),
        (dict(jv=None), "the Jacobian needs vels, nlayers and jvels"),
        (dict(jz=None), "the Jacobian needs jdepths when ldz > 0"),
        (dict(so=None), "the Jacobian needs src_offset and src_depth"),
        (dict(sd=None), "the Jacobian needs src_offset and src_depth"),
        (dict(t=None), "the Jacobian needs the forward's timeP and p"),
        (dict(p=None), "the Jacobian needs the forward's timeP and p"),
    ]
    for change, msg in cases:
        a = {**good, **change}
        rc = lib.rtb200_dff_jac_device(a["v"], a["z"], a["n"], 4, a["ldv"], a["ldz"], a["so"], a["sd"], 5,
                                       a["t"], a["p"], a["jv"], a["jz"], None, None, 0, None)
        assert rc != 0 and _lib.last_error() == msg, (change, _lib.last_error())
    # ldz = 0 needs no jdepths
    rc = lib.rtb200_dff_jac_device(P(tv), None, P(tn), 4, 4, 0, P(tso), P(tsd), 5, P(T), P(T), P(jv), None,
                                   None, None, 0, None)
    torch.cuda.synchronize()
    assert rc == 0 and _lib.last_error() == ""
    # the host entry: the same checks on host buffers
    dp = C.POINTER(C.c_double)
    hv, hz, hn = np.ascontiguousarray(v), np.ascontiguousarray(z), np.ascontiguousarray(n, np.int32)
    hjv, hjz = np.empty((4, 5, 4)), np.empty((4, 5, 3))
    d = lambda a: None if a is None else a.ctypes.data_as(dp)
    ci = lambda x: C.byref(C.c_int(x))
    for (vv, nn, jjv, jjz, ldv, off), msg in [
            ((hv, hn, hjv, hjz, 0, so), "ldv must be >= 1"),
            ((None, hn, hjv, hjz, 4, so), "the Jacobian needs vels, nlayers and jvels"),
            ((hv, None, hjv, hjz, 4, so), "the Jacobian needs vels, nlayers and jvels"),
            ((hv, hn, None, hjz, 4, so), "the Jacobian needs vels, nlayers and jvels"),
            ((hv, hn, hjv, None, 4, so), "the Jacobian needs jdepths when ldz > 0"),
            ((hv, hn, hjv, hjz, 4, None), "the Jacobian needs src_offset and src_depth")]:
        rc = lib.dff_batch_jac(d(vv), d(hz), None if nn is None else nn.ctypes.data_as(C.POINTER(C.c_int)),
                               ci(4), ci(ldv), ci(3), d(off), d(sd), ci(5), None, None, d(jjv), d(jjz), None, None)
        assert rc != 0 and _lib.last_error() == msg, msg


def test_offsets_past_2_to_the_31():
    """jvels with more than 2^31 elements: the last models' rows against the formula -T/V_0."""
    B, S, ldv, ldz = 4_200_000, 64, 9, 1
    assert B * S * ldv > 2 ** 31
    need = B * S * (ldv + ldz + 2) * 8 + B * (ldv + ldz) * 8
    free, _ = torch.cuda.mem_get_info()
    if free < need * 1.1:
        pytest.skip(f"needs {need / 2 ** 30:.0f} GiB of device memory, {free / 2 ** 30:.0f} GiB free")
    rng = np.random.default_rng(7)
    v = torch.empty((B, ldv), dtype=torch.float64, device=DEV).uniform_(1500.0, 5000.0)
    z = torch.zeros((B, ldz), dtype=torch.float64, device=DEV)
    n = torch.zeros(B, dtype=torch.int32, device=DEV)                   # half-spaces: one layer
    so, sd = _t(rng.uniform(100.0, 3000.0, S)), _t(rng.uniform(10.0, 2000.0, S))
    out = device.dff_batch_device(v, z, n, so, sd, want_times=True, want_p=True)
    J = device.dff_jac_device(v, z, n, so, sd, out["timeP"], out["p"])
    torch.cuda.synchronize()
    tail = slice(B - 2000, B)
    T = out["timeP"][tail].cpu().numpy()
    v0 = v[tail, 0].cpu().numpy()
    jv = J["jvels"][tail].cpu().numpy()
    assert np.all(T > 0)
    assert _bits_equal(jv[:, :, 0], -(T / v0[:, None]))
    assert np.all(jv[:, :, 1:] == 0) and torch.all(J["jdepths"][tail] == 0)
    head = J["jvels"][:2000, :, 0].cpu().numpy()
    assert _bits_equal(head, -(out["timeP"][:2000].cpu().numpy() / v[:2000, 0].cpu().numpy()[:, None]))
