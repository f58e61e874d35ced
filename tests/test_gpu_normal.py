"""The per-model normal equations on the B200 (DESIGN.md section 13): rtb200_dff_normal_device against
the numpy reference normal_batch bit for bit at the forward's own timeP and p; the host entry, the
contraction of grad.jacobian's rows, stream order, empty batches, refusals and 64-bit output
offsets."""
import numpy as np
import pytest
import torch

import raytracerfortran_b200 as rt
from raytracerfortran_b200 import _lib, device, grad, workloads

from normal_reference import normal_batch, reach_batch
from test_gpu_jac import DEV, _bits_equal, _check_forward_is_the_oracle, _t

pytestmark = pytest.mark.gpu

U = 2.0 ** -53


def _run(v, z, n, so, sd, kmode=False, seed=0, not_converged=0):
    """Forward on the device, then the normal equations on the device and in the reference, with
    and without tobs."""
    rng = np.random.default_rng(seed)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    torch.cuda.synchronize()
    T, p = out["timeP"], out["p"]
    if not_converged:
        idx = rng.choice(T.numel(), not_converged, replace=False)
        T.view(-1)[torch.as_tensor(idx, device=DEV)] = -999.0
    Tn, pn = T.cpu().numpy(), p.cpu().numpy()
    conv = Tn[Tn != -999.0]
    tobs = rng.uniform(conv.min() if conv.size else 0.0, conv.max() if conv.size else 1.0, so.size)
    got = device.dff_normal_device(tv, tz, tn, tso, tsd, T, p, tobs=_t(tobs), kmode=kmode)
    bare = device.dff_normal_device(tv, tz, tn, tso, tsd, T, p, kmode=kmode)
    torch.cuda.synchronize()
    JtJ, Jtr = normal_batch(v, z, n, so, sd, Tn, pn, tobs=tobs, kmode=kmode)
    assert _bits_equal(got["JtJ"], JtJ) and _bits_equal(got["Jtr"], Jtr)
    assert _bits_equal(bare["JtJ"], JtJ) and bare["Jtr"] is None
    return Tn, pn, got


def test_config1(golden):
    c = golden["config1"]
    v, z = np.array(c["vels"])[None], np.array(c["depths"])[None]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    n = np.array([z.shape[1]], np.int32)
    T, p, _ = _run(v, z, n, so, sd)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


@pytest.mark.parametrize("nl", [1, 2, 5, 10, 25, 50])
def test_random_batches(nl):
    v, z, n = workloads.make_models(61, nl, 700 + nl)
    so, sd = workloads.make_sources(24, nl)
    _run(v, z, n, so, sd, seed=nl)


def test_kmode_states_k_1_to_30():
    k, vp, zi = workloads.make_transd_models(200, 30, 31, uniform_k=True)
    so, sd = workloads.make_sources(48, 31)
    assert k.min() == 1 and k.max() == 30
    _, _, got = _run(vp, zi, k, so, sd, kmode=True, seed=3)
    one = torch.as_tensor(k == 1, device=DEV)
    assert torch.all(got["JtJ"][one][:, 1:] == 0) and torch.all(got["JtJ"][one][:, :, 1:] == 0)


def test_near_critical_deep_rays():
    v, z, n = workloads.make_models(16, 50, 5)
    so, sd = workloads.make_sources(64, 5, near_critical=True)
    _run(v, z, n, so, sd, seed=5)


def test_top_layer_and_not_converged_rays():
    v, z, n = workloads.make_models(60, 6, 9)
    so, sd = workloads.make_sources(40, 9)
    sd[:12] = z[:, 0].min() * np.linspace(0.1, 0.9, 12)
    _run(v, z, n, so, sd, seed=9, not_converged=300)


def test_widest_models_multi_block_triangle():
    """ldv = 255: P = 509, the triangle split over many CTAs a model."""
    rng = np.random.default_rng(255)
    B, L = 3, 254
    v = rng.uniform(workloads.VMIN, workloads.VMAX, (B, L + 1))
    z = np.cumsum(rng.uniform(20.0, 40.0, (B, L)), axis=1)
    n = np.array([L, 200, 160], np.int32)
    so, sd = workloads.make_sources(20, 254)
    sd = rng.uniform(100.0, z[:, -1].min() + 500.0, sd.size)
    _run(v, z, n, so, sd, seed=254)


def test_ragged_batch_not_a_multiple_of_any_tile():
    rng = np.random.default_rng(21)
    B, ldv, ldz = 37, 16, 14
    v, z, _ = workloads.make_models(B, 13, 21)
    n = rng.integers(1, 14, B).astype(np.int32)
    vp = np.zeros((B, ldv))
    vp[:, :14] = v
    zp = np.full((B, ldz), 1e30)
    zp[:, :13] = z
    so, sd = workloads.make_sources(30, 21)
    _run(vp, zp, n, so, sd, seed=21)


@pytest.mark.parametrize("nsrc", [1, 11, 13, 1024])
def test_source_counts(nsrc):
    """1, the config-2 chunk (12 sources) +- 1, and 1024."""
    v, z, n = workloads.make_models(41 if nsrc < 1024 else 19, 10, 30 + nsrc)
    so, sd = workloads.make_sources(nsrc, 30)
    _run(v, z, n, so, sd, seed=nsrc)


def test_jacobian_rows_contracted_in_torch_agree():
    v, z, n = workloads.make_models(300, 10, 4)
    so, sd = workloads.make_sources(64, 4)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    tobs = _t(np.random.default_rng(4).uniform(0.2, 2.0, so.size))
    N = grad.normal_equations(tv, tz, tn, tso, tsd, tobs=tobs)
    J = grad.jacobian(tv, tz, tn, tso, tsd)
    assert _bits_equal(N["timeP"], J["timeP"]) and N["JtJ"].grad_fn is None
    R = torch.as_tensor(reach_batch(v, z, n, so, sd, J["timeP"].cpu().numpy()), device=DEV)
    rows = torch.where(R, torch.cat([J["jvels"], J["jdepths"]], 2), 0.0)
    r = tobs[None, :] - J["timeP"]
    A = rows.transpose(1, 2) @ rows
    g = (rows.transpose(1, 2) @ r[:, :, None])[:, :, 0]
    Aabs = rows.abs().transpose(1, 2) @ rows.abs()
    gabs = (rows.abs().transpose(1, 2) @ r.abs()[:, :, None])[:, :, 0]
    S = so.size
    assert torch.all((N["JtJ"] - A).abs() <= 2 * S * U * Aabs + 1e-300)
    assert torch.all((N["Jtr"] - g).abs() <= 2 * (S + 1) * U * gabs + 1e-300)
    assert torch.equal(N["JtJ"], N["JtJ"].transpose(1, 2))


def test_host_entry_equals_device_entry():
    v, z, n = workloads.make_models(500, 10, 44)
    so, sd = workloads.make_sources(64, 44)
    tobs = np.random.default_rng(44).uniform(0.2, 2.0, so.size)
    h = rt.dff_batch_normal(v, z, n, so, sd, tobs=tobs, want_times=True, want_p=True)
    h0 = rt.dff_batch_normal(v, z, n, so, sd)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    d = device.dff_normal_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], tobs=_t(tobs))
    torch.cuda.synchronize()
    assert _bits_equal(h["timeP"], out["timeP"]) and _bits_equal(h["p"], out["p"])
    assert _bits_equal(h["JtJ"], d["JtJ"]) and _bits_equal(h["Jtr"], d["Jtr"])
    assert _bits_equal(h0["JtJ"], d["JtJ"]) and h0["Jtr"] is None


def test_side_stream_call_is_ordered_after_its_inputs():
    v, z, n = workloads.make_models(20000, 10, 3)
    so, sd = workloads.make_sources(64, 3)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    new_tobs = _t(np.random.default_rng(3).uniform(0.2, 2.0, so.size))
    ref = device.dff_normal_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], tobs=new_tobs)
    torch.cuda.synchronize()
    tobs = torch.zeros_like(new_tobs)
    s = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))        # about a second of GPU time queued ahead of the inputs
        tobs.copy_(new_tobs)
        r = device.dff_normal_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], tobs=tobs, stream=s)
    assert not s.query(), "the call waited for the stream"
    s.synchronize()
    assert _bits_equal(r["JtJ"], ref["JtJ"]) and _bits_equal(r["Jtr"], ref["Jtr"])


def test_empty_batches():
    v, z, n = workloads.make_models(40, 5, 13)
    tv, tz, tn = _t(v), _t(z), _t(n, torch.int32)
    e = torch.empty(0, dtype=torch.float64, device=DEV)
    e2 = torch.empty((40, 0), dtype=torch.float64, device=DEV)
    r = device.dff_normal_device(tv, tz, tn, e, e, e2, e2, tobs=e)
    torch.cuda.synchronize()
    assert r["JtJ"].shape == (40, 11, 11) and torch.all(r["JtJ"] == 0) and torch.all(r["Jtr"] == 0)
    so, sd = workloads.make_sources(8, 13)
    e3 = torch.empty((0, 8), dtype=torch.float64, device=DEV)
    r = device.dff_normal_device(tv[:0], tz[:0], tn[:0], _t(so), _t(sd), e3, e3)
    assert r["JtJ"].shape == (0, 11, 11)
    h = rt.dff_batch_normal(v, z, n, so[:0], sd[:0], tobs=np.zeros(0), want_times=True)
    assert np.all(h["JtJ"] == 0) and np.all(h["Jtr"] == 0) and h["timeP"].shape == (40, 0)
    h = rt.dff_batch_normal(v[:0], z[:0], n[:0], so, sd)
    assert h["JtJ"].shape == (0, 11, 11)
    torch.cuda.synchronize()


def test_refusals_name_the_bad_argument():
    lib = _lib.load()
    v, z, n = workloads.make_models(4, 3, 1)
    so, sd = workloads.make_sources(5, 1)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    T = torch.zeros((4, 5), dtype=torch.float64, device=DEV)
    A = torch.empty((4, 7, 7), dtype=torch.float64, device=DEV)
    g = torch.empty((4, 7), dtype=torch.float64, device=DEV)
    P = lambda t: t.data_ptr()
    good = dict(v=P(tv), n=P(tn), ldv=4, so=P(tso), sd=P(tsd), t=P(T), p=P(T), o=P(tso), A=P(A), g=P(g))
    cases = [
        (dict(ldv=0), "ldv must be >= 1"),
        (dict(ldv=256), "more than 254 interfaces per model are not supported"),
        (dict(v=None), "the normal equations need vels, nlayers and JtJ"),
        (dict(n=None), "the normal equations need vels, nlayers and JtJ"),
        (dict(A=None), "the normal equations need vels, nlayers and JtJ"),
        (dict(o=None), "tobs and Jtr must be given together"),
        (dict(g=None), "tobs and Jtr must be given together"),
        (dict(so=None), "the normal equations need src_offset and src_depth"),
        (dict(sd=None), "the normal equations need src_offset and src_depth"),
        (dict(t=None), "the normal equations need the forward's timeP and p"),
        (dict(p=None), "the normal equations need the forward's timeP and p"),
    ]
    for change, msg in cases:
        a = {**good, **change}
        rc = lib.rtb200_dff_normal_device(a["v"], P(tz), a["n"], 4, a["ldv"], 3, a["so"], a["sd"], 5,
                                          a["t"], a["p"], a["o"], a["A"], a["g"], 0, None)
        assert rc != 0 and _lib.last_error() == msg, (change, _lib.last_error())
    rc = lib.rtb200_dff_normal_device(P(tv), P(tz), P(tn), 4, 4, 3, P(tso), P(tsd), 5, P(T), P(T), None,
                                      P(A), None, 0, None)
    torch.cuda.synchronize()
    assert rc == 0 and _lib.last_error() == ""


def test_offsets_past_2_to_the_31():
    """JtJ with more than 2^31 elements: the last models against the reference."""
    B, S, nl = 220_000, 4, 50
    P = 2 * nl + 1
    assert B * P * P > 2 ** 31
    need = B * P * P * 8 + B * (P + 2 * S) * 8 * 2
    free, _ = torch.cuda.mem_get_info()
    if free < need * 1.2:
        pytest.skip(f"needs {need / 2 ** 30:.0f} GiB of device memory, {free / 2 ** 30:.0f} GiB free")
    v, z, n = workloads.make_models(B, nl, 77)
    so, sd = workloads.make_sources(S, 77)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    tobs = np.linspace(0.5, 1.5, S)
    N = device.dff_normal_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], tobs=_t(tobs))
    torch.cuda.synchronize()
    for sl in (slice(B - 40, B), slice(0, 8)):
        JtJ, Jtr = normal_batch(v[sl], z[sl], n[sl], so, sd, out["timeP"][sl].cpu().numpy(),
                                out["p"][sl].cpu().numpy(), tobs=tobs)
        assert _bits_equal(N["JtJ"][sl], JtJ) and _bits_equal(N["Jtr"][sl], Jtr)
