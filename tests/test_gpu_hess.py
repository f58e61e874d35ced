"""The per-model second derivatives on the B200 (DESIGN.md section 14): rtb200_dff_hess_device against
the numpy reference hess_batch bit for bit at the forward's own timeP and p over the shapes of the
normal-equations tests; the host entry, grad.newton_equations, stream order, empty batches,
refusals and 64-bit output offsets; and the kernel against the closed form in mpmath at its own p
and at the converged ray."""
import mpmath
import numpy as np
import pytest
import torch
from mpmath import mpf

import hp_reference as hp
import raytracerfortran_b200 as rt
from hess_reference import closed_form, hess_batch
from raytracerfortran_b200 import _lib, device, grad, workloads
from test_gpu_jac import DEV, _bits_equal, _check_forward_is_the_oracle, _t

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
C = 16      # as test_hess_cpu


def _run(v, z, n, so, sd, kmode=False, seed=0, not_converged=0):
    """Forward on the device, then the second derivatives on the device and in the reference."""
    rng = np.random.default_rng(seed)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    torch.cuda.synchronize()
    T, p = out["timeP"], out["p"]
    if not_converged:
        idx = rng.choice(T.numel(), not_converged, replace=False)
        T.view(-1)[torch.as_tensor(idx, device=DEV)] = -999.0
    Tn, pn = T.cpu().numpy(), p.cpu().numpy()
    w = rng.normal(0.0, 0.05, Tn.shape)
    got = device.dff_hess_device(tv, tz, tn, tso, tsd, T, p, _t(w), kmode=kmode)
    torch.cuda.synchronize()
    H = hess_batch(v, z, n, so, sd, Tn, pn, w, kmode=kmode)
    assert _bits_equal(got["H"], H)
    return Tn, pn, w, got


def test_config1(golden):
    c = golden["config1"]
    v, z = np.array(c["vels"])[None], np.array(c["depths"])[None]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    n = np.array([z.shape[1]], np.int32)
    T, p, _, _ = _run(v, z, n, so, sd)
    _check_forward_is_the_oracle(v, z, n, so, sd, T, p)


@pytest.mark.parametrize("nl", [1, 2, 5, 10, 25, 50])
def test_random_batches(nl):
    v, z, n = workloads.make_models(61, nl, 700 + nl)
    so, sd = workloads.make_sources(24, nl)
    _run(v, z, n, so, sd, seed=nl)


def test_kmode_states_k_1_to_30():
    k, vp, zi = workloads.make_transd_models(200, 30, 31, uniform_k=True)
    so, sd = workloads.make_sources(48, 31)
    sd[-1] = 12000.0                                      # below the k = 1 fake interface
    assert k.min() == 1 and k.max() == 30
    _, _, _, got = _run(vp, zi, k, so, sd, kmode=True, seed=3)
    one = torch.as_tensor(k == 1, device=DEV)
    assert torch.all(got["H"][one][:, 1:] == 0) and torch.all(got["H"][one][:, :, 1:] == 0)


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
    v, z, n = workloads.make_models(41 if nsrc < 1024 else 19, 10, 30 + nsrc)
    so, sd = workloads.make_sources(nsrc, 30)
    _run(v, z, n, so, sd, seed=nsrc)


def test_newton_matrix_is_JtJ_minus_the_residual_weighted_hessian():
    v, z, n = workloads.make_models(300, 10, 4)
    so, sd = workloads.make_sources(64, 4)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    tobs = _t(np.random.default_rng(4).uniform(0.2, 2.0, so.size))
    N = grad.newton_equations(tv, tz, tn, tso, tsd, tobs)
    ref = grad.normal_equations(tv, tz, tn, tso, tsd, tobs=tobs)
    S = grad.hessian(tv, tz, tn, tso, tsd, tobs[None, :] - ref["timeP"])
    assert _bits_equal(N["timeP"], ref["timeP"]) and _bits_equal(S["timeP"], ref["timeP"])
    assert _bits_equal(N["JtJ"], ref["JtJ"]) and _bits_equal(N["Jtr"], ref["Jtr"])
    assert _bits_equal(N["A"], ref["JtJ"] - S["H"]) and N["A"].grad_fn is None
    assert torch.equal(N["A"], N["A"].transpose(1, 2))


def test_host_entry_equals_device_entry():
    v, z, n = workloads.make_models(500, 10, 44)
    so, sd = workloads.make_sources(64, 44)
    w = np.random.default_rng(44).normal(0.0, 0.1, (500, so.size))
    h = rt.dff_batch_hess(v, z, n, so, sd, w, want_times=True, want_p=True)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    d = device.dff_hess_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], _t(w))
    torch.cuda.synchronize()
    assert _bits_equal(h["timeP"], out["timeP"]) and _bits_equal(h["p"], out["p"])
    assert _bits_equal(h["H"], d["H"])


def test_side_stream_call_is_ordered_after_its_inputs():
    v, z, n = workloads.make_models(20000, 10, 3)
    so, sd = workloads.make_sources(64, 3)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    new_w = _t(np.random.default_rng(3).normal(0.0, 0.1, (20000, so.size)))
    ref = device.dff_hess_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], new_w)
    torch.cuda.synchronize()
    w = torch.zeros_like(new_w)
    s = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))        # about a second of GPU time queued ahead of the inputs
        w.copy_(new_w)
        r = device.dff_hess_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], w, stream=s)
    assert not s.query(), "the call waited for the stream"
    s.synchronize()
    assert _bits_equal(r["H"], ref["H"])


def test_empty_batches():
    v, z, n = workloads.make_models(40, 5, 13)
    tv, tz, tn = _t(v), _t(z), _t(n, torch.int32)
    e = torch.empty(0, dtype=torch.float64, device=DEV)
    e2 = torch.empty((40, 0), dtype=torch.float64, device=DEV)
    r = device.dff_hess_device(tv, tz, tn, e, e, e2, e2, e2)
    torch.cuda.synchronize()
    assert r["H"].shape == (40, 11, 11) and torch.all(r["H"] == 0)
    so, sd = workloads.make_sources(8, 13)
    e3 = torch.empty((0, 8), dtype=torch.float64, device=DEV)
    r = device.dff_hess_device(tv[:0], tz[:0], tn[:0], _t(so), _t(sd), e3, e3, e3)
    assert r["H"].shape == (0, 11, 11)
    h = rt.dff_batch_hess(v, z, n, so[:0], sd[:0], np.zeros((40, 0)), want_times=True)
    assert np.all(h["H"] == 0) and h["timeP"].shape == (40, 0)
    h = rt.dff_batch_hess(v[:0], z[:0], n[:0], so, sd, np.zeros((0, 8)))
    assert h["H"].shape == (0, 11, 11)
    torch.cuda.synchronize()


def test_refusals_name_the_bad_argument():
    lib = _lib.load()
    v, z, n = workloads.make_models(4, 3, 1)
    so, sd = workloads.make_sources(5, 1)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    T = torch.zeros((4, 5), dtype=torch.float64, device=DEV)
    A = torch.empty((4, 7, 7), dtype=torch.float64, device=DEV)
    P = lambda t: t.data_ptr()
    good = dict(v=P(tv), n=P(tn), ldv=4, so=P(tso), sd=P(tsd), t=P(T), p=P(T), w=P(T), A=P(A))
    cases = [
        (dict(ldv=0), "ldv must be >= 1"),
        (dict(ldv=256), "more than 254 interfaces per model are not supported"),
        (dict(v=None), "the second derivatives need vels, nlayers and H"),
        (dict(n=None), "the second derivatives need vels, nlayers and H"),
        (dict(A=None), "the second derivatives need vels, nlayers and H"),
        (dict(so=None), "the second derivatives need src_offset, src_depth and w"),
        (dict(sd=None), "the second derivatives need src_offset, src_depth and w"),
        (dict(w=None), "the second derivatives need src_offset, src_depth and w"),
        (dict(t=None), "the second derivatives need the forward's timeP and p"),
        (dict(p=None), "the second derivatives need the forward's timeP and p"),
    ]
    for change, msg in cases:
        a = {**good, **change}
        rc = lib.rtb200_dff_hess_device(a["v"], P(tz), a["n"], 4, a["ldv"], 3, a["so"], a["sd"], 5,
                                        a["t"], a["p"], a["w"], a["A"], 0, None)
        assert rc != 0 and _lib.last_error() == msg, (change, _lib.last_error())
    rc = lib.rtb200_dff_hess_device(P(tv), P(tz), P(tn), 4, 4, 3, P(tso), P(tsd), 5, P(T), P(T), P(T),
                                    P(A), 0, None)
    torch.cuda.synchronize()
    assert rc == 0 and _lib.last_error() == ""


def test_offsets_past_2_to_the_31():
    """H with more than 2^31 elements: the last models against the reference."""
    B, S, nl = 220_000, 4, 50
    P = 2 * nl + 1
    assert B * P * P > 2 ** 31
    need = B * P * P * 8 + B * (P + 3 * S) * 8 * 2
    free, _ = torch.cuda.mem_get_info()
    if free < need * 1.2:
        pytest.skip(f"needs {need / 2 ** 30:.0f} GiB of device memory, {free / 2 ** 30:.0f} GiB free")
    v, z, n = workloads.make_models(B, nl, 77)
    so, sd = workloads.make_sources(S, 77)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True)
    w = np.linspace(-1.0, 1.0, B * S).reshape(B, S)
    H = device.dff_hess_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], _t(w))["H"]
    torch.cuda.synchronize()
    for sl in (slice(B - 40, B), slice(0, 8)):
        ref = hess_batch(v[sl], z[sl], n[sl], so, sd, out["timeP"][sl].cpu().numpy(),
                         out["p"][sl].cpu().numpy(), w[sl])
        assert _bits_equal(H[sl], ref)


def _against_closed_form(v, z, n, so, sd, kmode, seed):
    """Worst error/bound of the kernel's H against sum_s w_s d2T_s of the closed form in mpmath,
    (a) at the kernel's own p within the rounding bound, (b) at the converged p* within the
    rounding bound plus |dH/dp| |p - p*| (the solver's stopping rule)."""
    rng = np.random.default_rng(seed)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    T, p = out["timeP"].cpu().numpy(), out["p"].cpu().numpy()
    w = rng.normal(0.0, 1.0, T.shape)
    Hk = device.dff_hess_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], _t(w), kmode=kmode)["H"].cpu().numpy()
    B, S = T.shape
    ldv, ldz = v.shape[1], z.shape[1]
    worst_own, worst_conv = 0.0, 0.0
    with mpmath.workdps(hp.DPS):
        for b in range(B):
            Pn = ldv + ldz
            own, conv = np.full((Pn, Pn), mpf(0), object), np.full((Pn, Pn), mpf(0), object)
            bd, bdc = np.full((Pn, Pn), mpf(0), object), np.full((Pn, Pn), mpf(0), object)
            for s in range(S):
                if T[b, s] == hp.NOT_CONVERGED:
                    continue
                r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=ldv, ldz=ldz)
                ps = r.p_star()
                if ps is None:
                    continue
                q = mpf(float(p[b, s]))
                D2, M = closed_form(r, q, T=float(T[b, s]))
                D2s, _ = closed_form(r, ps)
                if r.n >= 2:
                    dp = abs(q - ps) * mpf("1e-3") + mpf(10) ** -30
                    Dp, _ = closed_form(r, q + dp)
                    Dm, _ = closed_form(r, q - dp)
                    V, _ = r.column()
                    cmin2 = min(1 - (q * x) ** 2 for x in V)
                    tstop = 0
                else:           # 2 T / V_0^2: the forward's T within its own bound
                    Dp = Dm = D2
                    dp, cmin2 = mpf(1), mpf(1)
                    tstop = 2 * r.t_bound(ps) / r.column()[0][0] ** 2
                kap = C * U * (1 + 1 / cmin2) + S * U
                cols = [c if c < r.nv else ldv + c - r.nv for c in range(r.nv + r.nz)]
                for x, cx in enumerate(cols):
                    for y, cy in enumerate(cols):
                        ws = mpf(float(w[b, s]))
                        own[cx, cy] += ws * D2[x][y]
                        conv[cx, cy] += ws * D2s[x][y]
                        bd[cx, cy] += abs(ws) * kap * M[x][y]
                        slope = abs(Dp[x][y] - Dm[x][y]) / (2 * dp)
                        bdc[cx, cy] += abs(ws) * (kap * M[x][y] + 2 * slope * abs(q - ps) + tstop)
            for i in range(Pn):
                for j in range(Pn):
                    g = mpf(float(Hk[b, i, j]))
                    if bd[i, j] > 0:
                        worst_own = max(worst_own, float(abs(g - own[i, j]) / bd[i, j]))
                        worst_conv = max(worst_conv, float(abs(g - conv[i, j]) / bdc[i, j]))
                    else:
                        assert g == 0
    return worst_own, worst_conv


def test_kernel_against_the_closed_form_in_mpmath():
    cases = []
    v, z, n = workloads.make_models(6, 6, 91)
    so, sd = workloads.make_sources(8, 91)
    cases.append((v, z, n, so, sd, False))
    v, z, n = workloads.make_models(3, 12, 92)
    so, sd = workloads.make_sources(6, 92, near_critical=True)
    cases.append((v, z, n, so, sd, False))
    k, vp, zi = workloads.make_transd_models(6, 5, 93, uniform_k=True)
    so, sd = workloads.make_sources(6, 93)
    sd[-1] = 12000.0
    cases.append((vp, zi, k, so, sd, True))
    worst = [0.0, 0.0]
    for i, c in enumerate(cases):
        a, b = _against_closed_form(*c, seed=i)
        worst = [max(worst[0], a), max(worst[1], b)]
    print(f"second derivatives: worst error/bound at the kernel's p {worst[0]:.3f}, "
          f"at the converged ray {worst[1]:.3f}")
    assert worst[0] <= 1.0 and worst[1] <= 1.0
