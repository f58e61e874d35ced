"""CPU checks of the travel-time gradient (DESIGN.md section 11): the formulas against finite
differences of an independently converged travel time, the effect of the solver's 0.1 m stopping
rule, the exact identity dT/dR = p, and the argument checks of the Python wrappers."""
import numpy as np
import pytest
import torch

import oracle
from raytracerfortran_b200 import _lib, device, grad, raymod, workloads

from grad_reference import column, converged_ray, grad_batch, offset_of, offset_slope, which_layer, model_columns


def _test1(golden):
    c = golden["config1"]
    return (np.array(c["vels"])[None, :], np.array(c["depths"])[None, :],
            np.array(c["src_offset_full"]), np.array(c["src_depth_full"]))


def _random_models(B, nl, seed):
    v, z, n = workloads.make_models(B, nl, seed)
    so, sd = workloads.make_sources(12, seed)
    return v, z, n, so, sd


def _clear_of_interfaces(z, sd, gap):
    return np.all(np.abs(z[:, :, None] - sd[None, None, :]) > gap, axis=1)


def _ray_grad(v, z, nl, R, d, p, T):
    """Gradient of one ray (one-hot weight): (dT/dV, dT/dz, dT/dR, dT/dd)."""
    gv, gz, dr, dd = grad_batch(v[None], z[None], [nl], [R], [d], [[T]], [[p]], [[1.0]])
    return gv[0], gz[0], dr[0, 0], dd[0, 0]


def _fd_ray(v, z, nl, R, d):
    """Central differences of the converged travel time."""
    T = lambda v_, z_, R_, d_: converged_ray(v_, z_, nl, R_, d_)[0]
    gv, gz = np.zeros_like(v), np.zeros_like(z)
    for i in range(v.size):
        h = 1e-5 * v[i]
        vp, vm = v.copy(), v.copy()
        vp[i] += h
        vm[i] -= h
        gv[i] = (T(vp, z, R, d) - T(vm, z, R, d)) / (2 * h)
    for j in range(z.size):
        h = 0.05
        zp, zm = z.copy(), z.copy()
        zp[j] += h
        zm[j] -= h
        gz[j] = (T(v, zp, R, d) - T(v, zm, R, d)) / (2 * h)
    h = 0.05
    dr = (T(v, z, R + h, d) - T(v, z, R - h, d)) / (2 * h)
    dd = (T(v, z, R, d + h) - T(v, z, R, d - h)) / (2 * h)
    return gv, gz, dr, dd


def _close(a, b, scale, rel=1e-6):
    """|a - b| <= rel * |b|, where |b| is floored at the largest derivative of the same units:
    a component far smaller than its siblings (eta_j ~ eta_{j+1}) is checked to that scale."""
    return np.all(np.abs(np.asarray(a) - np.asarray(b)) <= rel * np.maximum(np.abs(b), scale))


def _rays(golden):
    v1, z1, so1, sd1 = _test1(golden)
    yield v1[0], z1[0], so1, sd1
    v, z, _, so, sd = _random_models(6, 5, 11)
    for b in range(v.shape[0]):
        yield v[b], z[b], so, sd


def test_formulas_match_finite_differences_of_a_converged_time(golden):
    checked = 0
    for v, z, so, sd in _rays(golden):
        keep = _clear_of_interfaces(z[None], sd, 1.0)[0]
        for R, d in zip(so[keep], sd[keep]):
            T, p = converged_ray(v, z, z.size, R, d)
            if p * column(v, z, z.size, d)[0].max() > 0.999:
                continue        # near-critical: the finite differences themselves lose the digits
            gv, gz, dr, dd = _ray_grad(v, z, z.size, R, d, p, T)
            fv, fz, fr, fd = _fd_ray(v, z, z.size, R, d)
            per_m = max(np.max(np.abs(fz), initial=0.0), abs(fr), abs(fd))    # s/m: dz, dR, dd
            assert _close(gv, fv, np.max(np.abs(fv))), (gv, fv)
            assert _close(gz, fz, per_m) and _close(dr, fr, per_m) and _close(dd, fd, per_m), \
                (gz, fz, dr, fr, dd, fd)
            checked += 1
    assert checked >= 50


def test_oracle_p_is_within_the_stopping_rule_bound(golden):
    """At the oracle's own p, each component J differs from its converged value by at most
    |dJ/dp| * 0.1 m / |X'(p)|: the solver stops once |X(p) - R| < 0.1 m."""
    checked = 0
    for v, z, so, sd in _rays(golden):
        t_or, p_or, _ = oracle.trace_rays(v, z, so, sd)
        for k, (R, d) in enumerate(zip(so, sd)):
            V, H = column(v, z, z.size, d)
            if V.size < 2 or t_or[k] == -999.0 or abs(offset_of(p_or[k], V, H) - R) >= 0.1:
                continue
            T, p = converged_ray(v, z, z.size, R, d)
            if p * V.max() > 0.999:
                continue        # near-critical: dJ/dp varies too fast for a linear bound
            at = np.concatenate([np.atleast_1d(x) for x in _ray_grad(v, z, z.size, R, d, p_or[k], t_or[k])])
            ref = np.concatenate([np.atleast_1d(x) for x in _ray_grad(v, z, z.size, R, d, p, T)])
            dp = 1e-8 * p
            hi = np.concatenate([np.atleast_1d(x) for x in _ray_grad(v, z, z.size, R, d, p + dp, T)])
            lo = np.concatenate([np.atleast_1d(x) for x in _ray_grad(v, z, z.size, R, d, p - dp, T)])
            bound = np.abs((hi - lo) / (2 * dp)) * 0.1 / abs(offset_slope(p, V, H))
            assert np.all(np.abs(at - ref) <= 1.01 * bound + 1e-15 * np.abs(ref)), (at - ref, bound)
            checked += 1
    assert checked >= 50


def test_dT_dR_is_the_oracle_p_bit_for_bit(golden):
    v, z, n, so, sd = _random_models(40, 10, 5)
    ref = oracle.dff_batch(v, z, n, so, sd, want_p=True)
    w = np.ones_like(ref["timeP"])
    _, _, dtdr, _ = grad_batch(v, z, n, so, sd, ref["timeP"], ref["p"], w)
    conv = ref["timeP"] != -999.0
    assert np.array_equal(dtdr[conv].view(np.uint64), ref["p"][conv].view(np.uint64))
    assert np.all(dtdr[~conv] == 0.0)


def test_reference_which_layer_is_the_oracle_s(golden):
    v, z, n, so, sd = _random_models(30, 7, 8)
    sd = np.concatenate([sd, z[0, :4], z[3, 2:5]])       # sources exactly on interfaces too
    V, Z, H, NL, _ = model_columns(v, z, n)
    for d in sd:
        got = which_layer(Z, NL, d)
        want = [oracle.which_layer(z[b], d) for b in range(v.shape[0])]
        assert list(got) == want


def test_top_layer_and_kmode_half_space_rays():
    """Straight rays: dT/dV_0 = -T/V_0; at k = 1 both layers are vp_0 and the fake interface gets 0."""
    vp = np.array([[2500.0, 0.0], [3000.0, 4000.0]])
    zi = np.array([[0.0], [800.0]])
    k = np.array([1, 2])
    so, sd = np.array([100.0, 700.0]), np.array([500.0, 600.0])
    t = np.empty((2, 2))
    p = np.empty((2, 2))
    for b in range(2):
        ll, pred = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :k[b] - 1], so, sd, np.zeros(2), 1.0)
        t[b] = pred
        p[b] = (so / np.sqrt(sd * sd + so * so)) / vp[b, 0]
    gv, gz, dr, dd = grad_batch(vp, zi, k, so, sd, t, p, np.ones((2, 2)), kmode=True)
    assert gv[0, 0] == (0.0 + -(t[0, 0] / 2500.0)) + -(t[0, 1] / 2500.0)
    assert gv[0, 1] == 0.0 and gz[0, 0] == 0.0
    assert np.array_equal(dr, p)


# ---- argument checks: the wrappers refuse bad shapes before anything reaches the library ----

@pytest.fixture
def no_library(monkeypatch):
    def boom():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", boom)


def _cpu_batch(B=3, ldv=4, S=5):
    f = torch.float64
    return (torch.ones(B, ldv, dtype=f), torch.ones(B, ldv - 1, dtype=f), torch.full((B,), ldv - 1, dtype=torch.int32),
            torch.ones(S, dtype=f), torch.ones(S, dtype=f))


@pytest.mark.parametrize("bad", ["w", "timeP", "gvels", "nlayers", "src", "vels"])
def test_device_wrapper_rejects_bad_shapes(no_library, bad):
    v, z, n, so, sd = _cpu_batch()
    t = p = w = torch.zeros(3, 5, dtype=torch.float64)
    gvels = None
    if bad == "w":
        w = torch.zeros(3, 4, dtype=torch.float64)
    elif bad == "timeP":
        t = torch.zeros(5, 3, dtype=torch.float64)
    elif bad == "gvels":
        gvels = torch.zeros(3, 3, dtype=torch.float64)
    elif bad == "nlayers":
        n = torch.zeros(2, dtype=torch.int32)
    elif bad == "src":
        sd = torch.zeros(4, dtype=torch.float64)
    elif bad == "vels":
        v = torch.ones(3, 300, dtype=torch.float64)
    with pytest.raises(ValueError):
        device.dff_grad_device(v, z, n, so, sd, t, p, w, gvels=gvels)


def test_device_wrapper_needs_cuda_tensors(no_library):
    v, z, n, so, sd = _cpu_batch()
    t = torch.zeros(3, 5, dtype=torch.float64)
    with pytest.raises(ValueError, match="CUDA"):
        device.dff_grad_device(v, z, n, so, sd, t, t, t)


def test_autograd_wrappers_reject_bad_shapes(no_library):
    v, z, n, so, sd = _cpu_batch()
    with pytest.raises(ValueError):
        grad.travel_times(v, z[:2], n, so, sd)
    with pytest.raises(ValueError):
        grad.travel_times(v, z, n.to(torch.int64), so, sd)
    with pytest.raises(ValueError):
        grad.loglhood(v, z, n, so, sd, torch.zeros(4, dtype=torch.float64), torch.ones(3, dtype=torch.float64))
    with pytest.raises(ValueError):
        grad.loglhood(v, z, n, so, sd, torch.zeros(5, dtype=torch.float64), torch.ones(2, dtype=torch.float64))
    with pytest.raises(ValueError, match="CUDA"):
        grad.travel_times(v, z, n, so, sd)


def test_host_wrapper_rejects_bad_shapes(no_library):
    v, z, n = np.ones((3, 4)), np.ones((3, 3)), np.full(3, 3, np.int32)
    so = sd = np.ones(5)
    with pytest.raises(ValueError):
        raymod.dff_batch_grad(v, z, n, so, sd, np.ones((3, 4)))
    with pytest.raises(ValueError):
        raymod.dff_batch_grad(v, z, np.full(3, 4, np.int32), so, sd, np.ones((3, 5)))
    with pytest.raises(ValueError):
        raymod.dff_batch_grad(v, z[:2], n, so, sd, np.ones((3, 5)))
