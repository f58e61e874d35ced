"""CPU checks of the per-model second derivatives of the travel times (DESIGN.md section 14):

* the closed form against mpmath second derivatives of the converged travel time T*(theta), and
  at a fixed, non-converged p against mpmath derivatives of G(theta; p) and X'(p);
* the numpy reference hess_batch against an exact evaluation of the closed form, within the
  rounding bound, and its structure: exact symmetry, zero rows and columns, skipped rays;
* the reference against central differences of grad_reference's gradient at converged rays;
* plausible mistakes in the closed form are caught;
* the wrappers refuse bad arguments before anything reaches the library."""
import functools

import mpmath
import numpy as np
import pytest
import torch
from mpmath import mpf

import hp_reference as hp
from grad_reference import converged_ray, grad_batch
from hess_reference import MUTANTS, closed_form, hess_batch
from raytracerfortran_b200 import device, grad, raymod, workloads
from test_jac_cpu import _bits_equal, _forward

U = 2.0 ** -53
C = 16      # roundings a term may carry, each amplified by 1 / cos^2 near the critical angle


def _cases():
    """(label, Ray, columns) covering straight rays, n = 2..6, k = 1 on both sides of the fake
    interface, a source exactly on an interface and p V up to 1 - 1e-6."""
    v, z, n = workloads.make_models(6, 6, 41)
    yield "n = 1", hp.Ray(v[0], z[0], n[0], 1234.5, 0.5 * z[0, 0]), None
    for nl in range(2, 7):          # n = nl layers above the source, one more below it
        zz = z[nl - 2]
        d = 0.5 * (zz[nl - 2] + (zz[nl - 1] if nl - 1 < zz.size else zz[nl - 2] + 400.0))
        yield f"n = {nl}", hp.Ray(v[nl - 2, :nl + 1], zz[:nl], nl, 900.0 * nl, d), None
    vp, zi = [3100.0, 0.0], [0.0]
    yield "k = 1 below 9999.9", hp.Ray(vp, zi, 1, 4000.0, 12500.0, kmode=True), None
    yield "k = 1 above 9999.9", hp.Ray(vp, zi, 1, 4000.0, 2500.0, kmode=True), None
    yield "kmode k = 4", hp.Ray([2000.0, 3500.0, 3000.0, 5200.0], [800.0, 1900.0, 3000.0], 4, 5000.0, 3500.0,
                                kmode=True), None
    r = hp.Ray(v[2], z[2], n[2], 3000.0, z[2, 2])        # on an interface: n frozen below it
    assert r.n == 4 and float(r.column()[1][-1]) == 0.0
    yield "on an interface", r, None
    vv, zz = [2000.0, 3000.0, 9000.0, 2500.0], [500.0, 1500.0, 2500.0]
    for eps in (1e-3, 1e-6):
        r = hp.Ray(vv, zz, 3, 0.0, 3000.0)
        V, H = r.column()
        R = float(hp.offset(mpf(1 - eps) / max(V), V, H))
        yield f"p V = 1 - {eps:g}", hp.Ray(vv, zz, 3, R, 3000.0), None


def _with(th, pairs):
    t = list(th)
    for c, x in pairs:
        t[c] = x
    return t


@hp._hp
def _d2(f, th, x, y):
    """mpmath second derivative of f(theta) in columns x, y."""
    if x == y:
        return mpmath.diff(lambda a: f(_with(th, [(x, a)])), th[x], 2)
    return mpmath.diff(lambda a, b: f(_with(th, [(x, a), (y, b)])), (th[x], th[y]), (1, 1))


@functools.lru_cache(maxsize=None)
def _tstar_second_derivatives():
    """[(label, ray, p*, D2 of T* by mpmath)] over the model columns of every case; T* does not
    depend on a column the ray does not reach (velocity i >= n, interface j > n - 2), whose
    entries are 0."""
    out = []
    for label, r, _ in _cases():
        th = [mpf(x) for x in r.theta0]
        P = r.nv + r.nz
        reach = [c for c in range(P) if (c < min(r.n, r.nv) if c < r.nv else c - r.nv <= r.n - 2)]
        D2 = [[mpf(0)] * P for _ in range(P)]
        for x in reach:
            for y in (c for c in reach if c >= x):
                D2[x][y] = D2[y][x] = _d2(lambda t: r.T_star(t), th, x, y)
        out.append((label, r, r.p_star(), D2))
    return out


def _rel_err(a, b):
    P = len(a)
    scale = max(abs(b[x][y]) for x in range(P) for y in range(P))
    return max(abs(a[x][y] - b[x][y]) for x in range(P) for y in range(P)) / scale


def test_closed_form_is_the_second_derivative_of_the_converged_travel_time():
    worst = mpf(0)
    for label, r, ps, D2 in _tstar_second_derivatives():
        err = _rel_err(closed_form(r, ps)[0], D2)
        assert err < mpf(10) ** -25, (label, float(err))
        worst = max(worst, err)
    print(f"closed form vs T*: worst relative difference {float(worst):.1e}")


def test_closed_form_at_a_fixed_p_is_G_theta_theta_plus_the_implicit_term():
    """At p = 0.9 p* (not converged): G_thth + G_thp G_thp^T / X'(p), every piece by mpmath.diff of
    G(theta; p) and X' by offset_slope, independently of the closed forms."""
    for label, r, ps, _ in _tstar_second_derivatives():
        if r.n == 1:
            continue
        p = ps * mpf("0.9")
        th = [mpf(x) for x in r.theta0]
        P = r.nv + r.nz
        with mpmath.workdps(50):
            gp = r.dG_dp(p, list(range(P)))
            xs = hp.offset_slope(p, *r.column())
            G2 = [[_d2(lambda t: r.G(t, p), th, x, y) + gp[x] * gp[y] / xs for y in range(P)] for x in range(P)]
        err = _rel_err(closed_form(r, p)[0], G2)
        assert err < mpf(10) ** -25, (label, float(err))


def test_each_mutant_is_rejected():
    """Dropping the rank-one term, flipping the band's sign, X instead of X' and u_z from the next
    layer each miss T*'s second derivatives by far more than the closed form does."""
    for mutant in MUTANTS:
        worst = max(_rel_err(closed_form(r, ps, mutant)[0], D2) for _, r, ps, D2 in _tstar_second_derivatives())
        assert worst > 1e-3, (mutant, float(worst))


# ---- the binary64 reference -----------------------------------------------------------------
def _columns(r, ldv):
    return [c if c < r.nv else ldv + c - r.nv for c in range(r.nv + r.nz)]


def _check_against_exact(v, z, n, so, sd, T, P, w, kmode=False):
    """hess_batch against sum_s w_s d2T_s of the closed form in mpmath at the same p, within
    sum_s |w_s| (C u (1 + 1/cos_min^2) + S u) |terms|.  Returns the reference."""
    Hr = hess_batch(v, z, n, so, sd, T, P, w, kmode=kmode)
    B, S = T.shape
    ldv, ldz = v.shape[1], z.shape[1]
    worst = 0.0
    for b in range(B):
        ex = np.zeros((ldv + ldz, ldv + ldz), dtype=object)
        ex[:] = mpf(0)
        bd = np.zeros_like(ex)
        bd[:] = mpf(0)
        for s in range(S):
            if T[b, s] == -999.0:
                continue
            r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=ldv, ldz=ldz)
            q = mpf(float(P[b, s]))
            D2, M = closed_form(r, q, T=float(T[b, s]))
            V, _ = r.column()
            cmin2 = min(1 - (q * x) ** 2 for x in V) if r.n >= 2 else mpf(1)
            kap = C * U * (1 + 1 / cmin2) + S * U
            cols = _columns(r, ldv)
            for x, cx in enumerate(cols):
                for y, cy in enumerate(cols):
                    ex[cx, cy] += mpf(float(w[b, s])) * D2[x][y]
                    bd[cx, cy] += abs(float(w[b, s])) * kap * M[x][y]
        for i in range(ldv + ldz):
            for j in range(ldv + ldz):
                err = abs(mpf(float(Hr[b, i, j])) - ex[i, j])
                if bd[i, j] == 0:
                    assert err == 0, (b, i, j)
                else:
                    worst = max(worst, float(err / bd[i, j]))
    assert worst <= 1.0, worst
    assert _bits_equal(Hr, Hr.transpose(0, 2, 1))
    return Hr


@pytest.mark.parametrize("nl", [1, 2, 5])
def test_reference_within_the_rounding_bound(nl):
    v, z, n = workloads.make_models(3, nl, 600 + nl)
    so, sd = workloads.make_sources(6, nl)
    T, P = _forward(v, z, n, so, sd)
    w = np.random.default_rng(nl).normal(0.0, 0.05, T.shape)
    _check_against_exact(v, z, n, so, sd, T, P, w)


def test_kmode_and_the_k1_fake_interface():
    k, vp, zi = workloads.make_transd_models(8, 5, 31, uniform_k=True)
    so, sd = workloads.make_sources(5, 31)
    sd[-1] = 12000.0                                      # below the fake interface at 9999.9
    T, P = _forward(vp, zi, k, so, sd, kmode=True)
    w = np.random.default_rng(2).normal(0.0, 0.05, T.shape)
    Hr = _check_against_exact(vp, zi, k, so, sd, T, P, w, kmode=True)
    one = k == 1
    assert one.any()
    assert np.all(Hr[one][:, 1:, :] == 0) and np.all(Hr[one][:, :, 1:] == 0) and np.all(Hr[one][:, 0, 0] != 0)


def test_padding_gives_zero_rows_and_columns():
    rng = np.random.default_rng(3)
    B, ldv, ldz = 10, 12, 11
    v, z, _ = workloads.make_models(B, 6, 3)
    vp, zp = np.zeros((B, ldv)), np.full((B, ldz), 1e30)
    vp[:, :7], zp[:, :6] = v, z
    n = rng.integers(1, 7, B).astype(np.int32)
    so, sd = workloads.make_sources(18, 3)
    T, P = _forward(vp, zp, n, so, sd)
    Hr = hess_batch(vp, zp, n, so, sd, T, P, np.ones(T.shape))
    assert _bits_equal(Hr, Hr.transpose(0, 2, 1))
    for b in range(B):
        dead = np.r_[np.arange(n[b] + 1, ldv), ldv + np.arange(n[b], ldz)]
        assert np.all(Hr[b][dead] == 0) and np.all(Hr[b][:, dead] == 0)


def test_skipped_rays_zero_weights_and_one_hot_weights():
    v, z, n = workloads.make_models(8, 5, 7)
    so, sd = workloads.make_sources(15, 7)
    T, P = _forward(v, z, n, so, sd)
    w = np.random.default_rng(7).normal(0.0, 1.0, T.shape)
    T2 = T.copy()
    T2[0, :] = -999.0                      # a whole model
    T2[3, 4] = -999.0                      # one ray: as if its source were absent
    Hr = hess_batch(v, z, n, so, sd, T2, P, w)
    assert np.all(Hr[0] == 0)
    keep = np.arange(so.size) != 4
    A = hess_batch(v[3:4], z[3:4], n[3:4], so[keep], sd[keep], T2[3:4, keep], P[3:4, keep], w[3:4, keep])
    assert _bits_equal(Hr[3], A[0])
    assert np.all(hess_batch(v, z, n, so, sd, T, P, np.zeros(T.shape)) == 0)
    for s in (0, 6, 14):
        e = np.zeros(T.shape)
        e[:, s] = 1.0
        one = hess_batch(v, z, n, so[s:s + 1], sd[s:s + 1], T[:, s:s + 1], P[:, s:s + 1], np.ones((8, 1)))
        assert _bits_equal(hess_batch(v, z, n, so, sd, T, P, e), one)


def test_columns_are_central_differences_of_the_gradient():
    """H e_k of one ray at its converged p against (g(theta + h e_k) - g(theta - h e_k)) / 2h, g the
    gradient grad_reference returns at independently converged rays, to 1e-6 of max |H|."""
    v = np.array([[1800.0, 2600.0, 3300.0, 4100.0, 4800.0]])
    z = np.array([[400.0, 1100.0, 1900.0, 2600.0]])
    n = np.array([4], np.int32)
    for R, d in ((1500.0, 2300.0), (4200.0, 3000.0), (800.0, 900.0)):
        T, p = converged_ray(v[0], z[0], 4, R, d)
        Hr = hess_batch(v, z, n, [R], [d], [[T]], [[p]], [[1.0]])[0]
        theta = np.r_[v[0], z[0]]
        for k in range(theta.size):
            g = []
            for sgn in (1, -1):
                th = theta.copy()
                h = 1e-4 * abs(theta[k])
                th[k] += sgn * h
                vk, zk = th[None, :5], th[None, 5:]
                Tk, pk = converged_ray(vk[0], zk[0], 4, R, d)
                gv, gz, _, _ = grad_batch(vk, zk, n, [R], [d], [[Tk]], [[pk]], [[1.0]])
                g.append(np.r_[gv[0], gz[0]])
            fd = (g[0] - g[1]) / (2 * 1e-4 * abs(theta[k]))
            assert np.all(np.abs(Hr[:, k] - fd) <= 1e-6 * np.abs(Hr).max()), (R, d, k, Hr[:, k], fd)


def test_wrappers_refuse_bad_arguments():
    v, z, n = (torch.as_tensor(a) for a in workloads.make_models(3, 2, 1))
    n = n.to(torch.int32)
    so, sd = (torch.as_tensor(a) for a in workloads.make_sources(4, 1))
    T = torch.zeros((3, 4), dtype=torch.float64)
    with pytest.raises(ValueError, match="w must be"):
        device.dff_hess_device(v, z, n, so, sd, T, T, T[:, :3])
    with pytest.raises(ValueError, match="H must be"):
        device.dff_hess_device(v, z, n, so, sd, T, T, T, H=torch.empty((3, 5, 4), dtype=torch.float64))
    with pytest.raises(ValueError, match="CUDA tensors"):
        device.dff_hess_device(v, z, n, so, sd, T, T, T)
    with pytest.raises(ValueError, match="CUDA tensors"):
        grad.hessian(v, z, n, so, sd, T)
    with pytest.raises(ValueError, match="CUDA tensors"):
        grad.newton_equations(v, z, n, so, sd, so)
    with pytest.raises(ValueError, match="w must be"):
        raymod.dff_batch_hess(v.numpy(), z.numpy(), n.numpy(), so.numpy(), sd.numpy(), np.zeros((3, 3)))
    with pytest.raises(ValueError, match="ldv must be"):
        raymod.dff_batch_hess(np.zeros((3, 256)), z.numpy(), n.numpy(), so.numpy(), sd.numpy(), np.zeros((3, 4)))
