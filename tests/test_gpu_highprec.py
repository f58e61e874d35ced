"""The kernels against the independent high-precision reference (tests/hp_reference.py): travel
times, ray parameters, logL and the derivatives, each within an error bound computed from the
exact values at the same point, on the shapes where kernels go wrong.  The mpmath side runs on the
CPU, so every check samples rays rather than whole batches.  Each test prints the worst
error/bound ratio it saw (run with -s), so a change that erodes the margin shows."""
import math

import numpy as np
import pytest
import torch
from mpmath import mpf
import mpmath

import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import device, grad, workloads

import hp_reference as hp

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = hp.U


def _t(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=DEV)


def _report(record_property, what, worst, count):
    record_property(f"{what}_worst_ratio", worst)
    record_property(f"{what}_checked", count)
    print(f"\n{what}: worst error/bound {worst:.3g} over {count}")


# ---- shapes --------------------------------------------------------------------------------

def _interface_shape():
    """Sources exactly on an interface (z_3 = 4000) and one ulp either side, with the layer below
    it slower (even models) or faster (odd models) than everything above; R = 0 and very large R."""
    v, _, n = workloads.make_models(24, 6, 61)
    z = np.tile([500.0, 1500.0, 2800.0, 4000.0, 5200.0, 6500.0], (24, 1))
    top = v[:, :4].min(axis=1), v[:, :4].max(axis=1)
    v[:, 4] = np.where(np.arange(24) % 2 == 0, 0.9 * top[0], np.minimum(1.2 * top[1], 12000.0))
    d = [4000.0, np.nextafter(4000.0, 0.0), np.nextafter(4000.0, np.inf), 2500.0, 2500.0, 3000.0, 500.0,
         4000.0, 4000.0]
    R = [1500.0, 1500.0, 1500.0, 0.0, 1e6, 5e4, 0.0, 20.0, 1e5]
    return v, z, n, np.array(R), np.array(d), False


def _kmode_shape():
    k, vp, zi = workloads.make_transd_models(400, 30, 3, uniform_k=True)
    k[:60] = 1
    so, sd = workloads.make_sources(64, 3)
    sd[:16] = np.linspace(10050.0, 14000.0, 16)       # below the k = 1 fake interface at 9999.9
    sd[16] = hp.FAKE_IFACE
    return vp, zi, k, so, sd, True


def _near_critical_shape():
    v, z, n = workloads.make_models(64, 50, 5, min_thickness=False)
    so, sd = workloads.make_sources(128, 5, near_critical=True)
    return v, z, n, so, sd, False


def _wide_shape():
    rng = np.random.default_rng(254)
    B, L = 24, 254
    v = rng.uniform(workloads.VMIN, workloads.VMAX, (B, L + 1))
    z = np.cumsum(rng.uniform(20.0, 40.0, (B, L)), axis=1)
    n = rng.integers(150, L + 1, B).astype(np.int32)
    so, _ = workloads.make_sources(32, 254)
    sd = rng.uniform(100.0, z[:, -1].min() + 500.0, so.size)
    return v, z, n, so, sd, False


def _ragged_shape():
    rng = np.random.default_rng(21)
    B, ldv, ldz = 37, 16, 14
    v, z, _ = workloads.make_models(B, 13, 21)
    n = rng.integers(0, 14, B).astype(np.int32)
    vp = np.zeros((B, ldv))
    vp[:, :14] = v
    zp = np.full((B, ldz), 1e30)
    zp[:, :13] = z
    so, sd = workloads.make_sources(70, 21)
    return vp, zp, n, so, sd, False


def _many_sources_shape():
    v, z, n = workloads.make_models(50, 8, 12)
    so, sd = workloads.make_sources(300, 12)
    return v, z, n, so, sd, False


def _random_shape():
    v, z, n = workloads.make_models(300, 10, 2)
    so, sd = workloads.make_sources(64, 2)
    return v, z, n, so, sd, False


SHAPES = {"random": _random_shape, "kmode": _kmode_shape, "near_critical": _near_critical_shape,
          "wide": _wide_shape, "interfaces": _interface_shape, "ragged": _ragged_shape,
          "many_sources": _many_sources_shape}


def _sample(B, S, count, seed, first=()):
    rng = np.random.default_rng(seed)
    picks = [(b, s) for b, s in first] + [tuple(x) for x in zip(rng.integers(0, B, count), rng.integers(0, S, count))]
    return list(dict.fromkeys((int(b), int(s)) for b, s in picks))


def _first_rays(label, v, so):
    if label == "interfaces":
        return [(b, s) for b in range(3) for s in range(so.size)]
    if label == "kmode":
        return [(b, s) for b in range(4) for s in range(18)]
    return ()


def _oracle_capped(v, z, n, so, sd, kmode, b, s):
    """Whether the oracle's solve of ray (b, s) used up the Newton steps (sq:327-330, "sic")."""
    if kmode:
        vv, zz = (v[b, :n[b]], z[b, :n[b] - 1]) if n[b] > 1 else ([v[b, 0]] * 2, [hp.FAKE_IFACE])
    else:
        vv, zz = v[b, :n[b] + 1], z[b, :n[b]]
    _, _, tr = oracle.trace_rays(vv, zz, so[s:s + 1], sd[s:s + 1], want_trace=True)
    return abs(tr[0].f_final) >= hp.TOL


def check_forward(shape, T, p, rays):
    """Per ray with T != -999: T = T_exact(p) within the bound; |X_exact(p) - R| < 0.1 m + the
    bound of X; p max V < 1 over the traversed layers; for n = 1 p and T are the straight ray's
    (T against sqrt(d^2 + R^2) / V_0 itself: T(p) would amplify the rounding of p by R^2 / d^2).

    Two exemptions, both the reference's behaviour, which the oracle shares: a ray whose solve
    used up the 15 Newton steps keeps its T, converged or not (sq:327-330, "sic"); and a source
    exactly on an interface above a faster layer, where the zero-thickness layer below the source
    still enters 1/max V (sq:148, sq:299-304), so that no p in the solver's interval reaches a long
    offset (hp_reference.solve_p returns None) and the solve ends there as a Newton-cap ray.
    Returns (worst ratio, rays checked, capped rays, rays without an admissible p)."""
    v, z, n, so, sd, kmode = shape
    ldv, ldz = v.shape[1], z.shape[1]
    worst, checked, capped, no_ray = 0.0, 0, [], []
    for b, s in rays:
        if T[b, s] == hp.NOT_CONVERGED:
            continue
        r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=ldv, ldz=ldz)
        V, H = r.column()
        pk = mpf(p[b, s])
        if r.n == 1:
            with mpmath.workdps(hp.DPS):
                D = mpmath.sqrt(mpf(sd[s]) ** 2 + mpf(so[s]) ** 2)
                t_exact, p_exact = D / V[0], mpf(so[s]) / (D * V[0])
            worst = max(worst, float(abs(pk - p_exact) / (hp.C * U * p_exact + 1e-320)),
                        float(abs(mpf(T[b, s]) - t_exact) / (hp.C * U * t_exact)))
            checked += 1
            continue
        assert pk * max(V) < 1, (b, s)
        worst = max(worst, float(abs(mpf(T[b, s]) - r.T(pk)) / r.t_bound(pk)))
        checked += 1
        miss = abs(r.X(pk) - mpf(so[s]))
        if miss >= hp.TOL + r.x_bound(pk):
            assert _oracle_capped(v, z, n, so, sd, kmode, b, s), (b, s, float(miss))
            (no_ray if r.p_star() is None else capped).append((b, s))
    return worst, checked, capped, no_ray


def _forward(label, variant=-1):
    shape = SHAPES[label]()
    v, z, n, so, sd, kmode = shape
    rt.set_option("variant", variant)
    try:
        out = device.dff_batch_device(_t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd), want_times=True,
                                      want_p=True, kmode=kmode)
        torch.cuda.synchronize()
    finally:
        rt.set_option("variant", -1)
    return shape, out["timeP"].cpu().numpy(), out["p"].cpu().numpy()


@pytest.mark.parametrize("variant", [-1, 1, 3, 5])
@pytest.mark.parametrize("label", list(SHAPES))
def test_forward_against_exact_physics(label, variant, record_property):
    shape, T, p = _forward(label, variant)
    v, _, _, so, _, _ = shape
    rays = _sample(T.shape[0], T.shape[1], 24 if label in ("wide", "near_critical") else 40, 7,
                   _first_rays(label, v, so))
    worst, checked, capped, no_ray = check_forward(shape, T, p, rays)
    assert worst <= 1.0 and checked >= 20
    assert len(capped) <= max(1, checked // 50), capped
    assert label == "interfaces" or not no_ray, no_ray
    _report(record_property, f"forward {label} variant {variant}", worst,
            f"{checked} rays; Newton-cap rays {capped}; on an interface above a faster layer, no ray {no_ray}")


def test_one_model_latency_kernel(golden, record_property):
    """dff_ returns no p: its T is within p* |X(p) - R| <= p* 0.1 m (plus the second-order term)
    of the converged T(p*), the first-order effect of the solver's stopping rule."""
    c = golden["config1"]
    cases = [(c["vels"], c["depths"], c["src_offset_full"], c["src_depth_full"])]
    v, z, _ = workloads.make_models(4, 6, 77)
    so, sd = workloads.make_sources(24, 77)
    cases += [(v[b], z[b], so, sd) for b in range(4)]
    worst, checked = 0.0, 0
    for vv, zz, oo, dd in cases:
        t = rt.dff(vv, zz, oo, dd)
        for s in range(len(oo)):
            if t[s] == hp.NOT_CONVERGED:
                continue
            r = hp.Ray(vv, zz, len(zz), oo[s], dd[s])
            ps = r.p_star()
            V, H = r.column()
            slope = hp.offset_slope(ps, V, H)
            bound = ps * hp.TOL + hp.TOL ** 2 / slope + r.t_bound(ps) if r.n > 1 else r.t_bound(ps)
            worst = max(worst, float(abs(mpf(t[s]) - r.T(ps)) / bound))
            checked += 1
    assert worst <= 1.0 and checked >= 100
    _report(record_property, "dff_", worst, checked)


# ---- derivatives ---------------------------------------------------------------------------

def _columns(r, rng, limit=12):
    """At most `limit` parameter columns: all for narrow models, else the ones next to the source
    layer, the first, R and d, and a random rest."""
    allc = list(range(r.nv + r.nz + 2))
    if len(allc) <= limit:
        return allc
    near = {0, r.n - 1, r.n, r.nv + max(r.n - 2, 0), r.nv + r.n - 1, r.iR, r.id}
    near = {c for c in near if 0 <= c < len(allc)}
    rest = [c for c in allc if c not in near]
    return sorted(near | set(rng.choice(rest, max(limit - len(near), 0), replace=False).tolist()))


def check_rows(shape, T, p, J, rays, seed=0):
    """jvels / jdepths / dtdr / dtdd rows against mpmath.diff of G at the kernel's own p.  Columns
    past the row's parameters (padding, the k = 1 fake interface) must be exact zeros.  At a
    source on an interface the kernel returns the one-sided derivative on the side where the
    source is below the interface (n frozen), which is what G at frozen n gives."""
    v, z, n, so, sd, kmode = shape
    ldv, ldz = v.shape[1], z.shape[1]
    rng = np.random.default_rng(seed)
    worst, checked, entries = 0.0, 0, 0
    for b, s in rays:
        if T[b, s] == hp.NOT_CONVERGED:
            assert not J["jvels"][b, s].any() and not J["jdepths"][b, s].any()
            continue
        r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=ldv, ldz=ldz)
        assert not J["jvels"][b, s, r.nv:].any() and not J["jdepths"][b, s, r.nz:].any(), (b, s)
        row = np.concatenate([J["jvels"][b, s, :r.nv], J["jdepths"][b, s, :r.nz], [J["dtdr"][b, s], J["dtdd"][b, s]]])
        cols = _columns(r, rng)
        worst = max(worst, hp.ratio(row[cols], r.dG(p[b, s], cols), r.row_bounds(p[b, s], cols)))
        checked += 1
        entries += len(cols)
    return worst, checked, entries


def _jacobian(shape):
    v, z, n, so, sd, kmode = shape
    J = grad.jacobian(_t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd), kmode=kmode)
    torch.cuda.synchronize()
    return {k: x.cpu().numpy() for k, x in J.items()}


@pytest.mark.parametrize("label", list(SHAPES))
def test_jacobian_rows_against_exact_derivatives(label, record_property):
    shape = SHAPES[label]()
    J = _jacobian(shape)
    v, _, _, so, _, _ = shape
    rays = _sample(J["timeP"].shape[0], J["timeP"].shape[1], 12 if label in ("wide", "near_critical") else 24,
                   11, _first_rays(label, v, so)[:30])
    worst, checked, entries = check_rows(shape, J["timeP"], J["p"], J, rays)
    assert worst <= 1.0 and checked >= 10
    _report(record_property, f"Jacobian rows {label}", worst, f"{checked} rays, {entries} entries")


def check_converged(shape, J, rays, ncols=6):
    """The kernel's row minus mpmath.diff of the converged T*(theta) stays within the stopping-rule
    bound max|dJ/dp| |p - p*| (taken at both ends of [p, p*]) plus the row's rounding bound."""
    v, z, n, so, sd, kmode = shape
    rng = np.random.default_rng(3)
    worst, checked = 0.0, 0
    for b, s in rays:
        if J["timeP"][b, s] == hp.NOT_CONVERGED:
            continue
        r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=v.shape[1], ldz=z.shape[1])
        cols = _columns(r, rng, ncols)
        pk, ps = mpf(J["p"][b, s]), r.p_star()
        row = np.concatenate([J["jvels"][b, s, :r.nv], J["jdepths"][b, s, :r.nz],
                              [J["dtdr"][b, s], J["dtdd"][b, s]]])[cols]
        star = r.dT_star(cols)
        slope = [max(abs(a), abs(c)) for a, c in zip(r.dG_dp(pk, cols), r.dG_dp(ps, cols))]
        bound = [float(1.5 * g * abs(pk - ps)) + rb for g, rb in zip(slope, r.row_bounds(pk, cols))]
        worst = max(worst, hp.ratio(row, star, bound, noise=1e-25))
        checked += 1
    return worst, checked


@pytest.mark.parametrize("label", ["near_critical", "kmode"])
def test_jacobian_rows_against_the_converged_ray(label, record_property):
    shape = SHAPES[label]()
    J = _jacobian(shape)
    rays = _sample(J["timeP"].shape[0], J["timeP"].shape[1], 8, 5, [(0, 0), (0, 16)] if label == "kmode" else ())
    worst, checked = check_converged(shape, J, rays)
    assert worst <= 1.0 and checked >= 6
    _report(record_property, f"Fermat {label}", worst, checked)


def check_vjp(shape, T, p, w, g, models):
    """dff_grad_device's sums against sum_s w_s dG_s/dtheta over every column of the model."""
    v, z, n, so, sd, kmode = shape
    worst = 0.0
    for b in models:
        r0 = hp.Ray(v[b], z[b], n[b], so[0], sd[0], kmode=kmode, ldv=v.shape[1], ldz=z.shape[1])
        cols = list(range(r0.nv + r0.nz))
        exact, bound, mag = [mpf(0)] * len(cols), [0.0] * len(cols), [mpf(0)] * len(cols)
        for s in range(so.size):
            if T[b, s] == hp.NOT_CONVERGED:
                continue
            r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode, ldv=v.shape[1], ldz=z.shape[1])
            ws = mpf(w[b, s])
            for i, (d, rb) in enumerate(zip(r.dG(p[b, s], cols), r.row_bounds(p[b, s], cols))):
                exact[i] += ws * d
                mag[i] += abs(ws * d)
                bound[i] += abs(float(ws)) * rb
        bound = [bd + float(so.size * U * m) for bd, m in zip(bound, mag)]
        got = np.concatenate([g["gvels"][b, :r0.nv], g["gdepths"][b, :r0.nz]])
        assert not g["gvels"][b, r0.nv:].any() and not g["gdepths"][b, r0.nz:].any()
        worst = max(worst, hp.ratio(got, exact, bound))
    return worst


@pytest.mark.parametrize("label", ["random", "kmode", "interfaces"])
def test_gradient_vjp_against_exact_sums(label, record_property):
    v, z, n, so, sd, kmode = SHAPES[label]()
    B = 3
    so, sd = so[:16], sd[:16]
    shape = (v[:B], z[:B], n[:B], so, sd, kmode)
    tv, tz, tn, tso, tsd = _t(v[:B]), _t(z[:B]), _t(n[:B], torch.int32), _t(so), _t(sd)
    out = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True, want_p=True, kmode=kmode)
    w = torch.as_tensor(np.random.default_rng(4).normal(size=(B, so.size)), device=DEV)
    g = device.dff_grad_device(tv, tz, tn, tso, tsd, out["timeP"], out["p"], w, kmode=kmode)
    torch.cuda.synchronize()
    g = {k: x.cpu().numpy() for k, x in g.items() if x is not None}
    worst = check_vjp(shape, out["timeP"].cpu().numpy(), out["p"].cpu().numpy(), w.cpu().numpy(), g, range(B))
    assert worst <= 1.0
    _report(record_property, f"VJP {label}", worst, f"{B} models x {so.size} sources")


def test_loglhood_gradients_wrt_sigma_and_tobs(record_property):
    v, z, n = workloads.make_models(4, 6, 19)
    so, sd = workloads.make_sources(16, 19)
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    T = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True)["timeP"]
    rng = np.random.default_rng(19)
    tobs = _t(T[0].cpu().numpy() + rng.normal(0.0, 0.02, so.size)).requires_grad_(True)
    sigma = _t(rng.uniform(0.005, 0.05, 4)).requires_grad_(True)
    grad.loglhood(tv, tz, tn, tso, tsd, tobs, sigma).sum().backward()
    Tn, ob, sg = T.cpu().numpy(), tobs.detach().cpu().numpy(), sigma.detach().cpu().numpy()
    N = so.size
    worst = 0.0
    with mpmath.workdps(hp.DPS):
        res = [[mpf(ob[s]) - mpf(Tn[b, s]) for s in range(N)] for b in range(4)]
        for b in range(4):
            ss = mpmath.fsum(x * x for x in res[b])
            exact = mpmath.diff(lambda q: -ss / (2 * q * q) - N * mpmath.log(q), mpf(sg[b]))
            bound = (N + hp.C) * U * (ss / mpf(sg[b]) ** 3 + N / mpf(sg[b]))
            worst = max(worst, hp.ratio([sigma.grad[b].item()], [exact], [float(bound)]))
        for s in range(N):
            f = lambda x: mpmath.fsum(-((x - mpf(Tn[b, s])) ** 2) / (2 * mpf(sg[b]) ** 2) for b in range(4))
            exact = mpmath.diff(f, mpf(ob[s]))
            mag = mpmath.fsum(abs(res[b][s]) / mpf(sg[b]) ** 2 for b in range(4))
            worst = max(worst, hp.ratio([tobs.grad[s].item()], [exact], [float((hp.C + 4) * U * mag)]))
    assert worst <= 1.0
    _report(record_property, "grad.loglhood sigma, tobs", worst, f"4 sigmas, {N} tobs")


# ---- the likelihood ------------------------------------------------------------------------

def check_logl(got, T, tobs, sigma, stable=False, idxar=None, arpar=None, armx=0.5):
    worst = 0.0
    for b in range(got.size):
        want, bound, rejected = hp.loglhood(T[b], tobs, sigma[b], stable=stable,
                                            idxar=0 if idxar is None else idxar[b],
                                            arpar=0.0 if arpar is None else arpar[b], armx=armx)
        if rejected:
            assert got[b] == -hp.DBL_MAX, b
            continue
        w = hp.as_double(want)
        if math.isinf(w):
            assert got[b] == w, (b, got[b], float(want))
            continue
        worst = max(worst, float(abs(mpf(got[b]) - want) / bound))
    return worst


def _small_models(B, nsrc, seed):
    v, z, n = workloads.make_models(B, 4, seed)
    so, sd = workloads.make_sources(nsrc, seed)
    return v, z, n, so, sd


@pytest.mark.parametrize("shuffle", [0, 1])
@pytest.mark.parametrize("stable", [0, 1])
@pytest.mark.parametrize("N", [64, 771, 772, 773])
def test_dff_batch_device_logl(N, stable, shuffle, record_property):
    """logL at the kernel's own T, both residual orders and both normaliser constants.  The
    constant LOG(1/(2 pi)^(N/2)) first overflows at N = 773; sigma from 1e-100 to 1e200, and a
    residual whose square overflows (logL = -inf, the correctly rounded value)."""
    v, z, n, so, sd = _small_models(6, N, N)
    rng = np.random.default_rng(N)
    sigma = np.array([1e-100, 1e-6, 0.016, 3.0, 1e200, 0.02])
    tv, tz, tn, tso, tsd = _t(v), _t(z), _t(n, torch.int32), _t(so), _t(sd)
    T = device.dff_batch_device(tv, tz, tn, tso, tsd, want_times=True)["timeP"].cpu().numpy()
    tobs = T[0] + rng.normal(0.0, 0.02, N)
    rt.set_option("stable_lognorm", stable)
    rt.set_option("logl_shuffle", shuffle)
    try:
        out = device.dff_batch_device(tv, tz, tn, tso, tsd, tobs=_t(tobs), sigma=_t(sigma), want_times=True)
        # a residual whose square overflows: ss = Inf and logL = -Inf, the correctly rounded value
        # (with sigma^2 = Inf as well it would be Inf/Inf = NaN and -HUGE, ll:200-203: not used)
        tobs_big, sigma_big = tobs.copy(), np.where(sigma > 1e150, 1e6, sigma)
        tobs_big[N // 2] = 1e200
        big = device.dff_batch_device(tv, tz, tn, tso, tsd, tobs=_t(tobs_big), sigma=_t(sigma_big), want_times=True)
        torch.cuda.synchronize()
    finally:
        rt.set_option("stable_lognorm", 0)
        rt.set_option("logl_shuffle", 0)
    got, Tk = out["logL"].cpu().numpy(), out["timeP"].cpu().numpy()
    assert np.array_equal(Tk.view(np.uint64), T.view(np.uint64))
    if N >= 773 and not stable:
        assert np.all(np.isneginf(got))
    else:
        assert np.all(np.isfinite(got))
    worst = check_logl(got, Tk, tobs, sigma, stable=bool(stable))
    assert np.all(np.isneginf(big["logL"].cpu().numpy()))
    check_logl(big["logL"].cpu().numpy(), Tk, tobs_big, sigma_big, stable=bool(stable))
    assert worst <= 1.0
    _report(record_property, f"logL dff_batch_device N={N} stable={stable} shuffle={shuffle}", worst, 6)


def _kmode_states(B, nsrc, seed):
    k, vp, zi = workloads.make_transd_models(B, 12, seed, uniform_k=True)
    k[0] = 1
    so, sd = workloads.make_sources(nsrc, seed)
    return k, vp, zi, so, sd


def test_loglhood_batch_and_voro(record_property):
    k, vp, zi, so, sd = _kmode_states(24, 48, 8)
    rng = np.random.default_rng(8)
    sigma = rng.uniform(0.005, 0.05, k.size)
    sigma[:2] = [1e-100, 1e200]
    ll0, pred0 = rt.loglhood_batch(k, vp, zi, so, sd, np.zeros(so.size), np.ones(k.size), want_pred=True)
    tobs = pred0[1] + rng.normal(0.0, 0.02, so.size)
    ll, pred = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma, want_pred=True)
    worst = check_logl(ll, pred, tobs, sigma)
    # the same states as unsorted Voronoi nodes: node 0 at depth 0, node i at ziface(i-1), shuffled
    ldk = vp.shape[1]
    voro = np.zeros((k.size, 2, ldk))
    for b in range(k.size):
        order = rng.permutation(np.arange(1, k[b]))
        dep = np.concatenate([[0.0], zi[b, :k[b] - 1]])
        idx = np.concatenate([[0], order])
        voro[b, 0, :k[b]], voro[b, 1, :k[b]] = dep[idx], vp[b, :k[b]][idx]
    llv, predv, _ = rt.loglhood_batch_voro(k, voro, so, sd, tobs, sigma, want_pred=True)
    assert np.array_equal(predv.view(np.uint64), pred.view(np.uint64))
    worst = max(worst, check_logl(llv, predv, tobs, sigma))
    assert worst <= 1.0
    _report(record_property, "logL loglhood_batch / _voro", worst, 2 * k.size)


def test_loglhood_batch_ar_and_its_bound(record_property):
    """The AR(1) form, and states whose largest |DarRT| is exactly armx (kept: the reference
    rejects only beyond it, ll:686-695) or one ulp above armx (rejected: logL = -HUGE)."""
    k, vp, zi, so, sd = _kmode_states(16, 40, 9)
    rng = np.random.default_rng(9)
    sigma = rng.uniform(0.005, 0.05, k.size)
    _, pred = rt.loglhood_batch(k, vp, zi, so, sd, np.zeros(so.size), np.ones(k.size), want_pred=True)
    tobs = pred[2] + rng.normal(0.0, 0.02, so.size)
    idx = np.ones(k.size, np.int32)
    idx[::4] = 0
    ap = rng.uniform(-0.4, 0.4, k.size)
    ll, predk = rt.loglhood_batch_ar(k, vp, zi, so, sd, tobs, sigma, idx, ap, armxRT=10.0, want_pred=True)
    worst = check_logl(ll, predk, tobs, sigma, idxar=idx, arpar=ap, armx=10.0)
    # one state at the bound: armx = its largest |arpar * res(i-1)| as binary64 computes it
    b = 1
    dar = ap[b] * (tobs - predk[b])[:-2]
    armx = float(np.max(np.abs(dar)))
    for a, keep in ((armx, True), (np.nextafter(armx, 0.0), False)):
        llb, _ = rt.loglhood_batch_ar(k[b:b + 1], vp[b:b + 1], zi[b:b + 1], so, sd, tobs, sigma[b:b + 1],
                                      idx[b:b + 1], ap[b:b + 1], armxRT=a)
        ref = oracle.loglhood_from_times_ar(predk[b], tobs, sigma[b], 1, ap[b], a)
        assert (llb[0] != -hp.DBL_MAX) == keep and (ref != -hp.DBL_MAX) == keep, (a, llb[0], ref)
        if keep:
            want, bound, _ = hp.loglhood(predk[b], tobs, sigma[b], idxar=1, arpar=ap[b], armx=10.0)
            worst = max(worst, float(abs(mpf(llb[0]) - want) / bound))
    assert worst <= 1.0
    _report(record_property, "logL loglhood_batch_ar", worst, k.size + 1)
