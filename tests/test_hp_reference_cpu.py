"""CPU checks of the high-precision reference (tests/hp_reference.py) and, through it, of the C
oracle: the layer lookup, the reference's own ray dump, the solver's stopping rule, Fermat's
identity dT*/dtheta = dG/dtheta at p* (near-critical rays included), the likelihood's normaliser
boundary, and that the comparator rejects rows with the mistakes a kernel could plausibly make."""
import math

import numpy as np
import pytest
from mpmath import mpf

import oracle
from raytracerfortran_b200 import workloads

import hp_reference as hp


def _test1(golden):
    c = golden["config1"]
    return c["vels"], c["depths"], c["src_offset_full"], c["src_depth_full"]


def test_which_layer_is_the_oracles():
    v, z, _ = workloads.make_models(20, 7, 8)
    _, sd = workloads.make_sources(24, 8)
    for b in range(z.shape[0]):
        on = list(z[b]) + [np.nextafter(x, -np.inf) for x in z[b]] + [np.nextafter(x, np.inf) for x in z[b]]
        for d in list(sd) + on + [0.0, -1.0, 1e9]:
            assert hp.which_layer(list(z[b]), d) == oracle.which_layer(z[b], d), (b, d)
    assert hp.which_layer([], 5.0) == oracle.which_layer(np.zeros(0), 5.0) == 1


def test_converged_ray_reproduces_rays_dat(golden):
    """rays.dat holds the reference's rays (delta_i, h_i per layer, 17 digits).  The ray parameter
    they imply has the printed offset, the printed travel time, and misses R by < 0.1 m; p* differs
    from it by exactly that miss: T(p_ref) - T(p*) = p* (X(p_ref) - R) to second order."""
    v, z, so, sd = _test1(golden)
    for k, ray in enumerate(golden["config1"]["rays_dat"]):
        delta, h = ray["delta"], ray["h"]
        r = hp.Ray(v, z, len(z), so[k], sd[k])
        V, H = r.column()
        assert [float(x) for x in H] == pytest.approx(h, rel=1e-15)
        i = int(np.argmax(delta))
        p_ref = mpf(delta[i]) / (mpf(delta[i]) ** 2 + mpf(h[i]) ** 2).sqrt() / mpf(v[i])
        x_ref, t_ref = r.X(p_ref), r.T(p_ref)
        assert abs(float(x_ref) - sum(delta)) <= 1e-12 * sum(delta)
        t_dump = sum(math.sqrt(a * a + b * b) / v[j] for j, (a, b) in enumerate(zip(delta, h)))
        assert abs(float(t_ref) - t_dump) <= 1e-13 * t_dump
        miss = x_ref - so[k]
        assert abs(miss) < hp.TOL
        ps = r.p_star()
        assert abs(r.X(ps) - so[k]) < mpf(10) ** -40
        slope = hp.offset_slope(ps, V, H)
        assert abs(t_ref - r.T(ps) - ps * miss) <= miss ** 2 / slope, k


def _batches():
    v, z, n = workloads.make_models(12, 10, 31)
    so, sd = workloads.make_sources(64, 31)
    yield "random", v, z, n, so, sd, False
    v, z, n = workloads.make_models(3, 50, 5, min_thickness=False)
    so, sd = workloads.make_sources(64, 5, near_critical=True)
    yield "near-critical", v, z, n, so, sd, False
    k, vp, zi = workloads.make_transd_models(40, 30, 3, uniform_k=True)
    so, sd = workloads.make_sources(24, 3)
    sd[:4] = [12000.0, 9999.9, 10500.0, 20000.0]        # below the k = 1 fake interface
    so[:4] = [10.0, 3000.0, 25000.0, 0.0]
    yield "kmode", vp, zi, k, so, sd, True


def _oracle_rays(v, z, n, so, sd, kmode):
    """(model, trace per source) as the oracle traces them (kmode: the LOGLHOOD_RT mapping)."""
    for b in range(v.shape[0]):
        if kmode:
            vv, zz = (v[b, :n[b]], z[b, :n[b] - 1]) if n[b] > 1 else ([v[b, 0]] * 2, [hp.FAKE_IFACE])
        else:
            vv, zz = v[b, :n[b] + 1], z[b, :n[b]]
        t, p, tr = oracle.trace_rays(vv, zz, so, sd, want_trace=True)
        yield b, t, p, tr


def test_oracle_p_meets_the_stopping_rule():
    """|X_exact(p) - R| < 0.1 m + the rounding bound of X at the oracle's p, for every converged
    ray with n >= 2.  The exception is a ray that used up the 15 Newton steps: the reference then
    sets conv = 1 whatever |f| is (sq:327-330, "sic"); such rays must stay rare and are named."""
    checked, capped = 0, []
    for name, v, z, n, so, sd, kmode in _batches():
        for b, t, p, tr in _oracle_rays(v, z, n, so, sd, kmode):
            for s in range(so.size):
                if t[s] == hp.NOT_CONVERGED or tr[s].nl < 2:
                    continue
                r = hp.Ray(v[b], z[b], n[b], so[s], sd[s], kmode=kmode)
                assert r.n == tr[s].nl
                miss = abs(float(r.X(p[s]) - so[s]))
                if abs(tr[s].f_final) >= hp.TOL:
                    capped.append((name, b, s, miss))
                    continue
                assert miss < hp.TOL + r.x_bound(p[s]), (name, b, s, miss)
                checked += 1
    assert checked >= 1500
    assert len(capped) <= checked // 100, capped
    print(f"stopping rule: {checked} rays within 0.1 m; Newton-cap rays: {capped}")


def _fermat_rays():
    """(label, Ray, follow_layers, directions) for the Fermat check."""
    v, z, n = workloads.make_models(4, 6, 17)
    so, sd = workloads.make_sources(6, 17)
    for b in range(2):
        yield "random", hp.Ray(v[b], z[b], n[b], so[b], sd[b]), None
    yield "n = 1", hp.Ray(v[0], z[0], n[0], 1234.5, 0.5 * z[0, 0]), None
    yield "R = 0", hp.Ray(v[1], z[1], n[1], 0.0, sd[2]), None
    vp, zi = [3100.0, 0.0], [0.0]
    yield "k = 1 below 9999.9", hp.Ray(vp, zi, 1, 4000.0, 12500.0, kmode=True), None
    yield "k = 1 above 9999.9", hp.Ray(vp, zi, 1, 4000.0, 2500.0, kmode=True), None
    yield "kmode k = 4", hp.Ray([2000.0, 3500.0, 3000.0, 5200.0], [800.0, 1900.0, 3000.0], 4, 5000.0, 3500.0,
                                kmode=True), None
    # a source exactly on an interior interface: the side on which it is below the interface
    # (n frozen there); its one-sided derivatives are those of T* followed through whichLayer
    r = hp.Ray(v[2], z[2], n[2], so[3], z[2, 2])
    assert r.n == 4 and float(r.column()[1][-1]) == 0.0
    dirs = [0] * (r.nv + r.nz + 2)
    dirs[r.nv + 2], dirs[r.id] = -1, 1
    yield "on an interface", r, dirs
    # near-critical: the offset a ray of p V_max = 1 - eps reaches
    vv, zz, _ = workloads.make_models(1, 12, 23)
    for eps in (1e-3, 1e-5, 1e-6):
        r = hp.Ray(vv[0], zz[0], 12, 0.0, 9000.0)
        V, H = r.column()
        R = float(hp.offset(mpf(1 - eps) / max(V), V, H))
        yield f"p V = 1 - {eps:g}", hp.Ray(vv[0], zz[0], 12, R, 9000.0), None


def _cols(r, limit=8):
    cols = list(range(r.nv + r.nz + 2))
    if len(cols) <= limit:
        return cols
    rng = np.random.default_rng(len(cols))
    return sorted(set(rng.choice(cols[:-2], limit - 2, replace=False).tolist()) | {r.iR, r.id})


def test_fermat_identity_at_the_converged_ray():
    """mpmath.diff of the converged T*(theta) equals dG/dtheta at p* to >= 25 digits: the claim
    DESIGN.md section 11 rests on, checked on straight rays, R = 0, both sides of the k = 1 fake
    interface, a source on an interface (one-sided) and rays up to p V = 1 - 1e-6."""
    worst = 0.0
    for label, r, dirs in _fermat_rays():
        cols = list(range(r.nv + r.nz + 2)) if dirs else _cols(r)
        ps = r.p_star()
        a = r.dG(ps, cols)
        b = r.dT_star(cols, follow_layers=dirs is not None, directions=[dirs[c] for c in cols] if dirs else None)
        scale = max(abs(x) for x in a)
        err = max(abs(x - y) for x, y in zip(a, b)) / scale
        assert err < mpf(10) ** -25, (label, float(err))
        worst = max(worst, float(err))
    print(f"Fermat: worst relative difference {worst:.1e}")


# ---- the comparator must reject rows with plausible kernel mistakes ---------------------------

def _f64_row(r, p, h_last=None, second_term=True, eta_from=lambda j: j + 1):
    """A binary64 row [dT/dV..., dT/dz..., dT/dR, dT/dd] from the closed forms, with optional
    mistakes: another last thickness, the k = 1 lower layer's velocity term dropped, eta_{j+1}
    taken from another layer."""
    th = r.theta0
    V, Z = r._model(th)
    V, Z = [float(x) for x in V], [float(x) for x in Z]
    R, d, n = th[-2], th[-1], r.n
    H = [Z[0]] + [Z[i] - Z[i - 1] for i in range(1, n - 1)] + [d - Z[n - 2]] if n >= 2 else [d]
    if h_last is not None:
        H[-1] = h_last
    cos = [math.sqrt(1.0 - p * p * (v * v)) for v in V[:n]]
    eta = [c / v for c, v in zip(cos, V)]
    term = [-(h / ((v * v) * c)) for h, v, c in zip(H, V, cos)]
    jv = [0.0] * r.nv
    for i in range(n):
        if r.fake:
            if i == 0 or second_term:
                jv[0] += term[i]
        else:
            jv[i] = term[i]
    jz = [eta[j] - eta[eta_from(j)] if j <= n - 2 else 0.0 for j in range(r.nz)]
    return jv + jz + [p, eta[n - 1]]


def _reject_ratio(r, p, row):
    cols = list(range(r.nv + r.nz + 2))
    return hp.ratio(row, r.dG(p, cols), r.row_bounds(p, cols))


def test_comparator_rejects_wrong_rows():
    v, z, n = workloads.make_models(1, 6, 41)
    v, z = v[0], z[0]
    r = hp.Ray(v, z, 6, 3000.0, 0.5 * (z[2] + z[3]))             # n = 4: three interfaces above
    p = float(r.p_star())
    good = _reject_ratio(r, p, _f64_row(r, p))
    assert good <= 1.0
    ratios = {
        "p 1e-9 off": _reject_ratio(r, p, _f64_row(r, p * (1 + 1e-9))),
        "H_{n-1} = z_{n-1} - z_{n-2}": _reject_ratio(r, p, _f64_row(r, p, h_last=z[3] - z[2])),
        "eta_{j+1} from layer j+2": _reject_ratio(r, p, _f64_row(r, p, eta_from=lambda j: min(j + 2, r.n - 1))),
    }
    k1 = hp.Ray([3100.0], [0.0], 1, 4000.0, 12500.0, kmode=True)
    assert k1.n == 2
    pk = float(k1.p_star())
    assert _reject_ratio(k1, pk, _f64_row(k1, pk)) <= 1.0
    ratios["k = 1 second velocity term dropped"] = _reject_ratio(k1, pk, _f64_row(k1, pk, second_term=False))
    # the travel time at a p 1e-9 off is rejected too
    t_off = sum(h / (v * math.sqrt(1.0 - (p * (1 + 1e-9)) ** 2 * v * v)) for v, h in
                zip([float(x) for x in r.column()[0]], [float(x) for x in r.column()[1]]))
    ratios["T at p 1e-9 off"] = abs(t_off - float(r.T(p))) / r.t_bound(p)
    print(f"correct rows: ratio {good:.3f}; wrong rows: " + ", ".join(f"{k} {v:.3g}" for k, v in ratios.items()))
    for what, x in ratios.items():
        assert x > 10.0, (what, x)


# ---- the likelihood ---------------------------------------------------------------------------

@pytest.mark.parametrize("N", [771, 772, 773])
def test_normaliser_boundary_on_the_oracle(N):
    """(2 pi)^(N/2) first overflows binary64 at N = 773: the oracle's logL is finite at 771 and
    772 (where the power is 1.25e308) and -inf from 773, as loglhood.f90:194 computes it."""
    rng = np.random.default_rng(N)
    T = rng.uniform(0.5, 2.0, N)
    tobs = T + rng.normal(0.0, 0.02, N)
    got = oracle.loglhood_from_times(T, tobs, 0.02)
    want, bound, _ = hp.loglhood(T, tobs, 0.02)
    assert hp.lognorm_overflows(N) == (N >= 773)
    if N >= 773:
        assert got == -math.inf and want == -math.inf
    else:
        assert abs(mpf(got) - want) <= bound
    want_stable, bound, _ = hp.loglhood(T, tobs, 0.02, stable=True)
    assert math.isfinite(float(want_stable))


def test_oracle_loglhood_within_the_bound():
    rng = np.random.default_rng(5)
    worst = 0.0
    for N in (1, 2, 20, 256):
        T = rng.uniform(0.5, 2.0, N)
        tobs = T + rng.normal(0.0, 0.02, N)
        for sigma in (1e-100, 1e-6, 0.016, 3.0, 1e200):
            want, bound, _ = hp.loglhood(T, tobs, sigma)
            got = oracle.loglhood_from_times(T, tobs, sigma)
            worst = max(worst, float(abs(mpf(got) - want) / bound))
            ar, bound_ar, rej = hp.loglhood(T, tobs, sigma, idxar=1, arpar=0.3, armx=0.5)
            got_ar = oracle.loglhood_from_times_ar(T, tobs, sigma, 1, 0.3, 0.5)
            assert not rej
            worst = max(worst, float(abs(mpf(got_ar) - ar) / bound_ar))
    assert worst <= 1.0
    print(f"oracle logL: worst error/bound {worst:.3g}")
