"""GPU parity: the sm_100a path, called through the C ABI, against the CPU oracle.

Bars (BASELINE.json north_star: 1e-9 relative in travel time, converged p and logL):
  * travel times and ray parameters: BIT-EXACT against the oracle (same IEEE operations in
    the same order, no FMA), which in turn is pinned to the reference's rays.dat / notebook;
  * logL: 1e-12 relative to the size of its terms (the device `log` may differ from glibc's
    by an ulp; everything else in logL is bit-exact, including the order of the residual sum).
"""
import math
import os

import numpy as np
import pytest

import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import workloads

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def assert_bitexact(got, want, what):
    g, w = bits(got), bits(want)
    bad = np.flatnonzero(g.ravel() != w.ravel())
    assert bad.size == 0, (f"{what}: {bad.size} of {g.size} differ; first at {bad[:5]}: "
                           f"{np.ravel(got)[bad[:5]]} vs {np.ravel(want)[bad[:5]]}")


def assert_logl_close(got, want, nsrc, sigma):
    scale = np.maximum(np.maximum(np.abs(want), nsrc * np.abs(np.log(sigma))), 1.0)
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got))
    assert np.all(np.abs(got[fin] - want[fin]) <= 1e-12 * scale[fin])
    assert np.array_equal(got[~fin], want[~fin])


def _reset_options():
    for name in ("variant", "threads", "tile_models", "tile_sources", "chunk_models", "ctas_per_sm",
                 "comp_streams", "static_tiles"):
        rt.set_option(name, -1 if name == "variant" else 0)
    rt.set_option("stage_pageable", -1)
    rt.set_option("latency_path", 1)


@pytest.fixture(autouse=True)
def _defaults():
    _reset_options()
    yield
    _reset_options()


# ---------------------------------------------------------------------------------------------
# config 1: the reference's shipped example, through the reference's own entry points
# ---------------------------------------------------------------------------------------------
def test_config1_dff_matches_reference_goldens(golden):
    c = golden["config1"]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    t = rt.dff(c["vels"], c["depths"], so, sd)
    t_or, p_or, _ = oracle.trace_rays(c["vels"], c["depths"], so, sd)
    assert_bitexact(t, t_or, "timeP")
    # and directly against the reference's own ray dump (rays.dat): T = sum sqrt(h^2+d^2)/v
    v = np.array(c["vels"])
    for k, ray in enumerate(c["rays_dat"]):
        d, h = np.array(ray["delta"]), np.array(ray["h"])
        t_ref = float((np.sqrt(h * h + d * d) / v[:len(h)]).sum())
        assert abs(t[k] - t_ref) <= 1e-12 * t_ref


def test_notebook_known_answers_via_tracerays_and_dff7(golden):
    n = golden["notebook"]
    t8 = rt.TraceRays(n["vels"], n["depths"], len(n["depths"]), n["src_offset"], n["src_depth"], 5)
    t7 = rt.dff7(n["vels"], n["depths"], n["src_offset"], n["src_depth"])
    assert_bitexact(t8, t7, "TraceRays vs dff7")
    for got, want in zip(t8, n["timeP_7digits"]):
        assert abs(got - want) < 0.5e-7


def test_keep_delta_writes_rays_dat(golden, tmp_path, monkeypatch):
    c = golden["config1"]
    monkeypatch.chdir(tmp_path)
    rt.dff(c["vels"], c["depths"], c["src_offset_full"], c["src_depth_full"], keep_delta=10)
    rows = [[float(x) for x in l.split()] for l in open(tmp_path / "rays.dat") if l.strip()]
    assert len(rows) == 40
    for k, ray in enumerate(c["rays_dat"]):
        assert np.allclose(rows[2 * k], ray["delta"], rtol=1e-12, atol=0)
        assert np.allclose(rows[2 * k + 1], ray["h"], rtol=1e-15, atol=0)


def test_readme_example(golden):
    r = golden["readme_example"]
    t = rt.dff(r["vels"], r["depths"], r["src_offset"], r["src_depth"])
    want, _, _ = oracle.trace_rays(r["vels"], r["depths"], r["src_offset"], r["src_depth"])
    assert_bitexact(t, want, "README example")


# ---------------------------------------------------------------------------------------------
# batched sweeps against the oracle, every kernel variant.  The "variant" option forces 3 or 5;
# every other value runs variant 1, so the sweeps below that also pass 0 and 4 check that too.
# ---------------------------------------------------------------------------------------------
BATCH_SHAPES = [(1500, 10, 64, 2), (257, 4, 20, 11), (64, 29, 256, 3), (33, 1, 7, 5)]


def _dff_batch_bitexact(variant, B, nlayers, nsrc, seed):
    rt.set_option("variant", variant)
    v, z, nl = workloads.make_models(B, nlayers, seed)
    so, sd = workloads.make_sources(nsrc, seed)
    ref = oracle.dff_batch(v, z, nl, so, sd, want_p=True)
    tobs, sigma = workloads.make_observations(ref["timeP"][0], B, seed)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    assert_bitexact(got["timeP"], ref["timeP"], "timeP")
    assert_bitexact(got["p"], ref["p"], "p")
    assert_logl_close(got["logL"], ref["logL"], nsrc, sigma)


@pytest.mark.parametrize("variant", [1, 3, 5])
@pytest.mark.parametrize("B,nlayers,nsrc,seed", BATCH_SHAPES)
def test_dff_batch_bitexact(variant, B, nlayers, nsrc, seed):
    _dff_batch_bitexact(variant, B, nlayers, nsrc, seed)
    assert rt.get_stat("variant") == variant


@pytest.mark.parametrize("variant", [0, 2, 4])
@pytest.mark.parametrize("B,nlayers,nsrc,seed", BATCH_SHAPES)
def test_dff_batch_bitexact_other_variant_values(variant, B, nlayers, nsrc, seed):
    """Option values other than 3 and 5 run variant 1, with the oracle's bits."""
    _dff_batch_bitexact(variant, B, nlayers, nsrc, seed)
    assert rt.get_stat("variant") == 1


@pytest.mark.parametrize("variant", [0, 1, 3, 4, 5])
def test_near_critical_50_layers(variant):
    """config-5 style rays: p*v -> 1, ~99 % bisection, Newton clamps."""
    rt.set_option("variant", variant)
    B, nsrc = 48, 128
    v, z, nl = workloads.make_models(B, 50, 5, min_thickness=False)
    so, sd = workloads.make_sources(nsrc, 5, near_critical=True)
    ref = oracle.dff_batch(v, z, nl, so, sd, want_p=True)
    got = rt.dff_batch(v, z, nl, so, sd, want_p=True)
    assert_bitexact(got["timeP"], ref["timeP"], "timeP")
    assert_bitexact(got["p"], ref["p"], "p")
    st = oracle.batch_stats(v, z, nl, so, sd)
    assert st["bisect"] > 0.9 * (st["rays"] - st["top"])       # the workload is what it claims to be
    assert st["sum_nl"] / st["rays"] > 20


def test_transdimensional_loglhood_batch():
    """config-3 style: k = 1..30 nodes per state, incl. the k == 1 half-space special case."""
    B, nsrc = 600, 256
    k, vp, zi = workloads.make_transd_models(B, 30, 3, uniform_k=True)
    k[:5] = 1
    so, sd = workloads.make_sources(nsrc, 3)
    t0 = oracle.loglhood_rt(vp[7, :k[7]], zi[7, :k[7] - 1], so, sd, np.zeros(nsrc), 1.0)[1]
    tobs, sigma = workloads.make_observations(t0, B, 3)
    ll, pred = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma, want_pred=True)
    want_ll = np.empty(B)
    want_pred = np.empty((B, nsrc))
    for b in range(B):
        want_ll[b], want_pred[b] = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :k[b] - 1], so, sd, tobs, sigma[b])
    assert_bitexact(pred, want_pred, "DpredRT")
    assert_logl_close(ll, want_ll, nsrc, sigma)


def test_loglhood_overflowing_normaliser_is_minus_inf_like_the_reference():
    """(2 pi)^(N/2) overflows for N >= 773, so LOG(1/inf) = -inf (loglhood.f90:194)."""
    B, nsrc = 6, 800
    v, z, nl = workloads.make_models(B, 6, 9)
    so, sd = workloads.make_sources(nsrc, 9)
    tobs, sigma = np.ones(nsrc), np.full(B, 0.02)
    got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_times=False)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
    assert np.all(np.isneginf(ref["logL"])) and np.array_equal(got["logL"], ref["logL"])


def test_fast_division_matches_builtin():
    """The hot loop's rsqrt-seeded sqrt and divisions vs CUDA's correctly rounded built-ins,
    bit for bit, on 3e9 operand triples spanning the solver's range (near-critical included)."""
    assert rt.selftest_fast_division(3e9, seed=12345) == 0


# ---------------------------------------------------------------------------------------------
# edge cases
# ---------------------------------------------------------------------------------------------
def test_edge_geometry():
    v = np.array([[3000.0, 4500.0, 2500.0, 6000.0]])
    z = np.array([[1000.0, 2000.0, 3000.0]])
    nl = np.array([3], dtype=np.int32)
    # top layer, exactly on interfaces (1000, 2000, 3000), below everything, zero offset,
    # tiny offset, very long offset (near critical), source at the surface
    sd = np.array([500.0, 1000.0, 2000.0, 3000.0, 5000.0, 2500.0, 2500.0, 2999.999, 1e-3, 1500.0])
    so = np.array([800.0, 800.0, 800.0, 800.0, 800.0, 0.0, 1e-9, 90000.0, 10.0, 1e6])
    ref = oracle.dff_batch(v, z, nl, so, sd, want_p=True)
    got = rt.dff_batch(v, z, nl, so, sd, want_p=True)
    assert_bitexact(got["timeP"], ref["timeP"], "timeP")
    assert_bitexact(got["p"], ref["p"], "p")
    assert [oracle.which_layer(z[0], d) for d in sd[:5]] == [1, 2, 3, 3, 4]


@pytest.mark.parametrize("variant", [0, 1, 3, 4, 5])
def test_ragged_batches_and_chunking(variant):
    rt.set_option("variant", variant)
    rng = np.random.default_rng(77)
    B, ldv, nsrc = 1237, 13, 300          # odd B, odd row length, sources spill over one chunk
    nl = rng.integers(0, ldv, B).astype(np.int32)       # includes NLayers = 0 (bare half-space)
    v = rng.uniform(1500, 10000, (B, ldv))
    z = np.sort(rng.uniform(100, 9000, (B, ldv - 1)), axis=1)
    so, sd = workloads.make_sources(nsrc, 77)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B, 77)
    ref = oracle.dff_batch(v, z, np.maximum(nl, 0), so, sd, tobs=tobs, sigma=sigma, want_p=True)
    for opts in ({}, {"chunk_models": 100, "tile_models": 6, "tile_sources": 64},
                 {"threads": 128, "tile_sources": 37}):
        for k_, v_ in opts.items():
            rt.set_option(k_, v_)
        got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
        assert_bitexact(got["timeP"], ref["timeP"], f"timeP {opts}")
        assert_bitexact(got["p"], ref["p"], f"p {opts}")
        assert_logl_close(got["logL"], ref["logL"], nsrc, sigma)


@pytest.mark.parametrize("variant", [1, 3, 4, 5])
def test_tile_scheduling_and_host_pipeline_options(variant):
    """Many more tiles than persistent CTAs: tiles claimed from the global counter (repeated
    launches reuse counter slots the kernel must leave zeroed), the static stride, and the host
    pipeline on one or two compute streams all give the oracle's bits."""
    rt.set_option("variant", variant)
    B, nsrc = 24000, 16
    v, z, nl = workloads.make_models(B, 10, 31)
    so, sd = workloads.make_sources(nsrc, 31)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B, 31)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
    for opts in ({"tile_models": 4}, {"tile_models": 4}, {"tile_models": 4, "static_tiles": 1},
                 {"tile_models": 4, "static_tiles": 0, "chunk_models": 1000, "comp_streams": 1},
                 {"tile_models": 8, "chunk_models": 1000, "comp_streams": 2}):
        for k_, v_ in opts.items():
            rt.set_option(k_, v_)
        for _ in range(3):
            got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
            assert_bitexact(got["timeP"], ref["timeP"], f"timeP {opts}")
            assert_logl_close(got["logL"], ref["logL"], nsrc, sigma)
    assert rt.get_stat("grid") < B // 8          # the tiles did outnumber the CTAs


@pytest.mark.parametrize("variant", [0, 1, 4, 5])
def test_more_models_per_tile_than_threads(variant):
    """Few sources and shallow models let a tile hold more models than the CTA has threads."""
    rt.set_option("variant", variant)
    B, nsrc = 5000, 3
    v, z, nl = workloads.make_models(B, 2, 91)
    so, sd = workloads.make_sources(nsrc, 91)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B, 91)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
    for opts in ({}, {"threads": 64, "tile_models": 300}, {"threads": 128, "ctas_per_sm": 1, "tile_models": 600}):
        for k_, v_ in opts.items():
            rt.set_option(k_, v_)
        got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
        assert_bitexact(got["timeP"], ref["timeP"], f"timeP {opts}")
        assert_logl_close(got["logL"], ref["logL"], nsrc, sigma)
        if opts:
            assert rt.get_stat("tile_models") > rt.get_stat("threads")


def test_tracerays_under_the_compilers_module_procedure_names(golden):
    """Objects compiled against the reference's raymod.mod call __raymod_MOD_tracerays (gfortran),
    raymod_mp_tracerays_ (ifort) or raymod_tracerays_ (nvfortran): same entry, same bits."""
    c = golden["config1"]
    so, sd = np.array(c["src_offset_full"]), np.array(c["src_depth_full"])
    want = rt.TraceRays(c["vels"], c["depths"], len(c["depths"]), so, sd, len(so))
    ref, _, _ = oracle.trace_rays(c["vels"], c["depths"], so, sd)
    assert_bitexact(want, ref, "tracerays_")
    for name in ("__raymod_MOD_tracerays", "raymod_mp_tracerays_", "raymod_tracerays_"):
        assert_bitexact(rt.TraceRays(c["vels"], c["depths"], len(c["depths"]), so, sd, len(so), symbol=name), ref, name)


def test_empty_and_single():
    v, z, nl = workloads.make_models(1, 6, 1)
    so, sd = workloads.make_sources(1, 1)
    got = rt.dff_batch(v, z, nl, so, sd)
    ref = oracle.dff_batch(v, z, nl, so, sd)
    assert_bitexact(got["timeP"], ref["timeP"], "1x1")
    out = rt.dff_batch(v[:0], z[:0], nl[:0], so, sd)
    assert out["timeP"].shape == (0, 1)
    assert rt.dff(v[0], z[0], so[:0], sd[:0]).shape == (0,)


def test_device_resident_entry_including_unaligned_rows():
    import torch
    from raytracerfortran_b200 import device
    B, nlayers, nsrc = 999, 10, 64
    v, z, nl = workloads.make_models(B + 1, nlayers, 21)
    so, sd = workloads.make_sources(nsrc, 21)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B + 1, 21)
    dev = torch.device("cuda:0")
    tv, tz = torch.from_numpy(v).to(dev), torch.from_numpy(z).to(dev)
    tn = torch.from_numpy(nl).to(dev)
    ts, td = torch.from_numpy(so).to(dev), torch.from_numpy(sd).to(dev)
    to, tg = torch.from_numpy(tobs).to(dev), torch.from_numpy(sigma).to(dev)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    out = device.dff_batch_device(tv, tz, tn, ts, td, tobs=to, sigma=tg, want_times=True, want_p=True)
    torch.cuda.synchronize()
    assert_bitexact(out["timeP"].cpu().numpy(), ref["timeP"], "device timeP")
    assert_bitexact(out["p"].cpu().numpy(), ref["p"], "device p")
    assert_logl_close(out["logL"].cpu().numpy(), ref["logL"], nsrc, sigma)
    # rows starting 8 bytes off a 16-byte boundary: the kernel must fall back from TMA to plain loads
    out = device.dff_batch_device(tv[1:], tz[1:], tn[1:], ts, td, want_times=True)
    torch.cuda.synchronize()
    assert_bitexact(out["timeP"].cpu().numpy(), ref["timeP"][1:], "unaligned rows")


# ---------------------------------------------------------------------------------------------
# full benchmark size: size-independent properties
# ---------------------------------------------------------------------------------------------
def test_config2_full_size_properties():
    """1M models x 64 sources (BASELINE.json configs[1]).  The oracle cannot sweep 64M rays in
    seconds, so: (a) a random sample of models is checked bit-exactly against the oracle,
    (b) batch invariance: the same models evaluated alone give the same bits, (c) physical
    sanity of every ray: T >= depth / fastest velocity, 0 < p < 1/vmin."""
    cfg = workloads.CONFIGS["config2"]
    B, nlayers, nsrc = cfg["B"], cfg["nlayers"], cfg["nsrc"]
    v, z, nl = workloads.make_models(B, nlayers, cfg["seed"])
    so, sd = workloads.make_sources(nsrc, cfg["seed"])
    tobs, sigma = workloads.make_observations(
        oracle.dff_batch(v[:1], z[:1], nl[:1], so, sd)["timeP"][0], B, cfg["seed"])
    got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    T, P, LL = got["timeP"], got["p"], got["logL"]
    rng = np.random.default_rng(0)
    pick = np.sort(rng.choice(B, 3000, replace=False))
    ref = oracle.dff_batch(v[pick], z[pick], nl[pick], so, sd, tobs=tobs, sigma=sigma[pick], want_p=True)
    assert_bitexact(T[pick], ref["timeP"], "sampled timeP")
    assert_bitexact(P[pick], ref["p"], "sampled p")
    assert_logl_close(LL[pick], ref["logL"], nsrc, sigma[pick])
    again = rt.dff_batch(v[pick], z[pick], nl[pick], so, sd, tobs=tobs, sigma=sigma[pick], want_p=True)
    assert_bitexact(again["timeP"], T[pick], "batch invariance timeP")
    assert_bitexact(again["logL"], LL[pick], "batch invariance logL")
    conv = T != -999.0
    assert conv.mean() > 0.999
    # sum h/(v cos) >= depth / vmax at ANY p (the solver's quirky `conv` flag lets a ray that used
    # all 15 Newton updates return the time of whatever p it ended on -- SURVEY.md hazard list)
    vertical = sd[None, :] / v.max(axis=1)[:, None]
    assert np.all(T[conv] >= vertical[conv] * (1 - 1e-12))
    assert np.all(P > 0) and np.all(P < 1.0 / 1500.0)
    assert np.all(np.isfinite(LL))


def test_warp_shuffle_likelihood_reduction_option():
    """`logl_shuffle`: the residuals of a model are reduced by a warp-shuffle tree instead of in
    source order; same terms, so logL stays within 1e-12 relative (north star: 1e-9)."""
    B, nsrc = 900, 300
    v, z, nl = workloads.make_models(B, 10, 41)
    so, sd = workloads.make_sources(nsrc, 41)
    ref = oracle.dff_batch(v, z, nl, so, sd)
    tobs, sigma = workloads.make_observations(ref["timeP"][0], B, 41)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
    rt.set_option("logl_shuffle", 1)
    try:
        got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma)
    finally:
        rt.set_option("logl_shuffle", 0)
    assert_bitexact(got["timeP"], ref["timeP"], "timeP")
    assert_logl_close(got["logL"], ref["logL"], nsrc, sigma)


def test_pageable_inputs_through_the_pinned_ring():
    """Host arrays that are ordinary pageable memory are staged through the pinned ring (forced
    here for a batch small enough to compare with the oracle, with more chunks than ring slots);
    same bits as the direct path, logL through the bounce buffer, AR arrays included."""
    B, nsrc = 6000, 24
    v, z, nl = workloads.make_models(B, 10, 17)
    so, sd = workloads.make_sources(nsrc, 17)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B, 17)
    ref = oracle.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    rt.set_option("stage_pageable", 0)
    direct = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    for opts in ({"stage_pageable": 1}, {"stage_pageable": 1, "chunk_models": 500},
                 {"stage_pageable": 1, "chunk_models": 777, "comp_streams": 1}):
        for k_, v_ in opts.items():
            rt.set_option(k_, v_)
        got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
        assert_bitexact(got["timeP"], ref["timeP"], f"timeP {opts}")
        assert_bitexact(got["p"], ref["p"], f"p {opts}")
        assert np.array_equal(got["logL"].view(np.uint64), direct["logL"].view(np.uint64))


@pytest.mark.parametrize("NL,S", [(0, 1), (1, 7), (6, 20), (6, 33), (29, 500), (50, 64), (200, 40), (10, 8192)])
def test_one_model_latency_kernel(NL, S):
    """dff_ / TraceRays on one model run the one-warp-per-ray kernel on mapped pinned memory: the
    oracle's bits in T and p, and the batch kernel's, for shallow and deep columns, one source and
    thousands, near-critical rays and sources on interfaces."""
    rng = np.random.default_rng(1000 * NL + S)
    v = rng.uniform(1500, 10000, NL + 1)
    z = np.sort(rng.uniform(100, 9500, NL))
    so, sd = workloads.make_sources(S, NL + S, near_critical=(NL >= 29))
    if NL >= 3:
        sd[:3] = z[:3]                                   # sources exactly on interfaces
    ref, p_ref, _ = oracle.trace_rays(v, z, so, sd)
    got = rt.dff_batch(v[None, :], z[None, :] if NL else np.zeros((1, 0)), np.array([NL], np.int32), so, sd, want_p=True)
    assert rt.get_stat("variant") == 9
    assert_bitexact(got["timeP"][0], ref, "timeP latency kernel")
    assert_bitexact(got["p"][0], p_ref, "p latency kernel")
    t = rt.dff(v, z, so, sd)
    assert_bitexact(t, ref, "dff_")
    rt.set_option("latency_path", 0)
    t2 = rt.dff(v, z, so, sd)
    assert rt.get_stat("variant") != 9
    assert_bitexact(t2, ref, "dff_ batch kernel")


def test_one_model_latency_kernel_hostile_inputs():
    rng = np.random.default_rng(4)
    base_v = rng.uniform(1500, 10000, 8)
    base_z = np.sort(rng.uniform(100, 9000, 7))
    so, sd = workloads.make_sources(40, 3)
    so[1], sd[2], so[3], sd[4], so[5] = 0.0, 0.0, -50.0, -10.0, np.inf
    so[6], sd[7] = np.nan, np.nan
    for case in range(8):
        v, z = base_v.copy(), base_z.copy()
        if case == 1: z[3] = z[2]
        if case == 2: v[2] = -v[2]
        if case == 3: v[1] = 0.0
        if case == 4: v *= 1e12
        if case == 5: z = z[::-1].copy()
        if case == 6: v[3] = np.nan
        if case == 7: z[4] = np.inf
        with np.errstate(all="ignore"):
            ref, p_ref, _ = oracle.trace_rays(v, z, so, sd)
        got = rt.dff_batch(v[None, :], z[None, :], np.array([7], np.int32), so, sd, want_p=True)
        assert rt.get_stat("variant") == 9
        for g_, w_, nm in ((got["timeP"][0], ref, "T"), (got["p"][0], p_ref, "p")):
            nan = np.isnan(w_)
            assert np.array_equal(np.isnan(g_), nan), (case, nm)
            assert np.array_equal(g_[~nan].view(np.uint64), w_[~nan].view(np.uint64)), (case, nm)


def test_dff_batch_status_entry_for_r():
    """dff_batch_status: every argument by pointer, status through an int* (R's .C / .Fortran
    discard return values), optional outputs selected by the want flags."""
    import ctypes as C
    from raytracerfortran_b200 import _lib
    lib = _lib.load()
    B, nsrc = 300, 12
    v, z, nl = workloads.make_models(B, 5, 3)
    so, sd = workloads.make_sources(nsrc, 3)
    tobs, sigma = workloads.make_observations(np.ones(nsrc), B, 3)
    ref = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_p=True)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    P = lambda a: a.ctypes.data_as(dp)
    ci = lambda x: C.byref(C.c_int(x))
    for name in ("dff_batch_status", "dff_batch_status_"):
        t, ll, p = np.zeros((B, nsrc)), np.zeros(B), np.zeros(0)
        want = np.array([1, 1, 0], dtype=np.int32)
        status = C.c_int(-99)
        getattr(lib, name)(P(v), P(z), nl.ctypes.data_as(ip), ci(B), ci(v.shape[1]), ci(z.shape[1]), P(so), P(sd),
                           ci(nsrc), P(t), P(tobs), P(sigma), P(ll), P(p), want.ctypes.data_as(ip), C.byref(status))
        assert status.value == 0
        assert_bitexact(t, ref["timeP"], name)
        assert np.array_equal(ll.view(np.uint64), ref["logL"].view(np.uint64))
    # an impossible call reports through the status word instead of a return value
    status = C.c_int(0)
    lib.dff_batch_status(P(v), P(z), nl.ctypes.data_as(ip), ci(B), ci(0), ci(z.shape[1]), P(so), P(sd), ci(nsrc),
                         P(t), P(tobs), P(sigma), P(ll), P(p), want.ctypes.data_as(ip), C.byref(status))
    assert status.value != 0 and "ldv" in _lib.last_error()


def test_concurrent_host_threads_are_serialised():
    """The library keeps one context per process; every public entry takes one lock, so callers on
    several host threads (ctypes drops the GIL during the call) get the answers they would get
    alone: one-model dff_ calls, batched calls and option reads interleaved from four threads."""
    import threading
    rng = np.random.default_rng(77)
    jobs = []
    for t in range(4):
        L, S, B = int(rng.integers(2, 12)), int(rng.integers(8, 80)), int(rng.integers(50, 400))
        v, z, nl = workloads.make_models(B, L, 500 + t)
        so, sd = workloads.make_sources(S, 600 + t)
        jobs.append((v, z, nl, so, sd, oracle.dff_batch(v, z, nl, so, sd)["timeP"]))
    errors = []

    def worker(t):
        v, z, nl, so, sd, want = jobs[t]
        try:
            for it in range(25):
                got = rt.dff_batch(v, z, nl, so, sd)["timeP"]
                if not np.array_equal(got.view(np.uint64), want.view(np.uint64)):
                    errors.append((t, it, "batch"))
                one = rt.dff(v[0, :nl[0] + 1], z[0, :nl[0]], so, sd)
                if not np.array_equal(np.asarray(one).view(np.uint64), want[0].view(np.uint64)):
                    errors.append((t, it, "one model"))
                rt.get_stat("variant")
        except Exception as e:                      # noqa: BLE001 - reported below
            errors.append((t, -1, repr(e)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors[:5]
