"""GPU parity on the shapes of BASELINE.json configs 3, 4 and 5 (config 1 and 2 are in
test_gpu_parity.py).  Where the full configuration is too large for the oracle, a slice of the
models is compared bit for bit and the rest through batch invariance."""
import numpy as np
import pytest

import oracle
import raytracerfortran_b200 as rt
from raytracerfortran_b200 import workloads

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def logl_close(got, want, nsrc, sigma):
    scale = np.maximum(np.maximum(np.abs(want), nsrc * np.abs(np.log(sigma))), 1.0)
    return np.all(np.abs(got - want) <= 1e-12 * scale)


def test_config3_transdimensional_step():
    """4096 models/step, k = 1..30 (truncated Poisson, lambda 3.01), 256 sources, logL fused."""
    cfg = workloads.CONFIGS["config3"]
    B, nsrc = cfg["B"], cfg["nsrc"]
    k, vp, zi = workloads.make_transd_models(B, cfg["kmax"], cfg["seed"])
    so, sd = workloads.make_sources(nsrc, cfg["seed"])
    t0 = oracle.loglhood_rt(vp[0, :k[0]], zi[0, :max(k[0] - 1, 0)], so, sd, np.zeros(nsrc), 1.0)[1]
    tobs, sigma = workloads.make_observations(t0, B, cfg["seed"])
    ll, pred = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma, want_pred=True)
    pick = np.arange(0, B, 9)
    for b in pick:
        w_ll, w_pred = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :max(k[b] - 1, 0)], so, sd, tobs, sigma[b])
        assert np.array_equal(bits(pred[b]), bits(w_pred))
        assert logl_close(np.array([ll[b]]), np.array([w_ll]), nsrc, sigma[b:b + 1])
    assert np.all(np.isfinite(ll))
    assert (k == 1).any() and (k > 8).any()


def test_config4_replicas_on_one_rank():
    """One rank's share of config 4: 8 replicas x 1024 proposals x 256 sources, evaluated on
    device-resident tensors in one launch, then one (single-rank) swap round."""
    import torch
    from raytracerfortran_b200 import tempering
    cfg = workloads.CONFIGS["config4"]
    R, P, nsrc, kmax = 8, cfg["proposals"], cfg["nsrc"], cfg["kmax"]
    k, vp, zi = workloads.make_transd_models(R * P, kmax, cfg["seed"])
    so, sd = workloads.make_sources(nsrc, cfg["seed"])
    t0 = oracle.loglhood_rt(vp[1, :k[1]], zi[1, :max(k[1] - 1, 0)], so, sd, np.zeros(nsrc), 1.0)[1]
    tobs, sigma = workloads.make_observations(t0, R * P, cfg["seed"])
    dev = torch.device("cuda:0")
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ll = tempering.evaluate_replicas(f(k).reshape(R, P), f(vp).reshape(R, P, kmax),
                                     f(zi).reshape(R, P, kmax - 1), f(so), f(sd), f(tobs),
                                     f(sigma).reshape(R, P))
    torch.cuda.synchronize()
    ll = ll.cpu().numpy().reshape(-1)
    for b in range(0, R * P, 37):
        w_ll, _ = oracle.loglhood_rt(vp[b, :k[b]], zi[b, :max(k[b] - 1, 0)], so, sd, tobs, sigma[b])
        assert logl_close(np.array([ll[b]]), np.array([w_ll]), nsrc, sigma[b:b + 1])
    # the replicas' current states: best proposal of each; one swap round on a single rank
    cur = torch.from_numpy(ll.reshape(R, P).max(axis=1).copy())
    beta = torch.from_numpy(tempering.temperature_ladder(R, 1.4))
    new_beta, st = tempering.tempering_swap_round(cur, beta, seed=4, round_index=0)
    assert sorted(new_beta.tolist()) == sorted(beta.tolist()) and st["bytes_per_rank"] == 16 * R


def test_config5_stress_slice():
    """config-5 shape at reduced model count: 50 interfaces, 1024 near-critical sources
    (4 source chunks per tile), logL fused and no travel-time store."""
    cfg = workloads.CONFIGS["config5"]
    B, nsrc = 600, cfg["nsrc"]
    v, z, nl = workloads.make_models(B, cfg["nlayers"], cfg["seed"], min_thickness=False)
    so, sd = workloads.make_sources(nsrc, cfg["seed"], near_critical=True)
    tobs, sigma = workloads.make_observations(np.full(nsrc, 2.0), B, cfg["seed"])
    got = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_times=True, want_p=True)
    pick = np.arange(0, B, 25)
    ref = oracle.dff_batch(v[pick], z[pick], nl[pick], so, sd, tobs=tobs, sigma=sigma[pick], want_p=True)
    assert np.array_equal(bits(got["timeP"][pick]), bits(ref["timeP"]))
    assert np.array_equal(bits(got["p"][pick]), bits(ref["p"]))
    # N = 1024 overflows the reference's normaliser: logL = -inf on both sides (loglhood.f90:194)
    assert np.array_equal(got["logL"][pick], ref["logL"])
    only_ll = rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_times=False)
    assert np.array_equal(only_ll["logL"], got["logL"])
    assert np.all(np.isneginf(got["logL"]))
    # opt-in deviation: the same constant as -(N/2) log(2 pi) keeps logL finite for N >= 773
    rt.set_option("stable_lognorm", 1)
    try:
        st = rt.dff_batch(v[pick], z[pick], nl[pick], so, sd, tobs=tobs, sigma=sigma[pick], want_times=True)
    finally:
        rt.set_option("stable_lognorm", 0)
    assert np.array_equal(bits(st["timeP"]), bits(ref["timeP"]))
    res = tobs[None, :] - ref["timeP"]
    sg = sigma[pick]
    want = -(nsrc / 2.0) * np.log(2 * np.pi) - ((res * res).sum(axis=1) / (2 * sg * sg) + nsrc * np.log(sg))
    assert np.all(np.isfinite(st["logL"])) and np.allclose(st["logL"], want, rtol=1e-12, atol=0)


def test_next_row_n1_device_side_interplayer_novar():
    """SURVEY.md section 8f, N1: chain states arrive as UNSORTED Voronoi nodes; the device sorts
    them with the reference's quicksort (ties included) and evaluates LOGLHOOD."""
    rng = np.random.default_rng(17)
    B, kmax, nsrc = 3000, 30, 64
    k, vp, zi = workloads.make_transd_models(B, kmax, 8, uniform_k=True)
    voro = np.zeros((B, 2, kmax))
    for b in range(B):
        kb = k[b]
        dep = np.concatenate(([0.0], zi[b, :kb - 1]))
        perm = rng.permutation(kb)
        voro[b, 0, :kb] = dep[perm]
        voro[b, 1, :kb] = vp[b, :kb][perm]
    # ties in depth: the result depends on where the reference's Hoare partition leaves them
    voro[:200, 0, 1] = voro[:200, 0, 0]
    so, sd = workloads.make_sources(nsrc, 8)
    tobs, sigma = workloads.make_observations(np.full(nsrc, 1.2), B, 8)
    ll, pred, srt = rt.loglhood_batch_voro(k, voro, so, sd, tobs, sigma, want_pred=True, want_sorted=True)
    for b in list(range(0, 260, 7)) + list(range(260, B, 41)):
        kb = k[b]
        w_ll, w_pred, w_d, w_v = oracle.loglhood_voro(voro[b, 0, :kb], voro[b, 1, :kb], so, sd, tobs, sigma[b])
        assert np.array_equal(srt[b, 0, :kb], w_d) and np.array_equal(srt[b, 1, :kb], w_v)
        assert np.array_equal(bits(pred[b]), bits(w_pred))
        assert logl_close(np.array([ll[b]]), np.array([w_ll]), nsrc, sigma[b:b + 1])
    # sorted input: identical to loglhood_batch on the prepared rows
    ll2, _ = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma)
    same_rows = np.arange(200, B)
    voro2 = np.zeros((B, 2, kmax))
    voro2[:, 1, :] = vp
    voro2[:, 0, 1:] = zi
    ll3, _, _ = rt.loglhood_batch_voro(k, voro2, so, sd, tobs, sigma)
    assert np.array_equal(bits(ll3[same_rows]), bits(ll2[same_rows]))


def test_next_row_n4_ar1_residual_model():
    """SURVEY.md section 8f, N4: IAR = 1 -- ARPRED_RT (order 1) + CHECKBOUNDS_ARMXRT fused into the
    likelihood (loglhood.f90:171-182,616-701), incl. states rejected by the |DarRT| bound, states
    with the AR model switched off, and sources spilling over several chunks."""
    rng = np.random.default_rng(23)
    for B, nsrc in ((700, 64), (90, 300)):
        k, vp, zi = workloads.make_transd_models(B, 12, 9, uniform_k=True)
        so, sd = workloads.make_sources(nsrc, 9)
        t0 = oracle.loglhood_rt(vp[3, :k[3]], zi[3, :max(k[3] - 1, 0)], so, sd, np.zeros(nsrc), 1.0)[1]
        tobs, sigma = workloads.make_observations(t0, B, 9)
        idx = (rng.random(B) < 0.7).astype(np.int32)
        ar = rng.uniform(-0.9, 0.9, B)
        ar[:40] = rng.uniform(3.0, 30.0, 40)            # large coefficients: |DarRT| > armx for most
        ll, pred = rt.loglhood_batch_ar(k, vp, zi, so, sd, tobs, sigma, idx, ar, armxRT=0.5, want_pred=True)
        plain, _ = rt.loglhood_batch(k, vp, zi, so, sd, tobs, sigma)
        rejected = 0
        for b in range(B):
            want = oracle.loglhood_from_times_ar(pred[b], tobs, sigma[b], idx[b], ar[b], 0.5)
            if want == -np.finfo(float).max:
                rejected += 1
                assert ll[b] == want
            else:
                assert logl_close(np.array([ll[b]]), np.array([want]), nsrc, sigma[b:b + 1])
            if idx[b] == 0:
                assert ll[b] == plain[b]
        assert rejected > 0


def test_next_row_n3_replica_sweep_over_a_sample_file(tmp_path):
    """SURVEY.md section 8f, N3: parse a `_voro_sample.txt`, rebuild every kept state and
    re-evaluate LOGLHOOD in one batched call (replica.f90:173-232)."""
    from raytracerfortran_b200 import samplefile
    B, nlmx, nsrc = 500, 10, 20
    k, vp, zi = workloads.make_transd_models(B, nlmx, 14, uniform_k=True)
    rng = np.random.default_rng(14)
    voro = np.zeros((B, 2, nlmx))
    for b in range(B):                                   # nodes in the sampler's arbitrary order
        perm = rng.permutation(k[b])
        voro[b, 0, :k[b]] = np.concatenate(([0.0], zi[b, :k[b] - 1]))[perm]
        voro[b, 1, :k[b]] = vp[b, :k[b]][perm]
    so, sd = workloads.make_sources(nsrc, 14)
    sig = rng.uniform(0.001, 0.07, B)
    rows = samplefile.pack_rows(np.zeros(B), np.zeros(B), np.zeros(B), k, voro, sig)
    path = tmp_path / "t_voro_sample.txt"
    samplefile.write_samples(path, rows)
    tobs = 1.0 + 0.3 * rng.random(nsrc)
    smp, ll, pred = samplefile.replica_sweep(path, nlmx, so, sd, tobs, burnin=50, thin=2)
    assert len(ll) == len(range(50, B, 2))
    for j in range(0, len(ll), 9):                       # oracle on the file's (9-digit) states
        kb = smp["k"][j]
        w_ll, w_pred, _, _ = oracle.loglhood_voro(smp["voro"][j, 0, :kb], smp["voro"][j, 1, :kb], so, sd,
                                                  tobs, smp["sdparRT"][j, 0])
        assert np.array_equal(bits(pred[j]), bits(w_pred))
        assert logl_close(np.array([ll[j]]), np.array([w_ll]), nsrc, smp["sdparRT"][j])


def test_default_kernel_choice_by_shape():
    """Which kernel the library picks on its own (rt_api.cu choose_cfg): the deep-model kernel from
    40 velocities per row; for shallow models the segment kernel (5) when the batch is a long queue
    of tiles or a single wave of full tiles, the shared-pointer kernel (1) in between; the one-model
    kernel (reported as 9) for a single model.  The results are bit-identical whichever runs (the
    parity tests force each one); this pins the rule itself."""
    import torch
    from raytracerfortran_b200 import device
    dev = torch.device("cuda:0")
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sms = int(rt.get_stat("sms")) or 148

    def variant_for(B, L, S, kmode=False, seed=3):
        if kmode:
            n, v, z = workloads.make_transd_models(B, L, seed)
        else:
            v, z, n = workloads.make_models(B, L, seed)
        so, sd = workloads.make_sources(S, seed)
        out = device.dff_batch_device(f(v), f(z), f(n.astype(np.int32)), f(so), f(sd), want_times=True,
                                      kmode=kmode)
        torch.cuda.synchronize()
        slots = sms * int(rt.get_stat("ctas_per_sm"))
        tiles = -(-B // int(rt.get_stat("tile_models")))
        return int(rt.get_stat("variant")), tiles, slots

    rt.set_option("variant", -1)
    v, tiles, slots = variant_for(8 * sms * 4 * 32, 10, 64)          # a long queue of tiles
    assert tiles >= 6 * slots and v == 5
    v, tiles, slots = variant_for(3 * sms * 4 * 32, 10, 64)          # three rounds
    assert slots < tiles < 6 * slots and v == 1
    v, tiles, slots = variant_for(4096, 30, 256, kmode=True)         # one wave of full tiles (config 3)
    assert tiles <= slots and v == 5
    v, _, _ = variant_for(2048, 50, 128)                             # deep models
    assert v == 3
