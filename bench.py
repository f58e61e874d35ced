#!/usr/bin/env python
"""bench.py -- the hot path's headline benchmark (see DESIGN.md).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload at every N: BASELINE.json configs[1], "batched forward sweep: 1M random 10-layer
models x 64 sources, fp64" PER GPU (weak scaling: the model axis is sharded, no data-path
collective), with the Gaussian log-likelihood fused (one logL per model).  One step = one pass
of the hot path over that batch.

  value   (model x source) travel-time evaluations / s, inputs resident in HBM, CUDA events
  e2e     the same through the C ABI entry dff_batch with pinned HOST buffers: H2D of the
          models, kernel, D2H of logL inside the timed region
  roofline   FP64 pipe: W_min flops per evaluation (counted by the instrumented oracle on a
          sample of the same inputs) x evaluations / kernel time, against the FP64 FMA peak
          measured live on the same device by the library's DFMA microbenchmark
  cpu_baseline   the CPU oracle (a C restatement of the reference's gfortran path; the Fortran
          itself cannot be built here) on all host cores, on a bounded sample of the workload

  e2e.pageable   the same call from ordinary (pageable) numpy arrays, as R or Fortran callers hold
  configs   the other BASELINE.json shapes at this N: config 3 (4096 trans-dimensional states per
          step, k Poisson and k uniform), config 4 (64 tempering replicas x 1024 chains, sharded
          by replica over the N GPUs, one MH move of every chain per step and one swap round whose
          all-gather of (logL, beta) over NCCL is inside the timed region), a config-5 slice per GPU

--impl reference times that CPU oracle alone (rank 0 only).

--dump-outputs DIR writes what the timed device-resident path returned in its last step (logL, one
per model) as DIR/logL.npy (DIR/logL_rank<r>.npy on N > 1), float64; the inputs are seeded, so two
builds run with the same arguments can be compared value for value.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "model_source_travel_time_evals_per_s"
UNIT = "evals/s"
WORKLOAD = ("config2: batched forward sweep, 1M random 10-layer models x 64 sources per GPU, fp64, "
            "Gaussian logL fused (one logL per model)")
FP64_PEAK_THEORY_TFLOPS = 37.2     # 148 SMs x 64 DFMA/clk x 2 flop x 1.965 GHz
DUMP_BUDGET_BYTES = 64 << 20       # --dump-outputs, all ranks together


def config_dict(B, S, layers):
    """`config` of the JSON line: the same keys and strings in both arms (--impl ours / reference)."""
    return {"workload": WORKLOAD, "models_per_gpu": int(B), "sources": int(S), "layers": int(layers),
            "l2": "inputs (176 MB per step) exceed the 126 MB L2; no explicit flush"}


def kernel_sources_sha():
    """sha256 over the kernel sources: profiles/traffic.json records the one it was captured on."""
    import hashlib
    h = hashlib.sha256()
    for f in ("rt_kernels.cu", "rt_api.cu", "rt_internal.h"):
        h.update(open(os.path.join(ROOT, "raytracerfortran_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--models", type=int, default=0, help="override models per GPU (debug only)")
    ap.add_argument("--variant", type=int, default=-1, help="kernel variant (debug only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (debug only)")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (debug only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    return args


def dump_outputs(dirname, arrays, budget):
    """Write each array as dirname/<name>.npy in float64.  Over `budget` bytes in all, each array is
    cut to a fixed, seeded sample of its elements (in index order), the same from run to run."""
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.size * 8 for a in arrays.values())
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        if total > budget:
            keep = a.size * budget // total
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def workload(rank, models):
    from raytracerfortran_b200 import workloads
    cfg = dict(workloads.CONFIGS["config2"])
    if models:
        cfg["B"] = models
    v, z, nl = workloads.make_models(cfg["B"], cfg["nlayers"], cfg["seed"] + 1000 * rank)
    so, sd = workloads.make_sources(cfg["nsrc"], cfg["seed"])
    return cfg, v, z, nl, so, sd


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, False, [], set(), None
        self.recording = False      # NVML is initialised before the timed region; samples count only inside it

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            while not self.stop_flag:
                if not self.recording:
                    time.sleep(0.001)
                    continue
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        self.stop_flag = True
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None,
                "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def cpu_leg(v, z, nl, so, sd, tobs, sigma, budget_s=12.0):
    """Time the CPU oracle (all host threads, fused logL, no file I/O) on a bounded sample."""
    import oracle
    ncpu = os.cpu_count() or 1
    probe = min(len(v), 4000)
    t0 = time.perf_counter()
    oracle.dff_batch(v[:probe], z[:probe], nl[:probe], so, sd, tobs=tobs, sigma=sigma[:probe],
                     want_times=False, nthreads=ncpu)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    n = int(min(len(v), max(probe, rate * budget_s)))
    t0 = time.perf_counter()
    out = oracle.dff_batch(v[:n], z[:n], nl[:n], so, sd, tobs=tobs, sigma=sigma[:n],
                           want_times=False, nthreads=ncpu)
    dt = time.perf_counter() - t0
    # SURVEY 8(d): also one core, and the faithful call pattern (one model per call through the
    # 8-argument entry, which truncates ./rays.dat on every call, subroutineR-quiet.f90:432-433)
    n1 = int(min(n, max(500, rate / ncpu * 1.5)))
    t0 = time.perf_counter()
    oracle.dff_batch(v[:n1], z[:n1], nl[:n1], so, sd, tobs=tobs, sigma=sigma[:n1], want_times=False,
                     nthreads=1)
    dt1 = time.perf_counter() - t0
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        oracle.dff_batch_faithful(v[:n1], z[:n1], nl[:n1], so, sd, os.path.join(tmp, "rays.dat"))
        dtf = time.perf_counter() - t0
    return {"value": n * len(so) / dt, "unit": UNIT, "cores": int(out["threads"]), "kind": "port",
            "sample": f"first {n} of {len(v)} models x {len(so)} sources, fused logL, {dt:.2f} s; "
                      "C restatement of the gfortran path (gcc -O2 -ffp-contract=off, OpenMP), "
                      "no per-call rays.dat truncation",
            "single_core": {"value": n1 * len(so) / dt1, "sample": f"{n1} models, {dt1:.2f} s"},
            "faithful_single_core": {"value": n1 * len(so) / dtf,
                                     "sample": f"{n1} models, one dff call per model with the "
                                               f"per-call rays.dat truncate, {dtf:.2f} s"}}, n, dt


def run_reference(args, rank):
    if rank != 0:
        return
    cfg, v, z, nl, so, sd = workload(0, args.models)
    import oracle
    B, S = len(v), len(so)
    t_true = oracle.dff_batch(v[:1], z[:1], nl[:1], so, sd)["timeP"][0]
    from raytracerfortran_b200 import workloads
    tobs, sigma = workloads.make_observations(t_true, B, cfg["seed"])
    ncpu = os.cpu_count() or 1
    # each step = a bounded sample of the workload (~2 s of CPU work)
    probe = min(B, 4000)
    t0 = time.perf_counter()
    oracle.dff_batch(v[:probe], z[:probe], nl[:probe], so, sd, tobs=tobs, sigma=sigma[:probe],
                     want_times=False, nthreads=ncpu)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    n = int(min(B, max(probe, rate * 2.0)))
    times = []
    for i in range(args.warmup + args.steps):
        lo = (i * n) % max(B - n, 1)
        t0 = time.perf_counter()
        out = oracle.dff_batch(v[lo:lo + n], z[lo:lo + n], nl[lo:lo + n], so, sd, tobs=tobs,
                               sigma=sigma[lo:lo + n], want_times=False, nthreads=ncpu)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    value = n * S * len(times) / total
    cb = {"value": value, "unit": UNIT, "cores": int(out["threads"]), "kind": "port",
          "sample": f"{n} of {B} models x {S} sources per step, fused logL; C restatement of the "
                    "gfortran path (the reference Fortran cannot be compiled in this image)"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": config_dict(B, S, cfg["nlayers"]),
        "reference_sample": {"models_per_step": n, "note": "each step is a bounded sample of the workload"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# W_min (flops per evaluation, sqrt = div = 1) of the other shapes, counted by the instrumented
# oracle on these seeds (profiles/r01_h_other_configs.jsonl); re-counted live when the CPU leg runs.
W_MIN_FALLBACK = {"config3_poisson": 132.2, "config3_uniform_k": 580.3, "config4": 155.6, "config5_slice": 5716.1}


def _w_min_kmode(k, vp, zi, so, sd, nb):
    """W_min of trans-dimensional states: LOGLHOOD_RT's model mapping (loglhood.f90:128-146), then
    the instrumented oracle on the first nb states."""
    import oracle
    kk = k[:nb]
    nlay = np.where(kk > 1, kk - 1, 1).astype(np.int32)
    vv = vp[:nb].copy()
    zz = np.concatenate([zi[:nb], np.zeros((nb, 1))], axis=1)[:, :max(zi.shape[1], 1)].copy()
    one = kk <= 1
    vv[one, 1] = vv[one, 0]
    zz[one, 0] = 9999.9
    st = oracle.batch_stats(vv, zz, nlay, so, sd)
    return st["flops_min"] / st["rays"]


def time_steps(torch, dist, world, step, warmup, steps):
    """W warm-up steps, then K steps between CUDA events with a barrier + synchronize on both
    sides; returns ms per step, max over ranks."""
    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def other_configs(torch, dist, rt, rank, world, dev, peak_tf, count_w):
    """BASELINE.json configs 3, 4 and a config-5 slice at this N (see the module docstring)."""
    from raytracerfortran_b200 import chains, device, tempering, workloads
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = {}

    def entry(name, workload, models_total, S, ms, w_min, scaling, extra=None):
        evals = models_total * S / (ms * 1e-3)
        tf = w_min * evals / world / 1e12            # per GPU, against the per-GPU peak
        e = {"workload": workload, "scaling": scaling, "ms_per_step": ms, "evals_per_s": evals,
             "logL_per_s": models_total / (ms * 1e-3),
             "roofline": {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s per GPU",
                          "frac": tf / peak_tf if peak_tf else None, "flops_per_eval_min": w_min}}
        e.update(extra or {})
        out[name] = e

    # ---- config 3: 4096 trans-dimensional states per step and GPU, 256 sources -----------------
    c3 = workloads.CONFIGS["config3"]
    so, sd = workloads.make_sources(c3["nsrc"], c3["seed"])
    ts, td = f(so), f(sd)
    for name, uniform in (("config3_poisson", False), ("config3_uniform_k", True)):
        k, vp, zi = workloads.make_transd_models(c3["B"], c3["kmax"], c3["seed"] + (1 if uniform else 0) + 100 * rank,
                                                 uniform_k=uniform)
        tobs, sigma = workloads.make_observations(np.full(c3["nsrc"], 1.5), c3["B"], 1)
        tv, tz, tn, to, tg = f(vp), f(zi), f(k), f(tobs), f(sigma)
        ll = torch.empty(c3["B"], dtype=torch.float64, device=dev)
        step = lambda: device.dff_batch_device(tv, tz, tn, ts, td, tobs=to, sigma=tg, logL=ll, kmode=True)
        ms = time_steps(torch, dist, world, step, 5, 100)
        w = _w_min_kmode(k, vp, zi, so, sd, 234) if count_w else W_MIN_FALLBACK[name]
        entry(name, f"config3: {c3['B']} trans-dimensional states per step and GPU, k = 1..{c3['kmax']} "
                    f"({'uniform' if uniform else 'Poisson(3.01)'}), {c3['nsrc']} sources, logL fused",
              c3["B"] * world, c3["nsrc"], ms, w, "weak",
              {"tile_models": int(rt.get_stat("tile_models")), "grid": int(rt.get_stat("grid"))})

    # ---- config 4: 64 replicas x 1024 chains sharded by replica, swap all-gather in the step -----
    c4 = workloads.CONFIGS["config4"]
    R_all, C, ldk, S4 = c4["replicas"], c4["proposals"], c4["kmax"], c4["nsrc"]
    if R_all % world == 0:
        R = R_all // world
        B4 = R * C
        k, vp, zi = workloads.make_transd_models(B4, ldk, c4["seed"] + 100 * rank)
        voro = np.zeros((B4, 2, ldk))
        voro[:, 1, :] = vp
        voro[:, 0, 1:] = zi
        so, sd = workloads.make_sources(S4, c4["seed"])
        tobs, sigma = workloads.make_observations(np.full(S4, 1.3), B4, c4["seed"] + rank)
        tk, tvo, ts4, td4, to4, tg4 = f(k), f(voro), f(so), f(sd), f(tobs), f(sigma)
        ladder = tempering.temperature_ladder(R_all, 1.4)[rank * R:(rank + 1) * R]
        beta = f(np.repeat(ladder, C))
        tl = device.dff_batch_device(tvo[:, 1, :].contiguous(), tvo[:, 0, 1:].contiguous(), tk, ts4, td4,
                                     tobs=to4, sigma=tg4, kmode=True)["logL"]
        prior = chains.prior_array()
        nsteps, nwarm = 60, 6
        gen = torch.Generator(device=dev).manual_seed(400 + rank)
        total = nsteps + nwarm
        # every chain walks its own sweep (ivo, iwhich) = (1,2), (2,1), (2,2), ... (:725-731)
        period = (2 * tk - 1).to(torch.int64)
        j = torch.arange(total, device=dev, dtype=torch.int64)[:, None] % period[None, :] + 1
        ivo = (torch.div(j, 2, rounding_mode="floor") + 1).to(torch.int32).contiguous()
        iwh = (j % 2 + 1).to(torch.int32).contiguous()
        u = torch.rand((2, total, B4), dtype=torch.float64, device=dev, generator=gen)
        cauchy = chains.cauchy_deviates(u[0]).contiguous()
        uacc = u[1].contiguous()
        acc = torch.empty(B4, dtype=torch.int32, device=dev)
        sr = tempering.SwapRound(B4, dev)
        state = {"i": 0, "swap": True}

        def step4():
            i = state["i"] % total
            chains.mh_step_device(tk, tvo, tl, ivo[i], iwh[i], cauchy[i], uacc[i], beta, tg4, prior,
                                  ts4, td4, to4, accept=acc,
                                  beta_ready=sr.done if (state["swap"] and state["i"] > 0) else None)
            if state["swap"]:
                sr.launch(tl, beta, 2026, state["i"])
            state["i"] += 1

        ms_swap = time_steps(torch, dist, world, step4, nwarm, nsteps)
        sr.wait()
        torch.cuda.synchronize()
        state.update(i=0, swap=False)
        ms_noswap = time_steps(torch, dist, world, step4, nwarm, nsteps)
        w = _w_min_kmode(k, vp, zi, so, sd, 234) if count_w else W_MIN_FALLBACK["config4"]
        entry("config4", f"config4: {R_all} tempering replicas x {C} chains sharded by replica over {world} GPU(s), "
                         f"k ~ Poisson(3.01) in 1..{ldk}, {S4} sources; per step one MH move of every chain "
                         "(propose, likelihood, accept) and one swap round (pack, NCCL all-gather of "
                         "(logL, beta), swap kernel) on a side stream under the next step's proposal "
                         "and likelihood kernels",
              R_all * C, S4, ms_swap, w, "strong",
              {"mh_moves_per_s": R_all * C / (ms_swap * 1e-3), "ms_per_step_without_swap": ms_noswap,
               "swap_exposed_ms_per_round": max(0.0, ms_swap - ms_noswap),
               "swap_allgather_bytes_per_rank": 16 * B4, "collective": "nccl all_gather" if world > 1 else "none (1 GPU)",
               "chains_per_gpu": B4, "kernel_launches_per_step": 5})

    # ---- config 5 slice: 16384 models x 50 interfaces x 1024 near-critical sources per GPU -------
    c5 = workloads.CONFIGS["config5"]
    nb5 = 16384
    v5, z5, n5 = workloads.make_models(nb5, c5["nlayers"], c5["seed"] + 100 * rank, min_thickness=False)
    so5, sd5 = workloads.make_sources(c5["nsrc"], c5["seed"], near_critical=True)
    tobs5, sigma5 = workloads.make_observations(np.full(c5["nsrc"], 1.5), nb5, 1)
    tv, tz, tn, ts5, td5, to5, tg5 = f(v5), f(z5), f(n5), f(so5), f(sd5), f(tobs5), f(sigma5)
    ll5 = torch.empty(nb5, dtype=torch.float64, device=dev)
    step5 = lambda: device.dff_batch_device(tv, tz, tn, ts5, td5, tobs=to5, sigma=tg5, logL=ll5)
    ms = time_steps(torch, dist, world, step5, 2, 4)
    if count_w:
        import oracle
        st = oracle.batch_stats(v5[:58], z5[:58], n5[:58], so5, sd5)
        w = st["flops_min"] / st["rays"]
    else:
        w = W_MIN_FALLBACK["config5_slice"]
    finite = int(torch.isfinite(ll5).sum().item())
    entry("config5_slice", f"config5 slice: {nb5} of 16M models per GPU x {c5['nlayers']} interfaces x "
                           f"{c5['nsrc']} near-critical sources, logL fused",
          nb5 * world, c5["nsrc"], ms, w, "weak",
          {"logL_note": f"{finite} of {nb5} logL finite: with N = {c5['nsrc']} >= 772 sources the reference's "
                        "(2 pi)^(N/2) overflows (loglhood.f90:194) and every logL is -inf, reproduced here; "
                        "evals/s is the meaningful figure for this shape",
           "kernel_variant": int(rt.get_stat("variant"))})
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import raytracerfortran_b200 as rt
    from raytracerfortran_b200 import device, workloads

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    os.environ["RTB200_DEVICE"] = str(local)
    if args.variant >= 0:
        rt.set_option("variant", args.variant)
    for kv in args.opt:
        name, val = kv.split("=")
        rt.set_option(name, float(val))

    cfg, v, z, nl, so, sd = workload(rank, args.models)
    B, S = len(v), len(so)
    t_true = rt.dff_batch(v[:2], z[:2], nl[:2], so, sd)["timeP"][0]
    tobs, sigma = workloads.make_observations(t_true, B, cfg["seed"])

    # ---- device-resident inputs --------------------------------------------------------------
    f = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    tv, tz, tn, ts, td, to, tg = f(v), f(z), f(nl), f(so), f(sd), f(tobs), f(sigma)
    logL = torch.empty(B, dtype=torch.float64, device=dev)

    def step_resident():
        device.dff_batch_device(tv, tz, tn, ts, td, tobs=to, sigma=tg, logL=logL)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peak_tf = rt.fp64_peak_tflops(3)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler.recording = True
    launches0 = rt.get_stat("launches")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = int(rt.get_stat("launches") - launches0)
    sampler.recording = False
    logL_resident = logL.cpu().numpy().copy()
    # geometry of the timed (device-resident) launch, read before any other call changes it
    kernel_info = {k_: int(rt.get_stat(k_)) for k_ in ("variant", "tile_models", "tile_sources", "threads",
                                                       "grid", "smem_bytes", "ctas_per_sm")}

    # ---- end to end through the C ABI with pinned host buffers -------------------------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    hv, hz, hn, hg = pin(v), pin(z), pin(nl), pin(sigma)
    h_ll = torch.empty(B, dtype=torch.float64).pin_memory().numpy()

    def step_e2e():
        rt.dff_batch(hv, hz, hn, so, sd, tobs=tobs, sigma=hg, want_times=False, out_logL=h_ll)

    for _ in range(args.warmup):
        step_e2e()
    barrier()
    sampler.recording = True            # the end-to-end timed region is sampled as well
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.summary()
    e2e_gpu_span_ms = rt.get_stat("total_ms")        # first H2D to last D2H of the last call
    assert np.array_equal(h_ll.view(np.uint64), logL_resident.view(np.uint64)), \
        "host-buffer and device-resident paths disagree"
    h2d = hv.nbytes + hz.nbytes + hn.nbytes + hg.nbytes + so.nbytes + sd.nbytes + tobs.nbytes
    d2h = h_ll.nbytes

    # ---- the same call from pageable memory (what R vectors and Fortran arrays are) --------------
    p_ll = np.empty(B, dtype=np.float64)

    def step_pageable():
        rt.dff_batch(v, z, nl, so, sd, tobs=tobs, sigma=sigma, want_times=False, out_logL=p_ll)

    for _ in range(args.warmup):
        step_pageable()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_pageable()
    torch.cuda.synchronize()
    pageable_s = time.perf_counter() - t0
    assert np.array_equal(p_ll.view(np.uint64), logL_resident.view(np.uint64)), \
        "pageable-buffer and device-resident paths disagree"

    tt = torch.tensor([ms, e2e_s * 1e3, pageable_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max, pageable_ms_max = tt.tolist()

    count_w = world == 1 and not args.no_cpu
    configs = None
    if not args.models:
        try:
            configs = other_configs(torch, dist, rt, rank, world, dev, peak_tf, count_w and rank == 0)
        except Exception as e:       # the headline line must survive a failure in the extra shapes
            import traceback
            traceback.print_exc()
            configs = {"error": f"{type(e).__name__}: {e}"}

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logL" if world == 1 else f"logL_rank{rank}": logL_resident},
                     DUMP_BUDGET_BYTES // world)

    if rank == 0:
        evals_step = float(B) * S * world
        value = evals_step * args.steps / (ms_max * 1e-3)
        e2e_value = evals_step * args.steps / (e2e_ms_max * 1e-3)
        # ---- work per evaluation + CPU baseline, on a bounded sample (rank 0, N = 1 only) ----
        cpu = None
        w_min = w_ref = None
        if count_w:
            import oracle
            st = oracle.batch_stats(v[:2000], z[:2000], nl[:2000], so, sd)
            w_min, w_ref = st["flops_min"] / st["rays"], st["flops_ref"] / st["rays"]
            cpu, n_cpu, _ = cpu_leg(v, z, nl, so, sd, tobs, sigma)
            ref_ll = oracle.dff_batch(v[:n_cpu][:2000], z[:2000], nl[:2000], so, sd, tobs=tobs,
                                      sigma=sigma[:2000], want_times=False)["logL"]
            assert np.allclose(ref_ll, logL_resident[:2000], rtol=1e-12, atol=0), "parity lost"
        if w_min is None:
            w_min = 396.12   # config-2 inputs, counted by oracle.batch_stats (DESIGN.md)
        kernel_s = ms_max * 1e-3 / args.steps
        achieved_tf = w_min * float(B) * S / kernel_s / 1e12
        alg_bytes = float(B) * ((cfg["nlayers"] + 1 + cfg["nlayers"]) * 8 + 4 + 8 + 8)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # DRAM traffic and FP64-pipe activity come from one ncu --set full capture (profiles/);
        # they are quoted only while the kernel sources are the ones that capture was taken on
        traffic = ncu = None
        ncu_note = "profiles/traffic.json missing"
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if ncu.get("kernel_sources_sha") == kernel_sources_sha():
                traffic = ncu.get("dram_bytes_per_launch")
                ncu_note = None
            else:
                ncu_note = ("STALE: profiles/traffic.json was captured on other kernel sources "
                            f"({ncu.get('kernel_sources_sha')} != {kernel_sources_sha()}); not quoted")
                print("bench.py: " + ncu_note, file=sys.stderr)
                ncu = None
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(B, S, cfg["nlayers"]),
            "kernel": {"kernel_variant": kernel_info["variant"], "tile_models": kernel_info["tile_models"],
                       "tile_sources": kernel_info["tile_sources"], "threads": kernel_info["threads"],
                       "grid": kernel_info["grid"], "smem_bytes": kernel_info["smem_bytes"],
                       "ctas_per_sm": kernel_info["ctas_per_sm"],
                       "note": "geometry of the timed device-resident launch"},
            "logL_per_s": float(B) * world * args.steps / (ms_max * 1e-3),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms_max / args.steps,
                    "gpu_span_ms_last_step": e2e_gpu_span_ms,
                    "api": "dff_batch (C ABI, pinned host buffers, logL only)",
                    "pageable": {"value": evals_step * args.steps / (pageable_ms_max * 1e-3), "unit": UNIT,
                                 "ms_per_step": pageable_ms_max / args.steps,
                                 "frac_of_pinned": e2e_ms_max / pageable_ms_max,
                                 "api": "dff_batch (C ABI, ordinary pageable numpy arrays, logL only)"}},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {
                "bound": "fp64", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved_tf / peak_tf if peak_tf else None, "traffic": traffic,
                "peak_source": "measured live: DFMA microbenchmark in libraytrace_b200 "
                               "(MEASURED_PEAKS.json has no FP64 entry)",
                "peak_theoretical": FP64_PEAK_THEORY_TFLOPS,
                "frac_of_theoretical": achieved_tf / FP64_PEAK_THEORY_TFLOPS,
                "flops_per_eval_min": w_min, "flops_per_eval_reference": w_ref,
                "fp64_pipe_active_pct_ncu": (ncu or {}).get("fp64_pipe_active_pct"),
                "ncu_source": (ncu or {}).get("source"), "ncu_commit": (ncu or {}).get("commit"),
                "ncu_date": (ncu or {}).get("date"), "ncu_note": ncu_note,
                "note": "sqrt = div = 1 flop; a correctly rounded fp64 div/sqrt costs ~10 FP64-pipe "
                        "instructions, so pipe utilisation (ncu, profiles/) is several times this fraction",
                # the same kernel against the HBM roofline, in the contract's own keys: the path
                # streams 188 MB per launch and sits at a fraction of a percent of the copy bandwidth
                "hbm": {"bound": "hbm", "achieved": alg_bytes / kernel_s / 1e9, "peak": peaks.get("hbm_gbs"),
                        "unit": "GB/s",
                        "frac": (alg_bytes / kernel_s / 1e9 / peaks["hbm_gbs"]) if peaks.get("hbm_gbs") else None,
                        "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks.get("hbm_gbs") else None},
            },
            "cpu_baseline": cpu,
            "configs": configs,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
