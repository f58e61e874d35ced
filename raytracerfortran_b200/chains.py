"""Fixed-dimension Metropolis-Hastings moves of many independent chains on the GPU (SURVEY 8f rows
N1 + N2): the body of EXPLORE_MH_NOVARPAR's sweep (prjmh_temper_rf.f90:717-757) -- PROPOSAL
(:1386-1447), INTERPLAYER_novar (loglhood.f90:214-295), CHECKBOUNDS2 (:1681-1716), LOGLHOOD and the
accept test -- for B chains per launch through rtb200_mh_step_device (include/raytrace_b200.h).

The reference runs one chain per MPI rank and one proposal at a time; batching ACROSS chains leaves
every chain's Markov kernel unchanged.  Chain states live in HBM between moves: k [B] int32,
voro [B, 2, ldk] float64 (row 0 node depths, row 1 vp, sorted by depth), logL [B], beta [B],
sigma [B].  torch supplies the tensors, the stream and the random numbers; the move itself is the
library's kernels.  The birth/death move (BIRTH_FULL /
DEATH_FULL, :658-710) is `bd_step_device`, the data-error move of EXPLORE_MH (:545-575) `sd_step_device`, its AR(1) move (:583-631) `ar_step_device`.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .device import _ensure_device, _ptr, _stream_handle


def _move_prologue(name, voro, stream=None, accept=False):
    """The start every chain-move wrapper shares: voro [B, 2, ldk] a CUDA tensor, the library
    initialised on its device, and the C ABI's handle of `stream` (default: torch's current stream).
    `accept` is the caller's [B] i32 output of a single move, None to allocate one; the wrappers that
    have no such output leave it False.  Returns (dev, B, ldk, stream handle, accept)."""
    if not voro.is_cuda:
        raise ValueError(f"{name} needs CUDA tensors (there is no CPU path)")
    dev = voro.device
    _ensure_device(dev.index if dev.index is not None else torch.cuda.current_device())
    B, two, ldk = voro.shape
    if two != 2:
        raise ValueError("voro must be [B, 2, ldk]")
    if accept is None:
        accept = torch.empty((B,), dtype=torch.int32, device=dev)
    return dev, B, ldk, _stream_handle(stream, dev), accept


def _host_doubles(a, n, message):
    """A host array of exactly n doubles, contiguous for the C ABI."""
    arr = np.ascontiguousarray(a, dtype=np.float64)
    if arr.size != n:
        raise ValueError(message)
    return arr


_PRIOR_SIZE = "prior must hold 7 doubles (see prior_array)"
_AR_PRIOR_SIZE = "ar_prior must hold 4 doubles (see ar_prior_array)"


def prior_array(hmin=100.1, hmx=10000.1, vmin=1500.0, vmax=10000.0, pertsdsc=30.0, fact=1.0,
                factor=1.0):
    """The 7 doubles rtb200_mh_step_device takes as `prior`, from the parameter file's hmin / hmx
    the way read_input.f90:207-214 derives them: minlim = (hmin, 1500), maxlim = (hmx, 10000),
    pertsd = (maxlim - minlim)/pertsdsc (pertsdsc = 30, :169), step width fact/factor*pertsd
    (fact = 1, rjmcmc_com.f90:80; factor = 1 in EXPLORE_MH_NOVARPAR's call, :735)."""
    minlim = np.array([hmin, vmin], dtype=np.float64)
    maxlim = np.array([hmx, vmax], dtype=np.float64)
    pertsd = (maxlim - minlim) / np.float64(pertsdsc)
    scale = np.float64(fact) / np.float64(factor) * pertsd
    return np.array([scale[0], scale[1], minlim[0], minlim[1], maxlim[0], maxlim[1], hmin],
                    dtype=np.float64)


def cauchy_deviates(u):
    """TAN(PI2*(ran_uni - 0.5)) of PROPOSAL (:1405; PI2 is pi, data_type.f90:5) for uniforms u."""
    return torch.tan(math.pi * (u - 0.5))


def move_deviates(u, iwhich, enos=False):
    """The deviate PROPOSAL turns a uniform into: TAN(PI2*(ran_uni - 0.5)) (:1405, :1416), except
    for a depth move (iwhich == 1) under ENOS = 1, which uses ran_uni itself (:1428)."""
    c = cauchy_deviates(u)
    return torch.where(iwhich == 1, u, c) if enos else c


def mh_step_device(k, voro, logL, ivo, iwhich, cauchy, u_acc, beta, sigma, prior,
                   src_offset, src_depth, tobs, accept=None, stream=None, beta_ready=None, enos=False):
    """One move of every chain, in place on `voro` and `logL`.

    k [B] i32, voro [B, 2, ldk] f64, logL/beta/sigma/cauchy/u_acc [B] f64, ivo/iwhich [B] i32
    (1-based node, 1 = depth / 2 = vp), src_offset/src_depth/tobs [NSrc] f64: CUDA tensors.
    prior: 7 doubles on the host (prior_array).  Asynchronous on `stream` (default: torch's
    current stream).  `beta_ready` (a torch.cuda.Event, e.g. SwapRound.done) orders only the
    accept test behind it, so a swap round still running on another stream overlaps with the
    proposal and likelihood kernels.  `enos` selects the parameter file's ENOS = 1 (even-numbered
    order statistics prior, PROPOSAL :1418-1431): a depth move then takes the uniform itself in
    `cauchy` (see `move_deviates`).  Returns accept [B] i32: 1 accepted, 0 rejected, -1 outside
    the bounds."""
    _, B, ldk, st, accept = _move_prologue("mh_step_device", voro, stream, accept)
    pr = _host_doubles(prior, 7, _PRIOR_SIZE)
    f64, i32 = torch.float64, torch.int32
    rc = _lib.load().rtb200_mh_step_device_ev(
        _ptr(k, i32), _ptr(voro, f64), _ptr(logL, f64), B, ldk, _ptr(ivo, i32), _ptr(iwhich, i32),
        _ptr(cauchy, f64), _ptr(u_acc, f64), _ptr(beta, f64), _ptr(sigma, f64),
        pr.ctypes.data_as(C.POINTER(C.c_double)), _ptr(src_offset, f64), _ptr(src_depth, f64),
        _ptr(tobs, f64), src_offset.numel(), _ptr(accept, i32), st,
        beta_ready.cuda_event if beta_ready is not None else None, 1 if enos else 0)
    _lib.check(rc)
    return accept


def poisson_pk(lam, kmin, kmax):
    """pk(ik) = EXP(-lambda)*lambda**ik/EXP(LOGFACTORIAL(ik)) for ik = kmin..kmax
    (read_input.f90:78-81); returns an array of kmax doubles with pk[i-1] = pk(i)."""
    pk = np.zeros(kmax, dtype=np.float64)
    for ik in range(kmin, kmax + 1):
        pk[ik - 1] = math.exp(-lam) * lam ** float(ik) / math.exp(math.lgamma(ik + 1.0))
    return pk


def bd_step_device(k, voro, logL, u_k, idel, u_z, u_v, u_acc, beta, sigma, prior, pk, kmin, kmax,
                   src_offset, src_depth, tobs, accept=None, stream=None, enos=False):
    """The birth/death move of every chain (rtb200_bd_step_device), in place on k, voro, logL.
    u_k/u_z/u_v/u_acc [B] f64 uniforms, idel [B] i32 (node a death removes, 2..k), pk: host array
    (poisson_pk) or None.  Returns accept [B] i32: 1 / 0 / -1 outside / 2 no move proposed."""
    _, B, ldk, st, accept = _move_prologue("bd_step_device", voro, stream, accept)
    pr = _host_doubles(prior, 7, _PRIOR_SIZE)
    f64, i32 = torch.float64, torch.int32
    dp = C.POINTER(C.c_double)
    pkp = None
    if pk is not None:
        pka = np.ascontiguousarray(pk, dtype=np.float64)
        if pka.size < kmax:
            raise ValueError("pk must hold kmax values")
        pkp = pka.ctypes.data_as(dp)
    rc = _lib.load().rtb200_bd_step_device_ex(
        _ptr(k, i32), _ptr(voro, f64), _ptr(logL, f64), B, ldk, _ptr(u_k, f64), _ptr(idel, i32),
        _ptr(u_z, f64), _ptr(u_v, f64), _ptr(u_acc, f64), _ptr(beta, f64), _ptr(sigma, f64),
        pr.ctypes.data_as(dp), pkp, int(kmin), int(kmax), _ptr(src_offset, f64),
        _ptr(src_depth, f64), _ptr(tobs, f64), src_offset.numel(), _ptr(accept, i32), st, 1 if enos else 0)
    _lib.check(rc)
    return accept


def sd_prior_array(sdmn=0.001, sdmx=0.07, pertsdsdsc=10.0):
    """pertsdsdRT, minlimsdRT, maxlimsdRT from the parameter file's sdmn / sdmx
    (read_input.f90:237-241: pertsdsdRT = (sdmx - sdmn)/10)."""
    return np.array([(np.float64(sdmx) - np.float64(sdmn)) / np.float64(pertsdsdsc), sdmn, sdmx],
                    dtype=np.float64)


def sd_step_device(k, voro, logL, sigma, u_gate, gauss, u_acc, beta, sd_prior, src_offset, src_depth,
                   tobs, accept=None, stream=None):
    """The data-error move of every chain (rtb200_sd_step_device), in place on sigma and logL.
    Returns accept [B] i32: 1 / 0 / -1 outside / 2 no move proposed."""
    _, B, ldk, st, accept = _move_prologue("sd_step_device", voro, stream, accept)
    sp = _host_doubles(sd_prior, 3, "sd_prior must hold 3 doubles (see sd_prior_array)")
    f64, i32 = torch.float64, torch.int32
    rc = _lib.load().rtb200_sd_step_device(
        _ptr(k, i32), _ptr(voro, f64), _ptr(logL, f64), _ptr(sigma, f64), B, ldk, _ptr(u_gate, f64),
        _ptr(gauss, f64), _ptr(u_acc, f64), _ptr(beta, f64), sp.ctypes.data_as(C.POINTER(C.c_double)),
        _ptr(src_offset, f64), _ptr(src_depth, f64), _ptr(tobs, f64), src_offset.numel(), _ptr(accept, i32), st)
    _lib.check(rc)
    return accept


def set_chain_ar(idxar=None, arpar=None, armx=0.5):
    """IAR = 1: every likelihood evaluation of the move functions uses the chains' AR(1) state
    (idxar [B] i32, arpar [B] f64 CUDA tensors, kept by reference: ar_step_device updates them in
    place).  Call without arguments to return to IAR = 0 (rtb200_set_chain_ar)."""
    if idxar is None:
        _lib.check(_lib.load().rtb200_set_chain_ar(None, None, float(armx)))
        return
    _lib.check(_lib.load().rtb200_set_chain_ar(_ptr(idxar, torch.int32), _ptr(arpar, torch.float64), float(armx)))


def ar_prior_array(minlimar=-0.5, maxlimar=0.9, pertarsdsc=10.0, armx=0.5):
    """pertarsdRT, minlimarRT, maxlimarRT, armxRT: read_input.f90:223-227 (pertarsdRT =
    (maxlimarRT - minlimarRT)/10) and rjmcmc_com.f90:93 (armxRT = 0.5)."""
    lo, hi = np.float64(minlimar), np.float64(maxlimar)
    return np.array([(hi - lo) / np.float64(pertarsdsc), lo, hi, armx], dtype=np.float64)


def ar_step_device(k, voro, logL, sigma, idxar, arpar, u_choice, u_prop, gauss, u_acc, beta, ar_prior,
                   src_offset, src_depth, tobs, accept=None, stream=None):
    """The AR(1) move of every chain (rtb200_ar_step_device, IAR = 1), in place on idxar [B] i32,
    arpar [B] f64 and logL.  Returns accept [B] i32: 1 / 0 / -1 outside."""
    _, B, ldk, st, accept = _move_prologue("ar_step_device", voro, stream, accept)
    ap = _host_doubles(ar_prior, 4, _AR_PRIOR_SIZE)
    f64, i32 = torch.float64, torch.int32
    rc = _lib.load().rtb200_ar_step_device(
        _ptr(k, i32), _ptr(voro, f64), _ptr(logL, f64), _ptr(sigma, f64), _ptr(idxar, i32),
        _ptr(arpar, f64), B, ldk, _ptr(u_choice, f64), _ptr(u_prop, f64), _ptr(gauss, f64),
        _ptr(u_acc, f64), _ptr(beta, f64), ap.ctypes.data_as(C.POINTER(C.c_double)),
        _ptr(src_offset, f64), _ptr(src_depth, f64), _ptr(tobs, f64), src_offset.numel(), _ptr(accept, i32), st)
    _lib.check(rc)
    return accept


def mh_sweep_device(k, voro, logL, beta, sigma, prior, src_offset, src_depth, tobs, generator=None,
                    stats=None):
    """EXPLORE_MH_NOVARPAR's sweep (:725-760) for every chain: for ivo = 1..max(k) and
    iwhich = 1, 2 (skipping the fixed top node's depth, :730) propose, check, evaluate, accept.
    Chains with fewer than ivo nodes sit the move out.  Uniforms come from `generator` (a CUDA
    torch.Generator).  Returns (accepted, proposed) counts as device tensors [B]."""
    dev = voro.device
    B = voro.shape[0]
    kmax = int(k.max().item())
    acc_n = torch.zeros(B, dtype=torch.int64, device=dev)
    prop_n = torch.zeros(B, dtype=torch.int64, device=dev)
    accept = torch.empty(B, dtype=torch.int32, device=dev)
    for ivo in range(1, kmax + 1):
        iv = torch.full((B,), ivo, dtype=torch.int32, device=dev)
        for iwhich in (1, 2):
            if ivo == 1 and iwhich == 1:
                continue
            iw = torch.full((B,), iwhich, dtype=torch.int32, device=dev)
            u = torch.rand((2, B), dtype=torch.float64, device=dev, generator=generator)
            mh_step_device(k, voro, logL, iv, iw, cauchy_deviates(u[0]), u[1].contiguous(), beta,
                           sigma, prior, src_offset, src_depth, tobs, accept=accept)
            prop_n += (k >= ivo)
            acc_n += (accept == 1)
    return acc_n, prop_n


_moves_buffers = {}


def mh_moves_device(k, voro, logL, pos, n_moves, beta, sigma, prior, src_offset, src_depth, tobs,
                    generator=None, enos=False):
    """n_moves moves in which EVERY chain makes its next move: chain b walks its own sweep
    (ivo, iwhich) = (1,2), (2,1), (2,2), ..., (k_b,1), (k_b,2) -- EXPLORE_MH_NOVARPAR's order,
    :725-731 -- and wraps around after its 2 k_b - 1 moves, so short chains do not idle while long
    ones finish a lock-step sweep.  `pos` [B] i32 holds each chain's position in its sweep and is
    advanced in place.  The schedule and all random numbers are generated up front into buffers
    that persist between calls, and the run of moves goes to rtb200_mh_moves_device, which replays
    it as one CUDA graph.  Returns the number of accepted moves per chain [B]."""
    dev, B, ldk, st, _ = _move_prologue("mh_moves_device", voro)
    pr = _host_doubles(prior, 7, _PRIOR_SIZE)
    f64, i32 = torch.float64, torch.int32
    key = (dev, B, int(n_moves))
    buf = _moves_buffers.get(key)
    if buf is None:
        buf = {"ivo": torch.empty((n_moves, B), dtype=i32, device=dev),
               "iwhich": torch.empty((n_moves, B), dtype=i32, device=dev),
               "u": torch.empty((2, n_moves, B), dtype=f64, device=dev),
               "cauchy": torch.empty((n_moves, B), dtype=f64, device=dev),
               "accept": torch.empty((n_moves, B), dtype=i32, device=dev)}
        _moves_buffers.clear()                      # one shape at a time: the library caches one graph
        _moves_buffers[key] = buf
    period = (2 * k - 1).to(torch.int64)
    t = torch.arange(n_moves, device=dev, dtype=torch.int64)[:, None]
    j = (pos.to(torch.int64)[None, :] + t) % period[None, :] + 1
    buf["ivo"].copy_(torch.div(j, 2, rounding_mode="floor") + 1)
    buf["iwhich"].copy_(j % 2 + 1)
    buf["u"].uniform_(generator=generator)
    torch.tan(math.pi * (buf["u"][0] - 0.5), out=buf["cauchy"])
    if enos:
        buf["cauchy"].copy_(torch.where(buf["iwhich"] == 1, buf["u"][0], buf["cauchy"]))
    rc = _lib.load().rtb200_mh_moves_device_ex(
        _ptr(k, i32), _ptr(voro, f64), _ptr(logL, f64), B, ldk, int(n_moves), _ptr(buf["ivo"], i32),
        _ptr(buf["iwhich"], i32), _ptr(buf["cauchy"], f64), _ptr(buf["u"][1], f64), _ptr(beta, f64),
        _ptr(sigma, f64), pr.ctypes.data_as(C.POINTER(C.c_double)), _ptr(src_offset, f64),
        _ptr(src_depth, f64), _ptr(tobs, f64), src_offset.numel(), _ptr(buf["accept"], i32), st,
        1 if enos else 0)
    _lib.check(rc)
    pos.copy_(((pos.to(torch.int64) + n_moves) % period).to(i32))
    return (buf["accept"] == 1).sum(dim=0)


def mcmc_step_device(k, voro, logL, sigma, beta, prior, sd_prior, pk, kmin, kmax, src_offset,
                     src_depth, tobs, generator=None, ar=None):
    """One iteration of the sampler's worker loop (prjmh_temper_rf.f90:421-447) for every chain:
    EXPLORE_MH_NOVARPAR -- the birth/death move, then the sweep over ivo = 1..k, iwhich = 1, 2 --
    followed by EXPLORE_MH's data-error move.  All chains step together; a chain with fewer than
    ivo nodes sits that move out, exactly as its own loop would have ended.  Everything stays on
    the device; random numbers come from `generator`.  With `ar = (idxar, arpar, ar_prior)` the
    sampler's IAR = 1 mode is run: every move evaluates the AR(1) likelihood of the chain's state and
    EXPLORE_MH's AR move follows the data-error move (:583-631).  Returns a dict of per-chain
    counts (device tensors): accepted / proposed fixed-k moves, birth/death, sigma and AR outcomes."""
    if ar is not None:
        set_chain_ar(ar[0], ar[1], float(np.asarray(ar[2], dtype=np.float64)[3]))
    try:
        return _mcmc_step(k, voro, logL, sigma, beta, prior, sd_prior, pk, kmin, kmax, src_offset, src_depth,
                          tobs, generator, ar)
    finally:
        if ar is not None:      # always unregister, without letting a stale error mask the real one
            _lib.load().rtb200_set_chain_ar(None, None, 0.5)


def _mcmc_step(k, voro, logL, sigma, beta, prior, sd_prior, pk, kmin, kmax, src_offset, src_depth, tobs,
               generator, ar):
    dev = voro.device
    B, _, ldk = voro.shape
    f64 = torch.float64
    u = torch.rand((5, B), dtype=f64, device=dev, generator=generator)
    idel = (2 + torch.floor(u[4] * (k - 1).clamp(min=1))).to(torch.int32)
    bd = bd_step_device(k, voro, logL, u[0].contiguous(), idel, u[1].contiguous(), u[2].contiguous(),
                        u[3].contiguous(), beta, sigma, prior, pk, kmin, kmax, src_offset, src_depth,
                        tobs)
    kmax_now = int(k.max().item())
    n_moves = 2 * kmax_now - 1
    uu = torch.rand((2, max(n_moves, 1), B), dtype=f64, device=dev, generator=generator)
    cauchy, u_acc = cauchy_deviates(uu[0]).contiguous(), uu[1].contiguous()
    accept = torch.empty((max(n_moves, 1), B), dtype=torch.int32, device=dev)
    m = 0
    for ivo in range(1, kmax_now + 1):
        iv = torch.full((B,), ivo, dtype=torch.int32, device=dev)
        for iwhich in (1, 2):
            if ivo == 1 and iwhich == 1:
                continue
            iw = torch.full((B,), iwhich, dtype=torch.int32, device=dev)
            mh_step_device(k, voro, logL, iv, iw, cauchy[m], u_acc[m], beta, sigma, prior, src_offset,
                           src_depth, tobs, accept=accept[m])
            m += 1
    us = torch.rand((2, B), dtype=f64, device=dev, generator=generator)
    gauss = torch.randn(B, dtype=f64, device=dev, generator=generator)
    sd = sd_step_device(k, voro, logL, sigma, us[0].contiguous(), gauss, us[1].contiguous(), beta,
                        sd_prior, src_offset, src_depth, tobs)
    out = {"accepted": (accept[:m] == 1).sum(dim=0), "proposed": 2 * k.to(torch.int64) - 1,
           "bd": bd, "sd": sd}
    if ar is not None:
        ua = torch.rand((3, B), dtype=f64, device=dev, generator=generator)
        ga = torch.randn(B, dtype=f64, device=dev, generator=generator)
        out["ar"] = ar_step_device(k, voro, logL, sigma, ar[0], ar[1], ua[0].contiguous(), ua[1].contiguous(), ga,
                                   ua[2].contiguous(), beta, ar[2], src_offset, src_depth, tobs)
    return out


def mcmc_workspace_views(workspace, B, n_moves):
    """Named views into the workspace of rtb200_mcmc_iterations_device (a uint8 CUDA tensor of
    rtb200_mcmc_workspace_bytes(B, n_moves) bytes; layout: McmcWs, csrc/rt_internal.h): the
    iteration's deviates (u_k, u_z, u_v, u_acc_bd, u_gate, gauss, u_acc_sd, u_choice, u_prop_ar,
    gauss_ar, u_acc_ar [B]; dev, u_acc [M, B]; idel [B]; ivo, iwhich [M, B]) and outcomes (acc_bd,
    acc_sd, acc_ar [B]; acc_mh [M, B])."""
    M = int(n_moves)
    nd = (11 + 2 * M) * B
    d = workspace[:nd * 8].view(torch.float64)
    i = workspace[nd * 8:nd * 8 + (4 + 3 * M) * B * 4].view(torch.int32)
    names_d = ["u_k", "u_z", "u_v", "u_acc_bd", "u_gate", "gauss", "u_acc_sd", "u_choice", "u_prop_ar",
               "gauss_ar", "u_acc_ar"]
    out = {n: d[j * B:(j + 1) * B] for j, n in enumerate(names_d)}
    out["dev"] = d[11 * B:(11 + M) * B].view(M, B)
    out["u_acc"] = d[(11 + M) * B:(11 + 2 * M) * B].view(M, B)
    out["idel"], out["acc_bd"], out["acc_sd"], out["acc_ar"] = i[:B], i[B:2 * B], i[2 * B:3 * B], i[3 * B:4 * B]
    out["ivo"] = i[4 * B:(4 + M) * B].view(M, B)
    out["iwhich"] = i[(4 + M) * B:(4 + 2 * M) * B].view(M, B)
    out["acc_mh"] = i[(4 + 2 * M) * B:(4 + 3 * M) * B].view(M, B)
    return out


class McmcGraph:
    """The sampler's worker loop (prjmh_temper_rf.f90:420-458) for B chains as one CUDA graph per
    iteration, random numbers included (rtb200_mcmc_iterations_device): birth/death move, `n_moves`
    fixed-dimension moves of every chain's own sweep, data-error move, and with `ar` the AR(1) move.  Owns the sweep positions,
    the device iteration counter, the workspace and the tallies; `run(n)` replays the graph n
    times without touching the host again."""

    def __init__(self, k, voro, logL, sigma, beta, n_moves, prior, sd_prior, pk, kmin, kmax,
                 src_offset, src_depth, tobs, seed=1, enos=False, counter0=0, ar=None):
        dev, self.B, self.ldk, _, _ = _move_prologue("McmcGraph", voro)
        self.k, self.voro, self.logL, self.sigma, self.beta = k, voro, logL, sigma, beta
        self.src = (src_offset, src_depth, tobs)
        self.M = int(n_moves)
        both = "prior must hold 7 doubles and sd_prior 3 (prior_array, sd_prior_array)"
        self.prior, self.sd_prior = _host_doubles(prior, 7, both), _host_doubles(sd_prior, 3, both)
        self.pk = None if pk is None else np.ascontiguousarray(pk, dtype=np.float64)
        if self.pk is not None and self.pk.size < kmax:
            raise ValueError("pk must hold kmax values")
        self.kmin, self.kmax, self.seed, self.enos = int(kmin), int(kmax), int(seed), bool(enos)
        self.pos = torch.zeros(self.B, dtype=torch.int32, device=dev)
        self.counter = torch.tensor([int(counter0)], dtype=torch.int64, device=dev)
        nbytes = _lib.load().rtb200_mcmc_workspace_bytes(self.B, self.M)
        self.workspace = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        self.tally = torch.zeros((5, self.B), dtype=torch.int64, device=dev)
        # IAR = 1: ar = (idxar [B] i32, arpar [B] f64, ar_prior (ar_prior_array)); the iteration then
        # ends with the AR(1) move and every likelihood uses the chains' AR state
        self.ar = None if ar is None else (ar[0], ar[1], _host_doubles(ar[2], 4, _AR_PRIOR_SIZE))
        self.views = mcmc_workspace_views(self.workspace, self.B, self.M)

    def run(self, n_iterations=1, stream=None):
        f64, i32 = torch.float64, torch.int32
        dp = C.POINTER(C.c_double)
        so, sd, ob = self.src
        rc = _lib.load().rtb200_mcmc_iterations_device(
            _ptr(self.k, i32), _ptr(self.voro, f64), _ptr(self.logL, f64), _ptr(self.sigma, f64),
            _ptr(self.beta, f64), _ptr(self.pos, i32), self.B, self.ldk, self.M,
            self.prior.ctypes.data_as(dp), self.sd_prior.ctypes.data_as(dp),
            None if self.pk is None else self.pk.ctypes.data_as(dp), self.kmin, self.kmax,
            1 if self.enos else 0, _ptr(so, f64), _ptr(sd, f64), _ptr(ob, f64), so.numel(),
            self.seed & 0xFFFFFFFFFFFFFFFF, self.counter.data_ptr(), self.workspace.data_ptr(),
            self.tally.data_ptr(), int(n_iterations),
            None if self.ar is None else _ptr(self.ar[0], i32),
            None if self.ar is None else _ptr(self.ar[1], f64),
            None if self.ar is None else self.ar[2].ctypes.data_as(dp), _stream_handle(stream, self.voro.device))
        _lib.check(rc)
