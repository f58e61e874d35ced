"""Host-side mirror of the reference's interface for the ray-tracing path.

Names and argument meaning follow the reference (module raymod, subroutineR-quiet.f90, and
LOGLHOOD_RT, ray_tracing_sampling/loglhood.f90); every function goes through the C ABI of
libraytrace_b200.so with HOST buffers, exactly as R's .Fortran or a Fortran caller would:
scalars by reference, arrays as plain contiguous doubles.  Nothing here computes travel
times on the CPU.
"""
import ctypes as C

import numpy as np

from . import _lib

_DP = C.POINTER(C.c_double)
_IP = C.POINTER(C.c_int)


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return None if a is None else a.ctypes.data_as(_DP)


def _ci(v):
    return C.byref(C.c_int(int(v)))


def dff(vels, depths, src_offset, src_depth, keep_delta=-1, NLayers=None, NSrc=None):
    """`.Fortran("dff", vels, depths, NLayers, src_offset, src_depth, NSrc, timeP, keep_delta)`
    (rayTracerR.R:31-33; symbol dff_, subroutineR-quiet.f90:408).  Returns timeP[NSrc].
    keep_delta > 0 rewrites ./rays.dat."""
    v, z, so, sd = _d(vels), _d(depths), _d(src_offset), _d(src_depth)
    nlay = z.size if NLayers is None else int(NLayers)
    nsrc = so.size if NSrc is None else int(NSrc)
    if v.size < nlay + 1 or z.size < nlay or so.size < nsrc or sd.size < nsrc:
        raise ValueError("array sizes do not match NLayers / NSrc")
    t = np.zeros(nsrc)
    _lib.load().dff_(_p(v), _p(z), _ci(nlay), _p(so), _p(sd), _ci(nsrc), _p(t), _ci(keep_delta))
    _lib.check()
    return t


def dff7(vels, depths, src_offset, src_depth):
    """The 7-argument dff of subroutineR.f90:405 / README.md:16-21 (no keep_delta)."""
    v, z, so, sd = _d(vels), _d(depths), _d(src_offset), _d(src_depth)
    t = np.zeros(so.size)
    _lib.load().dff7_(_p(v), _p(z), _ci(z.size), _p(so), _p(sd), _ci(so.size), _p(t))
    _lib.check()
    return t


def TraceRays(vels, depths, NLayers, src_offset, src_depth, NSrc, keep_delta=-1, symbol="tracerays_"):
    """CALL TraceRays(vels, depths, NLayers, src_offset, src_depth, NSrc, timeP, keep_delta)
    (subroutineR-quiet.f90:467; call sites loglhood.f90:135,144).  Returns timeP.  `symbol` picks
    the exported name: tracerays_ (the shim's) or a compiler-mangled module-procedure name
    (__raymod_MOD_tracerays, raymod_mp_tracerays_, raymod_tracerays_)."""
    v, z, so, sd = _d(vels), _d(depths), _d(src_offset), _d(src_depth)
    t = np.zeros(int(NSrc))
    getattr(_lib.load(), symbol)(_p(v), _p(z), _ci(NLayers), _p(so), _p(sd), _ci(NSrc), _p(t),
                                 _ci(keep_delta))
    _lib.check()
    return t


def dff_batch(vels, depths, nlayers, src_offset, src_depth, tobs=None, sigma=None,
              want_times=True, want_p=False, out_times=None, out_logL=None, out_p=None):
    """Many models per call.  vels[B, ldv], depths[B, ldz], nlayers[B]; shared sources.

    Returns a dict with "timeP" [B, NSrc] (if want_times), "p" [B, NSrc] (if want_p) and
    "logL" [B] (if tobs and sigma are given: the fused LOGLHOOD_RT value)."""
    v = _d(vels)
    z = _d(depths)
    if v.ndim != 2 or z.ndim != 2 or v.shape[0] != z.shape[0]:
        raise ValueError("vels and depths must be [B, ldv] and [B, ldz]")
    nl = np.ascontiguousarray(nlayers, dtype=np.int32)
    so, sd = _d(src_offset), _d(src_depth)
    B, nsrc = v.shape[0], so.size
    if nl.size != B or sd.size != nsrc:
        raise ValueError("nlayers / source sizes do not match")
    nl_max = int(nl.max()) if B else 0
    if nl_max + 1 > v.shape[1] or nl_max > max(z.shape[1], 0):
        raise ValueError("nlayers exceeds the row length of vels / depths")
    def _out(a, shape, name):
        # the library writes prod(shape) doubles through this pointer: refuse anything else
        if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
                and a.flags["WRITEABLE"] and a.shape == shape):
            raise ValueError(f"{name} must be a writable C-contiguous float64 array of shape {shape}")
        return a

    t = _out(out_times, (B, nsrc), "out_times") if out_times is not None else (np.empty((B, nsrc)) if want_times else None)
    p = _out(out_p, (B, nsrc), "out_p") if out_p is not None else (np.empty((B, nsrc)) if want_p else None)
    ll = ob = sg = None
    if tobs is not None:
        if sigma is None:
            raise ValueError("sigma [B] is required with tobs (the fused likelihood)")
        ob, sg = _d(tobs), _d(sigma)
        if ob.size != nsrc or sg.size != B:
            raise ValueError("tobs must be [NSrc] and sigma [B]")
        ll = _out(out_logL, (B,), "out_logL") if out_logL is not None else np.empty(B)
    rc = _lib.load().dff_batch(_p(v), _p(z), nl.ctypes.data_as(_IP), _ci(B), _ci(v.shape[1]),
                               _ci(z.shape[1]), _p(so), _p(sd), _ci(nsrc), _p(t), _p(ob), _p(sg),
                               _p(ll), _p(p))
    _lib.check(rc)
    return {"timeP": t, "p": p, "logL": ll}


def dff_batch_grad(vels, depths, nlayers, src_offset, src_depth, w, want_times=False, want_p=False,
                   want_src=False):
    """dff_batch and the gradient of its travel times in one call (DESIGN.md section 11).

    w [B, NSrc] weights the rays.  Returns a dict with "gvels" [B, ldv] = sum_s w dT/dV,
    "gdepths" [B, ldz] = sum_s w dT/dz, and, on request, "timeP" / "p" [B, NSrc] of the forward
    and "dtdr" / "dtdd" [B, NSrc], the per-ray derivatives with respect to the source offset and
    depth (None otherwise)."""
    v = _d(vels)
    z = _d(depths)
    if v.ndim != 2 or z.ndim != 2 or v.shape[0] != z.shape[0]:
        raise ValueError("vels and depths must be [B, ldv] and [B, ldz]")
    nl = np.ascontiguousarray(nlayers, dtype=np.int32)
    so, sd = _d(src_offset), _d(src_depth)
    B, ldv, ldz, nsrc = v.shape[0], v.shape[1], z.shape[1], so.size
    if nl.shape != (B,) or so.ndim != 1 or sd.shape != so.shape:
        raise ValueError("nlayers must be [B], src_offset and src_depth [NSrc]")
    if not 1 <= ldv <= 255:
        raise ValueError("ldv must be 1..255 (at most 254 interfaces)")
    if B and (nl.min() < 0 or int(nl.max()) + 1 > ldv or int(nl.max()) > ldz):
        raise ValueError("nlayers exceeds the row length of vels / depths")
    ww = _d(w)
    if ww.shape != (B, nsrc):
        raise ValueError(f"w must be [B, NSrc] = [{B}, {nsrc}], got {list(ww.shape)}")
    gv, gz = np.empty((B, ldv)), np.empty((B, ldz))
    t = np.empty((B, nsrc)) if want_times else None
    p = np.empty((B, nsrc)) if want_p else None
    dr = np.empty((B, nsrc)) if want_src else None
    dd = np.empty((B, nsrc)) if want_src else None
    rc = _lib.load().dff_batch_grad(_p(v), _p(z), nl.ctypes.data_as(_IP), _ci(B), _ci(ldv), _ci(ldz),
                                    _p(so), _p(sd), _ci(nsrc), _p(ww), _p(t), _p(p), _p(gv), _p(gz),
                                    _p(dr), _p(dd))
    _lib.check(rc)
    return {"gvels": gv, "gdepths": gz, "timeP": t, "p": p, "dtdr": dr, "dtdd": dd}


def dff_batch_jac(vels, depths, nlayers, src_offset, src_depth, want_times=False, want_p=False,
                  want_src=False):
    """dff_batch and the Jacobian of its travel times in one call (DESIGN.md section 12).

    Returns a dict with "jvels" [B, NSrc, ldv] = dT/dV and "jdepths" [B, NSrc, ldz] = dT/dz per
    ray, and, on request, "timeP" / "p" [B, NSrc] of the forward and "dtdr" / "dtdd" [B, NSrc],
    the per-ray derivatives with respect to the source offset and depth (None otherwise)."""
    v = _d(vels)
    z = _d(depths)
    if v.ndim != 2 or z.ndim != 2 or v.shape[0] != z.shape[0]:
        raise ValueError("vels and depths must be [B, ldv] and [B, ldz]")
    nl = np.ascontiguousarray(nlayers, dtype=np.int32)
    so, sd = _d(src_offset), _d(src_depth)
    B, ldv, ldz, nsrc = v.shape[0], v.shape[1], z.shape[1], so.size
    if nl.shape != (B,) or so.ndim != 1 or sd.shape != so.shape:
        raise ValueError("nlayers must be [B], src_offset and src_depth [NSrc]")
    if not 1 <= ldv <= 255:
        raise ValueError("ldv must be 1..255 (at most 254 interfaces)")
    if B and (nl.min() < 0 or int(nl.max()) + 1 > ldv or int(nl.max()) > ldz):
        raise ValueError("nlayers exceeds the row length of vels / depths")
    jv, jz = np.empty((B, nsrc, ldv)), np.empty((B, nsrc, ldz))
    t = np.empty((B, nsrc)) if want_times else None
    p = np.empty((B, nsrc)) if want_p else None
    dr = np.empty((B, nsrc)) if want_src else None
    dd = np.empty((B, nsrc)) if want_src else None
    rc = _lib.load().dff_batch_jac(_p(v), _p(z), nl.ctypes.data_as(_IP), _ci(B), _ci(ldv), _ci(ldz),
                                   _p(so), _p(sd), _ci(nsrc), _p(t), _p(p), _p(jv), _p(jz), _p(dr),
                                   _p(dd))
    _lib.check(rc)
    return {"jvels": jv, "jdepths": jz, "timeP": t, "p": p, "dtdr": dr, "dtdd": dd}


def dff_batch_normal(vels, depths, nlayers, src_offset, src_depth, tobs=None, want_times=False,
                     want_p=False):
    """dff_batch and the Gauss-Newton normal equations of its travel times in one call (DESIGN.md
    section 13).

    Returns a dict with "JtJ" [B, P, P] = J^T J, P = ldv + ldz, over the rows dff_batch_jac
    returns ([jvels | jdepths]), "Jtr" [B, P] = J^T (tobs - timeP) when tobs [NSrc] is given, and,
    on request, "timeP" / "p" [B, NSrc] of the forward (None otherwise)."""
    v = _d(vels)
    z = _d(depths)
    if v.ndim != 2 or z.ndim != 2 or v.shape[0] != z.shape[0]:
        raise ValueError("vels and depths must be [B, ldv] and [B, ldz]")
    nl = np.ascontiguousarray(nlayers, dtype=np.int32)
    so, sd = _d(src_offset), _d(src_depth)
    B, ldv, ldz, nsrc = v.shape[0], v.shape[1], z.shape[1], so.size
    if nl.shape != (B,) or so.ndim != 1 or sd.shape != so.shape:
        raise ValueError("nlayers must be [B], src_offset and src_depth [NSrc]")
    to = None if tobs is None else _d(tobs)
    if to is not None and to.shape != so.shape:
        raise ValueError("tobs must be [NSrc]")
    if not 1 <= ldv <= 255:
        raise ValueError("ldv must be 1..255 (at most 254 interfaces)")
    if B and (nl.min() < 0 or int(nl.max()) + 1 > ldv or int(nl.max()) > ldz):
        raise ValueError("nlayers exceeds the row length of vels / depths")
    P = ldv + ldz
    jtj = np.empty((B, P, P))
    jtr = np.empty((B, P)) if to is not None else None
    t = np.empty((B, nsrc)) if want_times else None
    p = np.empty((B, nsrc)) if want_p else None
    rc = _lib.load().dff_batch_normal(_p(v), _p(z), nl.ctypes.data_as(_IP), _ci(B), _ci(ldv), _ci(ldz),
                                      _p(so), _p(sd), _ci(nsrc), _p(to), _p(t), _p(p), _p(jtj), _p(jtr))
    _lib.check(rc)
    return {"JtJ": jtj, "Jtr": jtr, "timeP": t, "p": p}


def loglhood_batch(k, voro_vp, ziface, src_offset, src_depth, DobsRT, sdparRT, want_pred=False):
    """LOGLHOOD / LOGLHOOD_RT (loglhood.f90:3-32,35-211) over B chain states.

    k[B] node counts, voro_vp[B, >=max k] = obj%voro(1:k,2), ziface[B, >=max(k)-1] =
    obj%ziface(1:k-1), sdparRT[B] = obj%sdparRT(1), DobsRT[NDAT_RT].  Returns (logL[B],
    DpredRT[B, NDAT_RT] or None)."""
    v, z = _d(voro_vp), _d(ziface)
    kk = np.ascontiguousarray(k, dtype=np.int32)
    so, sd, ob, sg = _d(src_offset), _d(src_depth), _d(DobsRT), _d(sdparRT)
    B, nsrc = v.shape[0], so.size
    if z.ndim != 2:
        z = z.reshape(B, -1)
    if B and (kk.min() < 1 or kk.max() > v.shape[1] or kk.max() - 1 > z.shape[1]):
        raise ValueError("k out of range for voro_vp / ziface")
    ll = np.empty(B)
    pred = np.empty((B, nsrc)) if want_pred else None
    rc = _lib.load().loglhood_batch(kk.ctypes.data_as(_IP), _p(v), _p(z) if z.size else None,
                                    _ci(B), _ci(v.shape[1]), _ci(z.shape[1]), _p(so), _p(sd),
                                    _ci(nsrc), _p(ob), _p(sg), _p(ll), _p(pred))
    _lib.check(rc)
    return ll, pred


def loglhood_batch_ar(k, voro_vp, ziface, src_offset, src_depth, DobsRT, sdparRT, idxarRT, arparRT,
                      armxRT=0.5, want_pred=False):
    """loglhood_batch with the AR(1) residual error model (IAR = 1; loglhood.f90:171-182,616-701):
    idxarRT[B] switches it per state, arparRT[B] is the coefficient, armxRT the bound."""
    v, z = _d(voro_vp), _d(ziface)
    kk = np.ascontiguousarray(k, dtype=np.int32)
    ix = np.ascontiguousarray(idxarRT, dtype=np.int32)
    so, sd, ob, sg, ap = _d(src_offset), _d(src_depth), _d(DobsRT), _d(sdparRT), _d(arparRT)
    B, nsrc = v.shape[0], so.size
    if z.ndim != 2:
        z = z.reshape(B, -1)
    if ix.size != B or ap.size != B:
        raise ValueError("idxarRT and arparRT must be [B]")
    ll = np.empty(B)
    pred = np.empty((B, nsrc)) if want_pred else None
    rc = _lib.load().loglhood_batch_ar(kk.ctypes.data_as(_IP), _p(v), _p(z) if z.size else None,
                                       _ci(B), _ci(v.shape[1]), _ci(z.shape[1]), _p(so), _p(sd),
                                       _ci(nsrc), _p(ob), _p(sg), ix.ctypes.data_as(_IP), _p(ap),
                                       C.byref(C.c_double(float(armxRT))), _p(ll), _p(pred))
    _lib.check(rc)
    return ll, pred


def loglhood_batch_voro(k, voro, src_offset, src_depth, DobsRT, sdparRT, want_pred=False,
                        want_sorted=False):
    """INTERPLAYER_novar + LOGLHOOD (loglhood.f90:214-295, :3-211) over B chain states given as
    unsorted Voronoi nodes voro[B, 2, ldk] (depth row, vp row).  Returns (logL[B], DpredRT or
    None, sorted voro or None)."""
    vo = _d(voro)
    kk = np.ascontiguousarray(k, dtype=np.int32)
    so, sd, ob, sg = _d(src_offset), _d(src_depth), _d(DobsRT), _d(sdparRT)
    if vo.ndim != 3 or vo.shape[1] != 2:
        raise ValueError("voro must be [B, 2, ldk]")
    B, ldk, nsrc = vo.shape[0], vo.shape[2], so.size
    if B and (kk.min() < 1 or kk.max() > ldk):
        raise ValueError("k out of range")
    ll = np.empty(B)
    pred = np.empty((B, nsrc)) if want_pred else None
    srt = np.empty_like(vo) if want_sorted else None
    rc = _lib.load().loglhood_batch_voro(kk.ctypes.data_as(_IP), _p(vo), _ci(B), _ci(ldk), _p(so),
                                         _p(sd), _ci(nsrc), _p(ob), _p(sg), _p(ll), _p(pred), _p(srt))
    _lib.check(rc)
    return ll, pred, srt


def set_option(name, value):
    if _lib.load().rtb200_set_option(name.encode(), float(value)) != 0:
        raise KeyError(name)


def get_stat(name):
    return _lib.load().rtb200_get_stat(name.encode())


def fp64_peak_tflops(repeats=3):
    v = _lib.load().rtb200_fp64_peak_tflops(int(repeats))
    _lib.check()
    return v


def selftest_fast_division(samples=1e9, seed=1):
    """Mismatches between the hot loop's rsqrt-seeded sqrt/divisions and CUDA's built-ins."""
    bad = _lib.load().rtb200_selftest_fast_division(float(samples), int(seed))
    if bad < 0:
        _lib.check(-1)
    return int(bad)


def shard_range(B, rank, world):
    lo, hi = C.c_longlong(), C.c_longlong()
    _lib.load().rtb200_shard_range(int(B), int(rank), int(world), C.byref(lo), C.byref(hi))
    return lo.value, hi.value
