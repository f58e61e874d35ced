"""The ray-tracing path on tensors that already live in HBM.

torch is used for device memory and streams only; the work is done by the sm_100a kernels in
libraytrace_b200.so through rtb200_dff_batch_device and, for derivatives, rtb200_dff_grad_device,
rtb200_dff_jac_device, rtb200_dff_normal_device and rtb200_dff_hess_device
(include/raytrace_b200.h).
"""
import torch

from . import _lib

_inited_device = None


def _ensure_device(index):
    global _inited_device
    if _inited_device != index:
        rc = _lib.load().rtb200_init(int(index))
        _lib.check(rc)
        _inited_device = index


def _ptr(t, dtype):
    if t is None:
        return None
    if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
        raise ValueError(f"expected a contiguous CUDA tensor of {dtype}, got {t.dtype} on {t.device}")
    return t.data_ptr()


def dff_batch_device(vels, depths, nlayers, src_offset, src_depth, tobs=None, sigma=None,
                     want_times=False, want_p=False, timeP=None, logL=None, p_out=None,
                     kmode=False, stream=None):
    """B models x NSrc sources on the GPU; every argument is a CUDA tensor.

    vels [B, ldv] f64, depths [B, ldz] f64, nlayers [B] i32, src_offset/src_depth [NSrc] f64,
    tobs [NSrc] f64 and sigma [B] f64 (both needed for logL).  Asynchronous on `stream`
    (default: torch's current stream).  Returns {"timeP", "p", "logL"} tensors (or None)."""
    dev = vels.device
    if not vels.is_cuda:
        raise ValueError("dff_batch_device needs CUDA tensors (there is no CPU path)")
    _ensure_device(dev.index if dev.index is not None else torch.cuda.current_device())
    B, ldv = vels.shape
    ldz = depths.shape[1] if depths.dim() == 2 else 0
    nsrc = src_offset.numel()
    f64 = torch.float64
    if timeP is None and want_times:
        timeP = torch.empty((B, nsrc), dtype=f64, device=dev)
    if p_out is None and want_p:
        p_out = torch.empty((B, nsrc), dtype=f64, device=dev)
    if tobs is not None and logL is None:
        logL = torch.empty((B,), dtype=f64, device=dev)
    rc = _lib.load().rtb200_dff_batch_device(
        _ptr(vels, f64), _ptr(depths, f64) if ldz else None, _ptr(nlayers, torch.int32), B, ldv, ldz,
        _ptr(src_offset, f64), _ptr(src_depth, f64), nsrc, _ptr(timeP, f64), _ptr(tobs, f64),
        _ptr(sigma, f64), _ptr(logL, f64), _ptr(p_out, f64), 1 if kmode else 0, _stream_handle(stream, dev))
    _lib.check(rc)
    return {"timeP": timeP, "p": p_out, "logL": logL}


def _stream_handle(stream, device):
    """The C ABI's handle of `stream` (default: torch's current stream on `device`)."""
    st = stream if stream is not None else torch.cuda.current_stream(device)
    # torch's default stream is the legacy stream (handle 0).  The C ABI reads NULL as "use the
    # library's own stream and synchronise", so name the legacy stream explicitly instead.
    return st.cuda_stream if st.cuda_stream != 0 else 1  # cudaStreamLegacy


def _check_grad_shapes(vels, depths, nlayers, src_offset, src_depth, per_ray):
    """Shapes of a gradient call, checked before anything touches the GPU.  Returns (B, ldv, ldz, S)."""
    if vels.dim() != 2 or depths.dim() != 2 or vels.shape[0] != depths.shape[0]:
        raise ValueError("vels and depths must be [B, ldv] and [B, ldz]")
    B, ldv = vels.shape
    ldz = depths.shape[1]
    if not 1 <= ldv <= 255:
        raise ValueError("ldv must be 1..255 (at most 254 interfaces)")
    if nlayers.dim() != 1 or nlayers.shape[0] != B:
        raise ValueError("nlayers must be [B]")
    if src_offset.dim() != 1 or src_depth.shape != src_offset.shape:
        raise ValueError("src_offset and src_depth must both be [NSrc]")
    S = src_offset.shape[0]
    for name, t in per_ray.items():
        if t is not None and tuple(t.shape) != (B, S):
            raise ValueError(f"{name} must be [B, NSrc] = [{B}, {S}], got {list(t.shape)}")
    return B, ldv, ldz, S


def _deriv_prologue(fn, vels, depths, nlayers, src_offset, src_depth, timeP, p, per_ray, outputs):
    """What the derivative wrappers share, every check before the library is loaded: the shapes
    (per_ray: the [B, NSrc] inputs by name; outputs(B, ldv, ldz, S): the wrapper's own checks, which
    return its (name, tensor or None, shape) outputs to check), CUDA tensors, the device.  Returns
    (B, ldv, ldz, S), the device and the 11 leading arguments of the C entry `fn`."""
    B, ldv, ldz, S = _check_grad_shapes(vels, depths, nlayers, src_offset, src_depth, per_ray)
    for name, t, shape in outputs(B, ldv, ldz, S):
        if t is not None and tuple(t.shape) != shape:
            raise ValueError(f"{name} must be {list(shape)}, got {list(t.shape)}")
    if not vels.is_cuda:
        raise ValueError(f"{fn} needs CUDA tensors (there is no CPU path)")
    dev = vels.device
    _ensure_device(dev.index if dev.index is not None else torch.cuda.current_device())
    f64 = torch.float64
    args = (_ptr(vels, f64), _ptr(depths, f64) if ldz else None, _ptr(nlayers, torch.int32), B, ldv, ldz,
            _ptr(src_offset, f64), _ptr(src_depth, f64), S, _ptr(timeP, f64), _ptr(p, f64))
    return (B, ldv, ldz, S), dev, args


def dff_grad_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, w, gvels=None,
                    gdepths=None, want_src=False, dtdr=None, dtdd=None, kmode=False, stream=None):
    """Vector-Jacobian product of the travel times dff_batch_device returned (timeP, p [B, NSrc])
    with weights w [B, NSrc], on the GPU (rtb200_dff_grad_device; DESIGN.md section 11).

    Returns {"gvels" [B, ldv], "gdepths" [B, ldz], "dtdr", "dtdd" [B, NSrc] or None}:
    gvels[b, i] = sum_s w[b, s] dT[b, s]/dV_i, gdepths likewise for the interfaces (kmode: ziface),
    dtdr / dtdd the per-ray derivatives with respect to the source offset and depth (want_src).
    Asynchronous on `stream` (default: torch's current stream)."""
    (B, ldv, ldz, S), dev, args = _deriv_prologue(
        "dff_grad_device", vels, depths, nlayers, src_offset, src_depth, timeP, p,
        {"timeP": timeP, "p": p, "w": w, "dtdr": dtdr, "dtdd": dtdd},
        lambda B, ldv, ldz, S: (("gvels", gvels, (B, ldv)), ("gdepths", gdepths, (B, ldz))))
    f64 = torch.float64
    if gvels is None:
        gvels = torch.empty((B, ldv), dtype=f64, device=dev)
    if gdepths is None:
        gdepths = torch.empty((B, ldz), dtype=f64, device=dev)
    if want_src and dtdr is None:
        dtdr = torch.empty((B, S), dtype=f64, device=dev)
    if want_src and dtdd is None:
        dtdd = torch.empty((B, S), dtype=f64, device=dev)
    rc = _lib.load().rtb200_dff_grad_device(
        *args, _ptr(w, f64), _ptr(gvels, f64), _ptr(gdepths, f64) if ldz else None, _ptr(dtdr, f64),
        _ptr(dtdd, f64), 1 if kmode else 0, _stream_handle(stream, dev))
    _lib.check(rc)
    return {"gvels": gvels, "gdepths": gdepths, "dtdr": dtdr, "dtdd": dtdd}


def dff_jac_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, jvels=None, jdepths=None,
                   want_src=False, dtdr=None, dtdd=None, kmode=False, stream=None):
    """Jacobian of the travel times dff_batch_device returned (timeP, p [B, NSrc]), per ray, on the
    GPU (rtb200_dff_jac_device; DESIGN.md section 12).

    Returns {"jvels" [B, NSrc, ldv], "jdepths" [B, NSrc, ldz], "dtdr", "dtdd" [B, NSrc] or None}:
    jvels[b, s, i] = dT[b, s]/dV_i, jdepths[b, s, j] = dT[b, s]/dz_j (kmode: ziface), dtdr / dtdd
    as dff_grad_device returns them (want_src).  Asynchronous on `stream` (default: torch's
    current stream)."""
    (B, ldv, ldz, S), dev, args = _deriv_prologue(
        "dff_jac_device", vels, depths, nlayers, src_offset, src_depth, timeP, p,
        {"timeP": timeP, "p": p, "dtdr": dtdr, "dtdd": dtdd},
        lambda B, ldv, ldz, S: (("jvels", jvels, (B, S, ldv)), ("jdepths", jdepths, (B, S, ldz))))
    f64 = torch.float64
    if jvels is None:
        jvels = torch.empty((B, S, ldv), dtype=f64, device=dev)
    if jdepths is None:
        jdepths = torch.empty((B, S, ldz), dtype=f64, device=dev)
    if want_src and dtdr is None:
        dtdr = torch.empty((B, S), dtype=f64, device=dev)
    if want_src and dtdd is None:
        dtdd = torch.empty((B, S), dtype=f64, device=dev)
    rc = _lib.load().rtb200_dff_jac_device(
        *args, _ptr(jvels, f64), _ptr(jdepths, f64) if ldz else None, _ptr(dtdr, f64), _ptr(dtdd, f64),
        1 if kmode else 0, _stream_handle(stream, dev))
    _lib.check(rc)
    return {"jvels": jvels, "jdepths": jdepths, "dtdr": dtdr, "dtdd": dtdd}


def dff_normal_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, tobs=None, JtJ=None, Jtr=None,
                      kmode=False, stream=None):
    """Gauss-Newton normal equations of the travel times dff_batch_device returned (timeP, p
    [B, NSrc]), per model, on the GPU without storing the Jacobian (rtb200_dff_normal_device;
    DESIGN.md section 13).

    Returns {"JtJ" [B, P, P], "Jtr" [B, P] or None}, P = ldv + ldz: with J the rows dff_jac_device
    writes, [jvels | jdepths], JtJ = J^T J and, given tobs [NSrc], Jtr = J^T (tobs - timeP), each
    sum in source order.  Asynchronous on `stream` (default: torch's current stream)."""
    def outputs(B, ldv, ldz, S):
        if tobs is not None and tuple(tobs.shape) != (S,):
            raise ValueError(f"tobs must be [NSrc] = [{S}], got {list(tobs.shape)}")
        if Jtr is not None and tobs is None:
            raise ValueError("Jtr needs tobs")
        P = ldv + ldz
        return ("JtJ", JtJ, (B, P, P)), ("Jtr", Jtr, (B, P))

    (B, ldv, ldz, S), dev, args = _deriv_prologue(
        "dff_normal_device", vels, depths, nlayers, src_offset, src_depth, timeP, p,
        {"timeP": timeP, "p": p}, outputs)
    f64 = torch.float64
    P = ldv + ldz
    if JtJ is None:
        JtJ = torch.empty((B, P, P), dtype=f64, device=dev)
    if tobs is not None and Jtr is None:
        Jtr = torch.empty((B, P), dtype=f64, device=dev)
    rc = _lib.load().rtb200_dff_normal_device(
        *args, _ptr(tobs, f64), _ptr(JtJ, f64), _ptr(Jtr, f64), 1 if kmode else 0, _stream_handle(stream, dev))
    _lib.check(rc)
    return {"JtJ": JtJ, "Jtr": Jtr}


def dff_hess_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, w, H=None, kmode=False,
                    stream=None):
    """Weighted second derivatives of the travel times dff_batch_device returned (timeP, p
    [B, NSrc]), per model, on the GPU (rtb200_dff_hess_device; DESIGN.md section 14).

    Returns {"H" [B, P, P]}, P = ldv + ldz: H[b] = sum_s w[b, s] d2T[b, s] / dtheta dtheta^T over the
    columns [vels | depths] of dff_normal_device, each sum in source order; exactly symmetric.
    Asynchronous on `stream` (default: torch's current stream)."""
    def outputs(B, ldv, ldz, S):
        P = ldv + ldz
        return (("H", H, (B, P, P)),)

    (B, ldv, ldz, S), dev, args = _deriv_prologue(
        "dff_hess_device", vels, depths, nlayers, src_offset, src_depth, timeP, p,
        {"timeP": timeP, "p": p, "w": w}, outputs)
    f64 = torch.float64
    P = ldv + ldz
    if H is None:
        H = torch.empty((B, P, P), dtype=f64, device=dev)
    rc = _lib.load().rtb200_dff_hess_device(
        *args, _ptr(w, f64), _ptr(H, f64), 1 if kmode else 0, _stream_handle(stream, dev))
    _lib.check(rc)
    return {"H": H}
