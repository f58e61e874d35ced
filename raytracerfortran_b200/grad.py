"""Travel times and LOGLHOOD_RT as torch.autograd functions (DESIGN.md section 11).

    T    = travel_times(vels, depths, nlayers, src_offset, src_depth, kmode=False)       # [B, S]
    logL = loglhood(vels, depths, nlayers, src_offset, src_depth, tobs, sigma, kmode=False)  # [B]

The forward values are those of device.dff_batch_device, bit for bit.  The backward pass runs the
library's gradient kernel (rtb200_dff_grad_device) at the ray parameters the forward returned: the
derivatives are those of the exact travel-time function there, not of the solver's stopped
iteration.  Gradients flow to vels, depths (kmode: vp nodes and ziface), src_offset, src_depth,
and for loglhood to tobs and sigma; nlayers is not differentiable.  Every tensor is a CUDA
tensor, float64 (nlayers int32).  Both functions are once differentiable.

    J = jacobian(vels, depths, nlayers, src_offset, src_depth, kmode=False)  # dict, no graph

returns the travel times with their per-ray derivatives (rtb200_dff_jac_device), the rows
Gauss-Newton and linearised-uncertainty computations need.

    N = normal_equations(vels, depths, nlayers, src_offset, src_depth, tobs=None, kmode=False)

returns the travel times with the per-model normal equations J^T J and J^T (tobs - T) of those
rows (rtb200_dff_normal_device), accumulated on the device without writing J.
"""
import torch
from torch.autograd.function import once_differentiable

from . import device

_HUGE = torch.finfo(torch.float64).max      # logL = -HUGE marks a rejected model (loglhood.f90:200-203)


def _src_grads(ctx, w, r, i_off, i_dep):
    """Source gradients: the sum over models of w dT/dR and w dT/dd."""
    g_off = (w * r["dtdr"]).sum(0) if ctx.needs_input_grad[i_off] else None
    g_dep = (w * r["dtdd"]).sum(0) if ctx.needs_input_grad[i_dep] else None
    return g_off, g_dep


class _TravelTimes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vels, depths, nlayers, src_offset, src_depth, kmode):
        out = device.dff_batch_device(vels, depths, nlayers, src_offset, src_depth, want_times=True,
                                      want_p=True, kmode=kmode)
        ctx.save_for_backward(vels, depths, nlayers, src_offset, src_depth, out["timeP"], out["p"])
        ctx.kmode = kmode
        return out["timeP"]

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_t):
        vels, depths, nlayers, src_offset, src_depth, timeP, p = ctx.saved_tensors
        w = grad_t.contiguous()
        r = device.dff_grad_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, w,
                                   want_src=ctx.needs_input_grad[3] or ctx.needs_input_grad[4],
                                   kmode=ctx.kmode)
        g_off, g_dep = _src_grads(ctx, w, r, 3, 4)
        return (r["gvels"] if ctx.needs_input_grad[0] else None,
                r["gdepths"] if ctx.needs_input_grad[1] else None, None, g_off, g_dep, None)


class _LogLhood(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vels, depths, nlayers, src_offset, src_depth, tobs, sigma, kmode):
        out = device.dff_batch_device(vels, depths, nlayers, src_offset, src_depth, tobs=tobs,
                                      sigma=sigma, want_times=True, want_p=True, kmode=kmode)
        ctx.save_for_backward(vels, depths, nlayers, src_offset, src_depth, tobs, sigma,
                              out["timeP"], out["p"], out["logL"])
        ctx.kmode = kmode
        return out["logL"]

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_l):
        vels, depths, nlayers, src_offset, src_depth, tobs, sigma, timeP, p, logL = ctx.saved_tensors
        # logL = C - sum(res^2) / (2 sigma^2) - N log sigma, res = tobs - T; a model whose logL was
        # replaced by -HUGE has zero gradient
        rejected = logL == -_HUGE
        zero = torch.zeros((), dtype=grad_l.dtype, device=grad_l.device)
        g = torch.where(rejected, zero, grad_l)
        res = tobs[None, :] - timeP
        # masked after the product too: sigma = 0 or NaN would make 0 * inf = NaN
        w = torch.where(rejected[:, None], zero, g[:, None] * (res / (sigma * sigma)[:, None])).contiguous()
        need_model = any(ctx.needs_input_grad[:5])
        r = None
        if need_model:
            r = device.dff_grad_device(vels, depths, nlayers, src_offset, src_depth, timeP, p, w,
                                       want_src=ctx.needs_input_grad[3] or ctx.needs_input_grad[4],
                                       kmode=ctx.kmode)
            g_off, g_dep = _src_grads(ctx, w, r, 3, 4)
        else:
            g_off = g_dep = None
        n = float(timeP.shape[1])
        g_tobs = -w.sum(0) if ctx.needs_input_grad[5] else None
        g_sigma = (torch.where(rejected, zero, g * ((res * res).sum(1) / (sigma * sigma * sigma) - n / sigma))
                   if ctx.needs_input_grad[6] else None)
        return (r["gvels"] if r is not None and ctx.needs_input_grad[0] else None,
                r["gdepths"] if r is not None and ctx.needs_input_grad[1] else None, None,
                g_off, g_dep, g_tobs, g_sigma, None)


def _check(vels, depths, nlayers, src_offset, src_depth):
    B, _, _, S = device._check_grad_shapes(vels, depths, nlayers, src_offset, src_depth, {})
    for name, t, dtype in (("vels", vels, torch.float64), ("depths", depths, torch.float64),
                           ("nlayers", nlayers, torch.int32), ("src_offset", src_offset, torch.float64),
                           ("src_depth", src_depth, torch.float64)):
        if t.dtype != dtype:
            raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if not all(t.is_cuda for t in (vels, depths, nlayers, src_offset, src_depth)):
        raise ValueError("the gradient path needs CUDA tensors (there is no CPU path)")
    return B, S


def travel_times(vels, depths, nlayers, src_offset, src_depth, kmode=False):
    """Travel times T [B, NSrc] of B layered models (vels [B, ldv], depths [B, ldz], nlayers [B];
    kmode: node counts k, vp nodes and ziface as in loglhood_batch) and shared sources, with
    gradients with respect to vels, depths, src_offset and src_depth."""
    _check(vels, depths, nlayers, src_offset, src_depth)
    return _TravelTimes.apply(vels.contiguous(), depths.contiguous(), nlayers.contiguous(),
                              src_offset.contiguous(), src_depth.contiguous(), bool(kmode))


def jacobian(vels, depths, nlayers, src_offset, src_depth, kmode=False, want_src=True):
    """Travel times and their Jacobian per ray, without an autograd graph (DESIGN.md section 12).

    Returns {"timeP", "p" [B, NSrc], "jvels" [B, NSrc, ldv], "jdepths" [B, NSrc, ldz],
    "dtdr", "dtdd" [B, NSrc] (None unless want_src)}: jvels[b, s, i] = dT[b, s]/dV_i and
    jdepths[b, s, j] = dT[b, s]/dz_j, the rows whose sums over s travel_times' backward forms.
    timeP is dff_batch_device's, bit for bit."""
    _check(vels, depths, nlayers, src_offset, src_depth)
    with torch.no_grad():
        args = tuple(t.detach().contiguous() for t in (vels, depths, nlayers, src_offset, src_depth))
        out = device.dff_batch_device(*args, want_times=True, want_p=True, kmode=bool(kmode))
        r = device.dff_jac_device(*args, out["timeP"], out["p"], want_src=want_src, kmode=bool(kmode))
    return {"timeP": out["timeP"], "p": out["p"], **r}


def normal_equations(vels, depths, nlayers, src_offset, src_depth, tobs=None, kmode=False):
    """Travel times and the Gauss-Newton normal equations of their Jacobian, per model, without an
    autograd graph (DESIGN.md section 13).

    Returns {"timeP", "p" [B, NSrc], "JtJ" [B, P, P], "Jtr" [B, P] or None}, P = ldv + ldz: with
    J_s = [jvels[b, s] | jdepths[b, s]] the rows jacobian() returns, JtJ[b] = sum_s J_s^T J_s and,
    given tobs [NSrc], Jtr[b] = sum_s J_s^T (tobs_s - timeP[b, s]).  The Jacobian is never stored.
    timeP is dff_batch_device's, bit for bit."""
    _, S = _check(vels, depths, nlayers, src_offset, src_depth)
    if tobs is not None and (tobs.dtype != torch.float64 or tuple(tobs.shape) != (S,)):
        raise ValueError(f"tobs must be a float64 [NSrc] = [{S}] tensor")
    with torch.no_grad():
        args = tuple(t.detach().contiguous() for t in (vels, depths, nlayers, src_offset, src_depth))
        out = device.dff_batch_device(*args, want_times=True, want_p=True, kmode=bool(kmode))
        r = device.dff_normal_device(*args, out["timeP"], out["p"],
                                     tobs=None if tobs is None else tobs.detach().contiguous(),
                                     kmode=bool(kmode))
    return {"timeP": out["timeP"], "p": out["p"], **r}


def loglhood(vels, depths, nlayers, src_offset, src_depth, tobs, sigma, kmode=False):
    """LOGLHOOD_RT logL [B] of B models against observations tobs [NSrc] with data errors
    sigma [B], with gradients with respect to the models, the sources, tobs and sigma."""
    B, S = _check(vels, depths, nlayers, src_offset, src_depth)
    if tobs.dim() != 1 or tobs.shape[0] != S:
        raise ValueError(f"tobs must be [NSrc] = [{S}], got {list(tobs.shape)}")
    if sigma.dim() != 1 or sigma.shape[0] != B:
        raise ValueError(f"sigma must be [B] = [{B}], got {list(sigma.shape)}")
    if tobs.dtype != torch.float64 or sigma.dtype != torch.float64 or not (tobs.is_cuda and sigma.is_cuda):
        raise ValueError("tobs and sigma must be CUDA float64 tensors")
    return _LogLhood.apply(vels.contiguous(), depths.contiguous(), nlayers.contiguous(),
                           src_offset.contiguous(), src_depth.contiguous(), tobs.contiguous(),
                           sigma.contiguous(), bool(kmode))
