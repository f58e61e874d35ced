"""ctypes binding of libraytrace_b200.so -- the C ABI declared in include/raytrace_b200.h.

Loading never falls back to anything: a missing library is an ImportError-like RuntimeError,
a missing GPU makes every compute call raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# RTB200_LIB lets profiling scripts load an experimental build of the same library
LIB_PATH = os.environ.get("RTB200_LIB") or os.path.join(_HERE, "libraytrace_b200.so")

# every symbol include/raytrace_b200.h declares
EXPORTS = (
    "dff_", "dff7_", "tracerays_", "__raymod_MOD_tracerays", "raymod_mp_tracerays_", "raymod_tracerays_", "dff_batch", "dff_batch_grad", "dff_batch_jac", "dff_batch_normal", "dff_batch_status", "dff_batch_status_", "loglhood_batch", "loglhood_batch_ar", "loglhood_batch_voro",
    "rtb200_dff_batch_device", "rtb200_dff_grad_device", "rtb200_dff_jac_device", "rtb200_dff_normal_device", "rtb200_mh_step_device", "rtb200_mh_step_device_ev", "rtb200_mh_moves_device", "rtb200_mh_moves_device_ex", "rtb200_bd_step_device_ex", "rtb200_bd_step_device", "rtb200_sd_step_device", "rtb200_ar_step_device", "rtb200_set_chain_ar",
    "rtb200_swap_pack_device", "rtb200_swap_round_device", "rtb200_mcmc_workspace_bytes", "rtb200_mcmc_iterations_device",
    "rtb200_init", "rtb200_shutdown", "rtb200_last_error", "rtb200_device_count",
    "rtb200_set_option", "rtb200_get_stat", "rtb200_fp64_peak_tflops", "rtb200_shard_range",
    "rtb200_selftest_fast_division",
)

_lib = None


class RayTraceError(RuntimeError):
    """A call into libraytrace_b200 failed (no GPU, CUDA error, bad geometry)."""


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RayTraceError(
            f"{LIB_PATH} is missing: build it with `python -m raytracerfortran_b200.build` "
            "(there is no CPU fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    dp, ip, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_int, C.c_double
    vp = C.c_void_p
    lib.dff_.restype = None
    lib.dff_.argtypes = [dp, dp, ip, dp, dp, ip, dp, ip]
    lib.tracerays_.restype = None
    lib.tracerays_.argtypes = [dp, dp, ip, dp, dp, ip, dp, ip]
    for alias in ("__raymod_MOD_tracerays", "raymod_mp_tracerays_", "raymod_tracerays_"):
        getattr(lib, alias).restype = None
        getattr(lib, alias).argtypes = [dp, dp, ip, dp, dp, ip, dp, ip]
    lib.dff7_.restype = None
    lib.dff7_.argtypes = [dp, dp, ip, dp, dp, ip, dp]
    lib.dff_batch.restype = i
    lib.dff_batch.argtypes = [dp, dp, ip, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp]
    for nm in ("dff_batch_status", "dff_batch_status_"):
        getattr(lib, nm).restype = None
        getattr(lib, nm).argtypes = [dp, dp, ip, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp, ip, ip]
    lib.loglhood_batch.restype = i
    lib.loglhood_batch.argtypes = [ip, dp, dp, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp]
    lib.loglhood_batch_ar.restype = i
    lib.loglhood_batch_ar.argtypes = [ip, dp, dp, ip, ip, ip, dp, dp, ip, dp, dp, ip, dp, dp, dp, dp]
    lib.loglhood_batch_voro.restype = i
    lib.loglhood_batch_voro.argtypes = [ip, dp, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp]
    lib.rtb200_dff_batch_device.restype = i
    lib.rtb200_dff_batch_device.argtypes = [vp, vp, vp, i, i, i, vp, vp, i, vp, vp, vp, vp, vp, i, vp]
    lib.rtb200_dff_grad_device.restype = i
    lib.rtb200_dff_grad_device.argtypes = [vp, vp, vp, i, i, i, vp, vp, i, vp, vp, vp, vp, vp, vp, vp, i, vp]
    lib.dff_batch_grad.restype = i
    lib.dff_batch_grad.argtypes = [dp, dp, ip, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp, dp, dp]
    lib.rtb200_dff_jac_device.restype = i
    lib.rtb200_dff_jac_device.argtypes = [vp, vp, vp, i, i, i, vp, vp, i, vp, vp, vp, vp, vp, vp, i, vp]
    lib.dff_batch_jac.restype = i
    lib.dff_batch_jac.argtypes = [dp, dp, ip, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp, dp]
    lib.rtb200_dff_normal_device.restype = i
    lib.rtb200_dff_normal_device.argtypes = [vp, vp, vp, i, i, i, vp, vp, i, vp, vp, vp, vp, vp, i, vp]
    lib.dff_batch_normal.restype = i
    lib.dff_batch_normal.argtypes = [dp, dp, ip, ip, ip, ip, dp, dp, ip, dp, dp, dp, dp, dp]
    lib.rtb200_mh_step_device.restype = i
    lib.rtb200_mh_step_device.argtypes = [vp, vp, vp, i, i, vp, vp, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp]
    lib.rtb200_mh_step_device_ev.restype = i
    lib.rtb200_mh_step_device_ev.argtypes = [vp, vp, vp, i, i, vp, vp, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp, vp, i]
    lib.rtb200_mh_moves_device_ex.restype = i
    lib.rtb200_mh_moves_device_ex.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp, i]
    lib.rtb200_bd_step_device_ex.restype = i
    lib.rtb200_bd_step_device_ex.argtypes = [vp, vp, vp, i, i, vp, vp, vp, vp, vp, vp, vp, dp, dp, i, i,
                                             vp, vp, vp, i, vp, vp, i]
    lib.rtb200_mh_moves_device.restype = i
    lib.rtb200_mh_moves_device.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp]
    lib.rtb200_bd_step_device.restype = i
    lib.rtb200_bd_step_device.argtypes = [vp, vp, vp, i, i, vp, vp, vp, vp, vp, vp, vp, dp, dp, i, i,
                                          vp, vp, vp, i, vp, vp]
    lib.rtb200_sd_step_device.restype = i
    lib.rtb200_sd_step_device.argtypes = [vp, vp, vp, vp, i, i, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp]
    lib.rtb200_ar_step_device.restype = i
    lib.rtb200_ar_step_device.argtypes = [vp, vp, vp, vp, vp, vp, i, i, vp, vp, vp, vp, vp, dp, vp, vp, vp, i, vp, vp]
    lib.rtb200_set_chain_ar.restype = i
    lib.rtb200_set_chain_ar.argtypes = [vp, vp, d]
    lib.rtb200_mcmc_workspace_bytes.restype = C.c_size_t
    lib.rtb200_mcmc_workspace_bytes.argtypes = [i, i]
    lib.rtb200_mcmc_iterations_device.restype = i
    lib.rtb200_mcmc_iterations_device.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, dp, dp, dp, i, i, i, vp, vp, vp, i,
                                                  C.c_ulonglong, vp, vp, vp, i, vp, vp, dp, vp]
    lib.rtb200_swap_pack_device.restype = i
    lib.rtb200_swap_pack_device.argtypes = [vp, vp, i, vp, vp]
    lib.rtb200_swap_round_device.restype = i
    lib.rtb200_swap_round_device.argtypes = [vp, i, i, i, C.c_ulonglong, C.c_ulonglong, vp, vp, vp, vp]
    lib.rtb200_init.restype = i
    lib.rtb200_init.argtypes = [i]
    lib.rtb200_shutdown.restype = None
    lib.rtb200_last_error.restype = C.c_char_p
    lib.rtb200_device_count.restype = i
    lib.rtb200_set_option.restype = i
    lib.rtb200_set_option.argtypes = [C.c_char_p, d]
    lib.rtb200_get_stat.restype = d
    lib.rtb200_get_stat.argtypes = [C.c_char_p]
    lib.rtb200_fp64_peak_tflops.restype = d
    lib.rtb200_fp64_peak_tflops.argtypes = [i]
    lib.rtb200_selftest_fast_division.restype = d
    lib.rtb200_selftest_fast_division.argtypes = [d, C.c_ulonglong]
    lib.rtb200_shard_range.restype = None
    lib.rtb200_shard_range.argtypes = [C.c_longlong, i, i, C.POINTER(C.c_longlong),
                                       C.POINTER(C.c_longlong)]
    _lib = lib
    return lib


def last_error():
    return load().rtb200_last_error().decode()


def check(rc=0):
    """Raise if the last call reported a failure (status code or recorded error string)."""
    err = last_error()
    if rc != 0 or err:
        raise RayTraceError(err or f"libraytrace_b200 status {rc}")
