"""raytracerfortran_b200 -- B200-native drop-in for the `dff` + `loglhood` hot path of
AntonBiryukovUofC/RayTracerFortran.

  raymod      host-buffer entry points mirroring the reference interface (dff, TraceRays,
              dff_batch, loglhood_batch) over the C ABI of libraytrace_b200.so
  device      the same path on CUDA tensors already resident in HBM (no copies)
  grad        torch.autograd functions: travel times and LOGLHOOD_RT with gradients with respect
              to the layered model, the sources, the observations and sigma; the per-ray Jacobian and
              the per-model Gauss-Newton normal equations
  tempering   model-axis sharding across ranks and the parallel-tempering swap step
              (one small all-gather of (logL, beta) per swap round)
  workloads   seeded synthetic models / sources of the benchmark shapes
  build       nvcc build of the in-tree shared library (sm_100a only)
"""
from ._lib import EXPORTS, LIB_PATH, RayTraceError  # noqa: F401
from .raymod import (TraceRays, dff, dff7, dff_batch, dff_batch_grad, dff_batch_jac, dff_batch_normal,  # noqa: F401
                     fp64_peak_tflops, get_stat, loglhood_batch, loglhood_batch_ar, loglhood_batch_voro, selftest_fast_division, set_option, shard_range)

__all__ = ["dff", "dff7", "TraceRays", "dff_batch", "dff_batch_grad", "dff_batch_jac", "dff_batch_normal", "loglhood_batch", "loglhood_batch_ar", "loglhood_batch_voro", "set_option", "get_stat",
           "fp64_peak_tflops", "shard_range", "selftest_fast_division", "RayTraceError", "EXPORTS", "LIB_PATH"]
