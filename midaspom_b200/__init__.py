"""midaspom_b200 -- B200-native SPOM likelihood / MCMC engine behind a C ABI.

The product is ``lib/libmidaspom_cuda.so`` (hand-written sm_100a CUDA, built in-tree by
``midaspom_b200.build``) whose entry points are declared in ``include/libmidaspom_cuda.h``.
``Engine`` is a thin ctypes mirror of that ABI for tests and benchmarks; there is no CPU fallback.
"""
from .engine import (Engine, MpConfig, MpParams, MpSamplerConfig, MpError, load_library, GEOM_LINEAR, GEOM_COORDS,
                     GEOM_DENSE, FP32, FP64, NDRAW, NLSIG, NPART, KERNEL_CATEGORIES, ABI_SYMBOLS, PPC_STATS, exact_posterior, exact_variant)
from .waic import waic, compare_waic
from .ppc import ppc_check
from .capacity import persistence
from .sources import colonisation_sources

__all__ = ["Engine", "MpConfig", "MpParams", "MpSamplerConfig", "MpError", "load_library", "GEOM_LINEAR",
           "GEOM_COORDS", "GEOM_DENSE", "FP32", "FP64", "NDRAW", "NLSIG", "NPART", "KERNEL_CATEGORIES", "ABI_SYMBOLS", "exact_posterior", "exact_variant",
           "waic", "compare_waic", "PPC_STATS", "ppc_check", "persistence", "colonisation_sources"]
