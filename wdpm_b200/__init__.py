"""wdpm_b200 - B200-native implementation of WDPM's water-redistribution path.

The product is the CUDA library (csrc/ -> libwdpm_b200.so, C ABI in
include/wdpm_b200.h) and the drop-in command-line host (host/). The Python
modules here are a thin ctypes mirror of that ABI plus the module driver used by
the tests and the benchmark.
"""
from .solver import (ADD, DRAIN, F32, F64, MAX_OUTLETS, KERNEL_AUTO, KERNEL_COLOUR, KERNEL_FUSED, KERNEL_RESIDENT, SCHED_OPENCL, SCHED_SERIAL, SUBTRACT,
                     BlockResult, Solver, WdpmError, library_path, load_library)

__all__ = ["ADD", "SUBTRACT", "DRAIN", "F32", "F64", "KERNEL_AUTO", "KERNEL_COLOUR", "KERNEL_FUSED", "KERNEL_RESIDENT", "SCHED_OPENCL",
           "SCHED_SERIAL", "MAX_OUTLETS", "BlockResult",
           "Solver", "WdpmError", "library_path", "load_library"]
