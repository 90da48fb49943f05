"""sparsh_amg_b200 — B200-native AMG solve phase behind the SParSH-AMG API.

Layout (only what the hot path needs — SURVEY.md §8):
  csrc/     hand-written sm_100a CUDA kernels + the C-ABI (include/sparsh_b200.h) -> lib/libsparsh_b200.so
  host/     C++ mirror of the reference's host interface (sp_matrix_mg, AMG_solver setup, AMG_Solver_* / Solver_PCG_*
            entry points) on top of the C-ABI -> lib/libsparsh_amg.so
  capi.py   ctypes binding of the C-ABI          device.py  thin object wrappers
  host.py   ctypes binding of the host library   (hierarchy setup, synthetic matrices, reference-named solvers)

There is no CPU fallback: importing is cheap, but every compute call needs lib/libsparsh_b200.so and a GPU.
"""
from . import capi  # noqa: F401
from .capi import SparshError  # noqa: F401
from .device import (DeviceHierarchy, DeviceMatrix, DeviceVector, PendingSolve, axpby, axpbypcz, axpy, dot,  # noqa: F401
                     galerkin_rap, init, launch_count, nrm2, set_stream, sync)
