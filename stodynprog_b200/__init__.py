"""stodynprog_b200 - B200-native Bellman backward-induction engine.

Drop-in for the Bellman sweep of pierre-haessig/stodynprog: the same
`SysDescription` / `DPSolver` API (reference stodynprog/__init__.py:15), with the
state x control x perturbation loop nest running in hand-written sm_100a CUDA
kernels behind a C ABI (include/sdp_b200.h).

    from stodynprog_b200 import SysDescription, DPSolver

Importing the package needs neither a GPU nor the built extension (grids and
problem descriptions are host objects); running a solver does, and fails
loudly without them - there is no CPU fallback.
"""
from .sysdesc import SysDescription
from .solver import DPSolver
from .risk import MeanCVaR
from .interp import (MlinInterpolator, MultilinearInterpolator, multilinear_interpolation,
                     mlinspace)

__version__ = "0.1.0"
__all__ = ["SysDescription", "DPSolver", "MeanCVaR", "MlinInterpolator", "MultilinearInterpolator",
           "multilinear_interpolation", "mlinspace"]
