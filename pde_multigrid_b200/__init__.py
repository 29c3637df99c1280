"""pde_multigrid_b200 -- B200-native geometric multigrid behind the entry points of MisterPup/PDE-MultiGrid.

The product is libmg_b200.so (C host drivers + hand-written sm_100a CUDA kernels, C ABI in
include/mg_b200.h).  This package only loads it (ctypes) and mirrors the reference's class interface
for tests and benchmarks.  There is no CPU or PyTorch compute path.
"""
from ._lib import (MG_CORRECTED, MG_F32, MG_F64, MG_FIELD_F, MG_FIELD_V, MG_REF_COMPAT, MG_SMOOTHER_AUTO,
                   MG_SMOOTHER_COLOUR, MG_SMOOTHER_FUSED, MG_SMOOTHER_JACOBI, MG_SMOOTHER_TMA, MG_SMOOTHER_PIPE,
                   MG_ARITH_EXACT, MG_ARITH_FAST, MGError, lib)
from .multigrid import MultiGrid1D, MultiGrid2D, MultiGrid3D, MultiGrid3DBox, SolveResult

__all__ = ["MultiGrid1D", "MultiGrid2D", "MultiGrid3D", "MultiGrid3DBox", "SolveResult", "MGError", "lib", "MG_F32", "MG_F64", "MG_REF_COMPAT",
           "MG_CORRECTED", "MG_FIELD_V", "MG_FIELD_F", "MG_SMOOTHER_AUTO", "MG_SMOOTHER_COLOUR", "MG_SMOOTHER_FUSED",
           "MG_SMOOTHER_JACOBI", "MG_SMOOTHER_TMA", "MG_SMOOTHER_PIPE", "MG_ARITH_EXACT", "MG_ARITH_FAST"]
