"""sdplrplus.jl_b200 -- B200-native hot path of SDPLRPlus.jl behind its own seam.

Layout
  csrc/            hand-written sm_100a CUDA kernels + the C ABI (include/sdplrp_b200.h)
  _lib.py          ctypes binding of libsdplrp_b200.so (what the Julia ccall shim does)
  types.py         SymLowRankMatrix, SparseMatrixCOO, Diagonal, ConstraintBatch, SDPData
  problems.py      MaxCut / Lovasz theta / min-bisection / cut-norm / mu-conductance generators
  solver.py        BurerMonteiroConfig, B200Engine, linesearch_, _sdplr, sdplr (Python loop or the native sdplrp_solve),
                   hyperplane_rounding / sweep_rounding (best-of-K +-1 cuts from the solution, on the device)
  formats.py       SDPA / SDPLR-1.03 writers and readers, Gset and MATLAB v7.3 graph readers (exps/data_utils.jl)

The directory name contains a dot, so it is imported through the tiny
`sdplrplus` shim at the repo root: `import sdplrplus.jl_b200 as sp`.
"""
from . import _lib
from ._lib import Handle, SdplrpError, tridiag_mineig
from .types import (ConstraintBatch, Diagonal, SDPData, SparseMatrixCOO, SymLowRankMatrix, assemble_sparse,
                    b_vector, C_matrix, frobenius_norm)
from .solver import (B200Engine, BurerMonteiroConfig, GenericExecutionStats, Solver, SolverStats, _sdplr, barvinok_pataki,
                     hyperplane_rounding, linesearch_, linesearch_armijo_, pick_alpha, sdplr, sweep_rounding)
from . import problems
from . import formats

__all__ = ["Handle", "SdplrpError", "tridiag_mineig", "ConstraintBatch", "Diagonal", "SDPData", "SparseMatrixCOO",
           "SymLowRankMatrix", "assemble_sparse", "b_vector", "C_matrix", "frobenius_norm", "B200Engine",
           "BurerMonteiroConfig", "GenericExecutionStats", "Solver", "SolverStats", "_sdplr", "barvinok_pataki", "hyperplane_rounding", "linesearch_", "linesearch_armijo_",
           "pick_alpha", "sdplr", "sweep_rounding", "problems", "formats"]
