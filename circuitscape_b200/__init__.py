"""circuitscape_b200 -- B200-native (sm_100a) drop-in for Circuitscape.jl's inner
Laplacian-solve loop (pairwise + advanced mode).  See DESIGN.md / INTEGRATION.md.

Layout: csrc/ (CUDA kernels + C ABI -> lib/libcsb200.so), solver.py (the
reference's Solver plug-in surface), core.py (pairwise / advanced drivers),
graph.py (problem assembly just before the path), dist.py (pair sharding over
GPUs with torch.distributed / NCCL).
"""
from .solver import (CUDAB200, CUDASolver, B200Factor, SolverResidualError,  # noqa: F401
                     construct_cholesky_factor, solve_linear_system, multiple_solve)
from .core import (GraphProblem, AdvancedProblem, Flags, OutputFlags, get_solver,  # noqa: F401
                   single_ground_all_pairs, solve, advanced_kernel, multiple_solver, compute_3col,
                   RasterData, onetoall_kernel, resolve_conflicts, compute_omniscape_current,
                   all_to_one_batched, raster_pairwise)
from ._lib import B200Unavailable, B200Error, LIB_PATH, EXPORTED_SYMBOLS  # noqa: F401
