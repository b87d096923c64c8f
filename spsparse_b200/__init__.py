"""spsparse_b200 -- B200-native (sm_100a) implementation of spsparse's hot path: COO consolidate()
and the sparse*sparse multiply(), as hand-written CUDA kernels behind a C ABI
(include/spsparse_b200.h).  This package is the Python host mirror used by tests and bench.py; the
drop-in for C++ callers is the header layer in include/spsparse/.  There is no CPU fallback:
importing the device API without the built CUDA library raises."""
from .coo import (ADD, COL_MAJOR, LEAVE_ALONE, REPLACE, ROW_MAJOR, ConsolidatePlan, Context, CooArray, MultiplyPlan,  # noqa: F401
                  consolidate, copy,
                  gen_banded, gen_dup_coo, gen_regrid, gen_rmat, gen_vector, multiply, multiply_prepared,
                  to_dense, to_sparse, transpose)
from ._lib import SpbError, load  # noqa: F401
