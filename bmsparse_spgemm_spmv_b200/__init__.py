"""bmsparse_spgemm_spmv_b200 -- B200-native bmSparse SpMV / SpGEMM hot path.

Product code: csrc/ (hand-written sm_100a CUDA behind the C ABI of include/bmsparse_b200.h) and this thin
host mirror of the reference's bmSpMatrix / bmSparse_SpMV / bmSparse_mult interface.  Nothing here imports
oracle/: the CPU oracle is test infrastructure.
"""
from ._lib import BmspError, LIB_PATH, SYMBOLS, lib  # noqa: F401
from .matrix import bmSpMatrix  # noqa: F401
from .ops import SpGEMMPlan, bmSparse_SpMV, bmSparse_SpMV_host, bmSparse_add, bmSparse_mult, bmSparse_mult_plan  # noqa: F401
from . import generators  # noqa: F401
