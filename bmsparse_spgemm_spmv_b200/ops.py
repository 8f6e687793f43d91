"""The two operators of the reference, same names and argument order, over the C ABI.

  bmSparse_SpMV(A, v, u, batched)                    src/bmSparse_SPMV.cu:191-230
  bmSparse_mult(A, B, C, mode, VERBOSE, tc_version)  src/bmSparse_SPGEMM.cu:827-1223

and bmSparse_mult_plan, which the reference does not have: the same product, kept so that C's values can be recomputed after the
operands' values change; and bmSparse_add, C = alpha*A + beta*B, which the reference does not have either.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .matrix import bmSpMatrix, _dt, _stream_ptr


def bmSparse_SpMV(A: bmSpMatrix, v: torch.Tensor, u: torch.Tensor | None = None, batched: bool = False, stream=None):
    """u = A v.  v: CUDA fp32 or fp16 [num_cols]; u: CUDA fp32 [num_rows] (allocated when None).
    `batched` selected the reference's second kernel (broken as shipped, SURVEY Appendix B); accepted, ignored."""
    view = A._view()
    if not v.is_cuda or v.numel() != view.num_cols:
        raise ValueError("v must be a CUDA tensor with num_cols elements")
    v = v.contiguous()
    if u is None:
        u = torch.empty(view.num_rows, dtype=torch.float32, device=v.device)
    if not u.is_cuda or u.dtype != torch.float32 or u.numel() != view.num_rows or not u.is_contiguous():
        raise ValueError("u must be a contiguous CUDA fp32 tensor with num_rows elements")
    L.check(L.lib().bmsp_spmv(A._h, C.c_void_p(v.data_ptr()), _dt(v.dtype), C.c_void_p(u.data_ptr()), _stream_ptr(stream)))
    return u


def bmSparse_SpMV_host(A: bmSpMatrix, v: torch.Tensor, u: torch.Tensor | None = None, stream=None):
    """u = A v with v and u in HOST memory (pin them for full PCIe speed): what the reference's driver does by hand
    around the operator (cudaMemcpy v, bmSparse_SpMV, cudaMemcpy u -- SPMV.cu:276-309), as one pipelined call.
    u is complete after the stream (default: the current one) is synchronised."""
    view = A._view()
    if v.is_cuda or v.numel() != view.num_cols or not v.is_contiguous():
        raise ValueError("v must be a contiguous host tensor with num_cols elements")
    if u is None:
        u = torch.empty(view.num_rows, dtype=torch.float32).pin_memory()
    if u.is_cuda or u.dtype != torch.float32 or u.numel() != view.num_rows or not u.is_contiguous():
        raise ValueError("u must be a contiguous host fp32 tensor with num_rows elements")
    L.check(L.lib().bmsp_spmv_host(A._h, C.c_void_p(v.data_ptr()), _dt(v.dtype), C.c_void_p(u.data_ptr()), _stream_ptr(stream)))
    return u


def _spgemm_opts(mode, tc_version, VERBOSE, numeric_path, brow_range):
    return L.SpgemmOpts(int(mode), int(tc_version), int(bool(VERBOSE)), int(numeric_path),
                        brow_range[0] if brow_range is not None else 0, brow_range[1] if brow_range is not None else 0,
                        int(brow_range is not None))


def bmSparse_mult(A: bmSpMatrix, B: bmSpMatrix, C_out: bmSpMatrix | None = None, mode=0, VERBOSE: bool = False,
                  tc_version: int = 5, numeric_path: int = -1, brow_range=None, stream=None):
    """C = A * B with B in transposed-operand form (built with transpose=True, SPGEMM.cu:1262).
    Returns (C, info).  `mode` / `tc_version` are accepted for drop-in compatibility and ignored."""
    opts = _spgemm_opts(mode, tc_version, VERBOSE, numeric_path, brow_range)
    info = L.SpgemmInfo()
    out = C_out if C_out is not None else bmSpMatrix()
    if out._h:
        L.lib().bmsp_destroy(out._h)
        out._h = C.c_void_p()
    L.check(L.lib().bmsp_spgemm(A._h, B._h, C.byref(opts), _stream_ptr(stream), C.byref(out._h), C.byref(info)))
    return out, info


class SpGEMMPlan:
    """C = A * B kept for reuse: C's structure and what its numeric pass reads.  After A's or B's values change
    (bmSpMatrix.set_values / set_values_csr), numeric() recomputes C's values alone.  Holds A, B and C, so the plan is always
    released before them.  Its calls must be ordered on one stream at a time."""

    def __init__(self, h, A, B, C, info):
        self._h, self.A, self.B, self.C, self.info = h, A, B, C, info

    def numeric(self, stream=None):
        """Recompute C's values from A's and B's current values: enqueued on the stream, no host synchronisation and no
        allocation, so it can be captured into a CUDA graph."""
        if not self._h:
            raise ValueError("SpGEMMPlan is closed")
        L.check(L.lib().bmsp_spgemm_numeric(self._h, _stream_ptr(stream)))
        return self.C

    @property
    def nbytes(self) -> int:
        """device memory the plan retains besides C and the operands"""
        n = C.c_int64()
        L.check(L.lib().bmsp_spgemm_plan_bytes(self._h, C.byref(n)))
        return n.value

    def close(self):
        if self._h:
            L.lib().bmsp_spgemm_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bmSparse_mult_plan(A: bmSpMatrix, B: bmSpMatrix, VERBOSE: bool = False, numeric_path: int = -1, brow_range=None, stream=None):
    """bmSparse_mult(A, B, ...) that keeps its plan: returns a SpGEMMPlan whose .C and .info are what bmSparse_mult returns."""
    opts = _spgemm_opts(0, 5, VERBOSE, numeric_path, brow_range)
    info = L.SpgemmInfo()
    out = bmSpMatrix()
    h = C.c_void_p()
    L.check(L.lib().bmsp_spgemm_plan_create(A._h, B._h, C.byref(opts), _stream_ptr(stream), C.byref(h), C.byref(out._h), C.byref(info)))
    return SpGEMMPlan(h, A, B, out, info)


def bmSparse_add(A: bmSpMatrix, B: bmSpMatrix, alpha: float = 1.0, beta: float = 1.0, dtype=None, stream=None) -> bmSpMatrix:
    """C = alpha*A + beta*B as a new matrix (bmsp_add).  A and B have the same shape and storage form (block_transpose converts
    one); C is stored in that form.  C's pattern is the union of A's and B's: entries that cancel are kept.  Each value is
    fl(fl(alpha*a) + fl(beta*b)) in fp32, a missing entry counting as 0, rounded once to dtype.  dtype None: fp32 if either
    operand holds fp32 values, else fp16.  Synchronises the stream (default: the current one) once; C does not depend on A or B
    afterwards.  Shape and form errors raise BmspError with the library's code."""
    if dtype is None:
        dtype = torch.float32 if torch.float32 in (A.dtype, B.dtype) else torch.float16
    out = bmSpMatrix()
    L.check(L.lib().bmsp_add(C.c_float(alpha), A._h, C.c_float(beta), B._h, _dt(dtype), _stream_ptr(stream), C.byref(out._h)))
    return out
