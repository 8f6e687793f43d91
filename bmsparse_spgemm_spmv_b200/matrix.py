"""Host-side mirror of the reference's bmSpMatrix class (include/bmSpMatrix.h:20-40) over the C ABI.

Same public names: keys, bmps, offsets, values, num_rows, num_cols, nnz, block_num, generate_coo(),
compare(); constructors map to the reference's three (default / (path, transpose) / adopt arrays) plus
the CSR entry the north star adds.  All arrays live in HBM; properties return torch tensors that alias
the handle's device memory (zero copy) and are only valid while the matrix is alive.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple

import numpy as np
import torch

from . import _lib as L


def _stream_ptr(stream=None):
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


class _DevArray:
    """__cuda_array_interface__ shim so torch can alias handle-owned device memory."""

    def __init__(self, ptr, n, typestr, owner):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr or 0), False),
                                         "version": 2}
        self._owner = owner


def _alias(ptr, n, typestr, torch_dtype, owner):
    if n == 0 or not ptr:
        return torch.empty(0, dtype=torch_dtype, device="cuda")
    return torch.as_tensor(_DevArray(ptr, n, typestr, owner), device="cuda")


class bmSpMatrix:
    def __init__(self, path: str | None = None, transpose: bool = False, dtype=torch.float16, _handle=None, merge_duplicates: bool = False):
        self._h = C.c_void_p(_handle) if _handle else C.c_void_p()
        if path is not None:
            L.check(L.lib().bmsp_create_from_mtx_ex(path.encode(), int(transpose), _dt(dtype), int(bool(merge_duplicates)), _stream_ptr(),
                                                    C.byref(self._h)))

    # ---- constructors -------------------------------------------------------------------------
    @classmethod
    def from_csr(cls, num_rows, num_cols, row_ptr, col_idx, vals, transpose=False, dtype=torch.float16, stream=None):
        """CSR (torch CUDA tensors, numpy arrays or anything array-like on the host) -> bmSparse."""
        m = cls()
        rp = _array(row_ptr, np.int32)
        ci = _array(col_idx, np.int32, mem=rp.mem)
        v = _array(vals, values=True, mem=rp.mem)
        L.check(L.lib().bmsp_create_from_csr(int(num_rows), int(num_cols), C.c_int64(ci.n), rp.ptr, ci.ptr, v.ptr, v.dt, rp.mem,
                                             int(transpose), _dt(dtype), _stream_ptr(stream), C.byref(m._h)))
        if rp.mem == L.DEVICE:
            (stream if stream is not None else torch.cuda.current_stream()).synchronize()      # rp / ci / v temporaries die here
        return m

    @classmethod
    def from_coo(cls, num_rows, num_cols, rows, cols, vals, transpose=False, dtype=torch.float16, merge_duplicates=False):
        m = cls()
        r = np.ascontiguousarray(rows, np.int32); c = np.ascontiguousarray(cols, np.int32)
        v = np.ascontiguousarray(vals, np.float64)
        L.check(L.lib().bmsp_create_from_coo_ex(int(num_rows), int(num_cols), C.c_int64(r.size), r.ctypes.data_as(C.c_void_p),
                                                c.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p), int(transpose),
                                                _dt(dtype), int(bool(merge_duplicates)), _stream_ptr(), C.byref(m._h)))
        return m

    @classmethod
    def from_arrays(cls, num_rows, num_cols, block_num, keys, bmps, offsets, values, transpose=False):
        """bmSpMatrix(num_rows, num_cols, block_num, keys, bmps, offsets, values) -- src/bmSpMatrix.cu:30-43."""
        m = cls()
        assert not isinstance(keys, torch.Tensor) or keys.is_cuda, "from_arrays: tensors must be CUDA tensors"
        k = _array(keys, np.uint64)
        b, o = (_array(a, np.uint64, mem=k.mem) for a in (bmps, offsets))
        v = _array(values, values=k.mem == L.HOST, mem=k.mem)        # device values are adopted as they are: fp16 or fp32 only
        L.check(L.lib().bmsp_create_from_arrays(int(num_rows), int(num_cols), C.c_int64(block_num), C.c_int64(v.n), k.ptr, b.ptr,
                                                o.ptr, C.c_int64(o.n), v.ptr, v.dt, k.mem, int(transpose), _stream_ptr(), C.byref(m._h)))
        torch.cuda.current_stream().synchronize()
        return m

    # ---- reference-named fields ---------------------------------------------------------------
    def _view(self) -> L.View:
        v = L.View()
        L.check(L.lib().bmsp_get(self._h, C.byref(v)))
        return v

    num_rows = property(lambda s: s._view().num_rows)
    num_cols = property(lambda s: s._view().num_cols)
    nnz = property(lambda s: s._view().nnz)
    block_num = property(lambda s: s._view().block_num)
    transposed = property(lambda s: bool(s._view().transposed))
    num_block_rows = property(lambda s: s._view().num_block_rows)

    @property
    def dtype(self):
        return torch.float16 if self._view().dtype == L.F16 else torch.float32

    # torch has no uint64 arithmetic; the 64-bit words are exposed as int64 (same bits)
    @property
    def keys(self):
        v = self._view(); return _alias(v.keys, v.block_num, "<i8", torch.int64, self)

    @property
    def bmps(self):
        v = self._view(); return _alias(v.bmps, v.block_num, "<i8", torch.int64, self)

    @property
    def offsets(self):
        v = self._view(); return _alias(v.offsets, v.offsets_len, "<i8", torch.int64, self)

    @property
    def values(self):
        """The values in compact order, aliasing the handle's memory.  After writing through this alias, call set_values(None): the
        library keeps copies of a SpGEMM B operand's values, and only set_values refreshes them."""
        v = self._view()
        return _alias(v.values, v.nnz, "<f2" if v.dtype == L.F16 else "<f4", self.dtype, self)

    # ---- new values, same structure -----------------------------------------------------------
    def set_values(self, values, stream=None):
        """Overwrite the values in compact order (the order of .values): a torch tensor (CUDA: asynchronous on the stream; CPU:
        synchronous) or a numpy array, fp16 or fp32 (anything else is taken as fp32), converted to the matrix's dtype.  None: the
        values were written in place through .values; refresh the library's copies of them."""
        lib = L.lib()
        if values is None:
            L.check(lib.bmsp_set_values(self._h, None, L.F32, L.DEVICE, _stream_ptr(stream)))
            return
        v = _array(values, values=True)
        if v.n != self.nnz:
            raise ValueError(f"set_values: {v.n} values for a matrix with {self.nnz}")
        L.check(lib.bmsp_set_values(self._h, v.ptr, v.dt, v.mem, _stream_ptr(stream)))
        if v.mem == L.DEVICE and v.keep is not values and stream is not None:
            v.keep.record_stream(stream)        # the temporary outlives this call on `stream`

    def set_values_csr(self, row_ptr, col_idx, vals, stream=None):
        """New values as a CSR with exactly this matrix's pattern (the arrays from_csr took, for either orientation): CUDA tensors
        or host arrays, as from_csr takes them.  A different pattern raises BmspError (INVALID) and leaves the values unchanged."""
        lib = L.lib()
        v = self._view()
        rp = _array(row_ptr, np.int32)
        ci = _array(col_idx, np.int32, mem=rp.mem)
        x = _array(vals, values=True, mem=rp.mem)
        if rp.n != v.num_rows + 1 or ci.n != x.n:
            raise ValueError("set_values_csr: row_ptr needs num_rows + 1 entries, col_idx and vals one per value")
        if ci.n != v.nnz:      # the library reads nnz entries of col_idx and vals
            raise L.BmspError(1, f"set_values_csr: the CSR has {ci.n} entries, the matrix {v.nnz} values")
        L.check(lib.bmsp_set_values_csr(self._h, rp.ptr, ci.ptr, x.ptr, x.dt, rp.mem, _stream_ptr(stream)))
        if rp.mem == L.DEVICE:
            (stream if stream is not None else torch.cuda.current_stream()).synchronize()      # rp / ci / x temporaries die here

    @property
    def block_row_ptr(self):
        v = self._view(); return _alias(v.block_row_ptr, v.num_block_rows + 1, "<i4", torch.int32, self)

    @property
    def block_col(self):
        v = self._view(); return _alias(v.block_col, v.block_num, "<i4", torch.int32, self)

    # ---- host copies / utilities ----------------------------------------------------------------
    def download(self):
        """(keys, bmps, offsets, values) as numpy arrays: uint64 x3 + float16/float32."""
        v = self._view()
        k = np.empty(v.block_num, np.uint64); b = np.empty(v.block_num, np.uint64); o = np.empty(v.offsets_len, np.uint64)
        vals = np.empty(v.nnz, np.float16 if v.dtype == L.F16 else np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        L.check(L.lib().bmsp_download(self._h, p(k), p(b), p(o), p(vals)))
        return k, b, o, vals

    def generate_coo(self):
        """bmSparse -> COO (rows, cols, fp32 values); src/bmSpMatrix.cu:320-363."""
        n = self.nnz
        r = np.empty(n, np.int32); c = np.empty(n, np.int32); v = np.empty(n, np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        L.check(L.lib().bmsp_to_coo(self._h, p(r), p(c), p(v)))
        return r, c, v

    def compare(self, rows, cols, vals):
        """Unlike src/bmSpMatrix.cu:381-432 this reports: (only_in_self, only_in_other, mean_rel, max_rel)."""
        r = np.ascontiguousarray(rows, np.int32); c = np.ascontiguousarray(cols, np.int32); v = np.ascontiguousarray(vals, np.float32)
        a = C.c_int64(); b = C.c_int64(); mean = C.c_double(); mx = C.c_double()
        p = lambda x: x.ctypes.data_as(C.c_void_p)
        L.check(L.lib().bmsp_compare(self._h, C.c_int64(r.size), p(r), p(c), p(v), C.byref(a), C.byref(b), C.byref(mean), C.byref(mx)))
        return a.value, b.value, mean.value, mx.value

    def to_csr(self):
        """bmSparse -> CSR on the device: (row_ptr int32[rows+1], col_idx int32[nnz], vals fp32[nnz]) as CUDA tensors."""
        v = self._view()
        rp = torch.empty(v.num_rows + 1, dtype=torch.int32, device="cuda"); ci = torch.empty(max(v.nnz, 1), dtype=torch.int32, device="cuda")
        vals = torch.empty(max(v.nnz, 1), dtype=torch.float32, device="cuda")
        L.check(L.lib().bmsp_to_csr(self._h, C.c_void_p(rp.data_ptr()), C.c_void_p(ci.data_ptr()), C.c_void_p(vals.data_ptr()), L.DEVICE, _stream_ptr()))
        return rp, ci[:v.nnz], vals[:v.nnz]

    def compare_csr(self, row_ptr, col_idx, vals):
        """device-side compare against a CSR held in CUDA tensors: (only_in_self, only_in_other, mean_rel, max_rel)"""
        rp = row_ptr.to(torch.int32).contiguous(); ci = col_idx.to(torch.int32).contiguous(); v = vals.to(torch.float32).contiguous()
        a = C.c_int64(); b = C.c_int64(); mean = C.c_double(); mx = C.c_double()
        L.check(L.lib().bmsp_compare_csr(self._h, C.c_void_p(rp.data_ptr()), C.c_void_p(ci.data_ptr()), C.c_void_p(v.data_ptr()), L.DEVICE,
                                         _stream_ptr(), C.byref(a), C.byref(b), C.byref(mean), C.byref(mx)))
        return a.value, b.value, mean.value, mx.value

    def block_transpose(self, dtype=None):
        out = bmSpMatrix()
        L.check(L.lib().bmsp_block_transpose(self._h, _dt(dtype or self.dtype), _stream_ptr(), C.byref(out._h)))
        return out

    def matrix_transpose(self, dtype=None, transpose=False, stream=None) -> "bmSpMatrix":
        """The transpose A^T as a new matrix (num_rows and num_cols swapped).  Unlike block_transpose, which stores the same matrix A
        in the other form, this returns a different matrix.  transpose: as in from_csr, store A^T in transposed-operand form, ready
        to be the B of a product (A.matrix_transpose(transpose=True) is the B of A * A^T).  dtype None keeps this matrix's dtype.
        This matrix may be in either form.  Enqueued on the stream (default: the current one) without a host synchronisation; the
        result does not depend on this matrix afterwards."""
        out = bmSpMatrix()
        L.check(L.lib().bmsp_matrix_transpose(self._h, _dt(dtype or self.dtype), int(bool(transpose)), _stream_ptr(stream), C.byref(out._h)))
        return out

    def slice_block_rows(self, r0, r1, rebase=False):
        out = bmSpMatrix()
        L.check(L.lib().bmsp_slice_block_rows(self._h, int(r0), int(r1), int(rebase), _stream_ptr(), C.byref(out._h)))
        return out

    def partition_block_rows(self, nparts, Bt=None):
        bounds = np.empty(nparts + 1, np.int32)
        L.check(L.lib().bmsp_partition_block_rows(self._h, Bt._h if Bt is not None else None, int(nparts), int(Bt is not None),
                                                  bounds.ctypes.data_as(C.c_void_p), _stream_ptr()))
        return bounds

    def spmv_bytes(self, x_dtype=torch.float32) -> int:
        n = C.c_int64()
        L.check(L.lib().bmsp_spmv_bytes(self._h, _dt(x_dtype), C.byref(n)))
        return n.value

    def __del__(self):
        try:
            if self._h:
                L.lib().bmsp_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


_Array = namedtuple("_Array", "ptr n dt mem keep")


def _array(a, dtype=None, values=False, mem=None) -> _Array:
    """One array argument of a C call: its pointer, element count, dtype code (_dt; None for index arrays), mem, and the object
    that must stay alive while the call's work runs.  A CUDA tensor is passed where it is (L.DEVICE); a CPU tensor, a numpy array or
    anything array-like becomes a contiguous host array (L.HOST).  dtype: the element type of an index array (host arrays are
    converted to it; CUDA tensors to int32 only -- torch has no uint64 arithmetic, so 64-bit words are taken as they are).
    values: fp16 and fp32 are kept, anything else becomes fp32.  mem: the mem of the call's other arrays, which this one must share."""
    if isinstance(a, torch.Tensor) and a.is_cuda:
        x = (a.to(torch.int32) if dtype == np.int32 else a).contiguous()
        if values and x.dtype not in (torch.float16, torch.float32):
            x = x.to(torch.float32)
        ptr, n, where = C.c_void_p(x.data_ptr()), x.numel(), L.DEVICE
    else:
        x = np.ascontiguousarray(np.asarray(a, dtype).reshape(-1))
        if values and x.dtype not in (np.float16, np.float32):
            x = x.astype(np.float32)
        ptr, n, where = x.ctypes.data_as(C.c_void_p), x.size, L.HOST
    if mem is not None and where != mem:
        raise ValueError("the arrays of one call must all be CUDA tensors or all be host arrays")
    return _Array(ptr, n, _dt(x.dtype) if dtype is None else None, where, x)


def _dt(dtype) -> int:
    if dtype in (torch.float16, np.float16):
        return L.F16
    if dtype in (torch.float32, np.float32):
        return L.F32
    raise TypeError(f"unsupported dtype {dtype}")
