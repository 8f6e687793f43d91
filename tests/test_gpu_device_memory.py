"""GPU: the library's device memory comes back.

The library allocates from the device's default memory pool only (stream-ordered), which torch's default allocator does not use, so
the pool's own counters account for the library alone.  Every case runs an entry point on a small input and destroys every handle
and plan it made; used memory must then be where it was before the case.  Validation failures must leave it there too.

Each case prints its peak above that baseline (CU_MEMPOOL_ATTR_USED_MEM_HIGH after a reset) as `POOL_PEAK <case> <bytes>`.  The
ABI is stable, so running this file against another build (BMSP_LIB_PATH) and comparing the printed peaks shows whether a change
moved any allocation or free."""
import ctypes
import gc
import inspect
import os

import numpy as np
import pytest
import torch

from tests.test_gpu_spgemm_paths import _strided_b
from tests.test_gpu_spmv_palette import _patterned_blocks_csr
from tests.util import random_csr

pytestmark = pytest.mark.gpu

USED_MEM_CURRENT, USED_MEM_HIGH = 7, 8      # CUmemPool_attribute


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


class _Pool:
    """the default memory pool of the current device, through the driver API"""
    def __init__(self):
        self.cu = ctypes.CDLL("libcuda.so.1")
        dev = ctypes.c_int()
        assert self.cu.cuDeviceGet(ctypes.byref(dev), torch.cuda.current_device()) == 0
        self.pool = ctypes.c_void_p()
        assert self.cu.cuDeviceGetDefaultMemPool(ctypes.byref(self.pool), dev) == 0

    def get(self, attr):
        v = ctypes.c_uint64()
        assert self.cu.cuMemPoolGetAttribute(self.pool, attr, ctypes.byref(v)) == 0
        return v.value

    def reset_high(self):
        zero = ctypes.c_uint64(0)
        assert self.cu.cuMemPoolSetAttribute(self.pool, USED_MEM_HIGH, ctypes.byref(zero)) == 0


@pytest.fixture(scope="module")
def pool(B):
    if "cudaMallocAsync" in os.environ.get("PYTORCH_CUDA_ALLOC_CONF", ""):
        pytest.skip("torch allocates from the same pool")
    torch.cuda.init()
    return _Pool()


def _run(pool, name, fn):
    """fn() with every object it makes gone afterwards; used memory back at its baseline; prints the peak above it"""
    gc.collect(); torch.cuda.synchronize()
    base = pool.get(USED_MEM_CURRENT)
    pool.reset_high()
    fn()
    gc.collect(); torch.cuda.synchronize()
    print(f"POOL_PEAK {name} {pool.get(USED_MEM_HIGH) - base}")
    assert pool.get(USED_MEM_CURRENT) == base, f"{name}: {pool.get(USED_MEM_CURRENT) - base} bytes not freed"


def _csr(B):
    nr, nc, rp, ci, v = B.generators.poisson5pt(40, 36)
    return nr, nc, rp, ci, v


def _spmv(B, M, nc):
    y = B.bmSparse_SpMV(M, torch.from_numpy(B.generators.x_vector(nc)).cuda())
    torch.cuda.synchronize()
    return y


# ---- conversions and utilities --------------------------------------------------------------------------------------
def _from_csr_host(B):
    nr, nc, rp, ci, v = _csr(B)
    B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=torch.float32)


def _from_csr_device(B):
    nr, nc, rp, ci, v = _csr(B)
    d = lambda a: torch.from_numpy(a).cuda()
    B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v), transpose=True)


def _from_coo(B):
    r, c = np.array([0, 5, 5, 17, 30]), np.array([3, 1, 20, 17, 2])
    B.bmSpMatrix.from_coo(31, 21, r, c, np.arange(5.0) + 1)


def _from_mtx(B, tmp_path):
    p = tmp_path / "m.mtx"
    p.write_text("%%MatrixMarket matrix coordinate real symmetric\n20 20 4\n1 1 2.0\n5 2 -1.0\n17 9 0.5\n20 20 3.0\n")
    B.bmSpMatrix(str(p))


def _from_arrays(B):
    nr, nc, rp, ci, v = _csr(B)
    k, b, o, vals = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v).download()
    B.bmSpMatrix.from_arrays(nr, nc, k.size, k, b, o, vals)


def _transpose_slice_partition(B):
    nr, nc, rp, ci, v = _csr(B)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    Mt = M.block_transpose()
    M.slice_block_rows(1, 4, rebase=True)
    M.partition_block_rows(3)
    M.partition_block_rows(2, Bt=Mt)


def _export_compare(B):
    nr, nc, rp, ci, v = _csr(B)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    r, c, x = M.generate_coo()
    assert M.compare(r, c, x)[:2] == (0, 0)
    drp, dci, dv = M.to_csr()
    assert M.compare_csr(drp, dci, dv)[:2] == (0, 0)
    hrp = np.empty(nr + 1, np.int32); hci = np.empty(ci.size, np.int32); hv = np.empty(ci.size, np.float32)     # bmsp_to_csr to host
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    B._lib.check(B.lib().bmsp_to_csr(M._h, p(hrp), p(hci), p(hv), B._lib.HOST, None))
    assert np.array_equal(hrp, rp) and np.array_equal(hci, ci)


def _set_values(B):
    nr, nc, rp, ci, v = _csr(B)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    B.bmSparse_mult(A, M)                                  # M keeps packed records: set_values rewrites them
    M.set_values(np.ones(M.nnz, np.float16))              # same dtype
    M.set_values(np.ones(M.nnz, np.float32))              # converted through a device buffer
    M.set_values(torch.ones(M.nnz, device="cuda"))
    M.set_values_csr(rp, ci, v)
    d = lambda a: torch.from_numpy(a).cuda()
    M.set_values_csr(d(rp), d(ci), d(v))


# ---- SpMV -----------------------------------------------------------------------------------------------------------
def _spmv_palette(B):
    nr, nc, rp, ci, v = _csr(B)
    _spmv(B, B.bmSpMatrix.from_csr(nr, nc, rp, ci, v), nc)


def _spmv_no_palette(B):
    nr, nc, rp, ci, v = _patterned_blocks_csr(300, 256, seed=256)     # 257 distinct bitmaps: more than a palette holds
    _spmv(B, B.bmSpMatrix.from_csr(nr, nc, rp, ci, v), nc)


def _spmv_per_tile(B, monkeypatch):
    monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
    nr, nc, rp, ci, v = _csr(B)
    _spmv(B, B.bmSpMatrix.from_csr(nr, nc, rp, ci, v), nc)
    rp, ci, v = random_csr(256, 512, 0.3, seed=9)                     # dense blocks: 16-row tiles
    _spmv(B, B.bmSpMatrix.from_csr(256, 512, rp, ci, v), 512)


def _spmv_block_parallel(B):
    rng = np.random.default_rng(4)
    nc = 80000
    rows = [np.sort(rng.choice(nc, 5000 if r in (9, 10) else (0 if r >= 16 else 3), replace=False)) for r in range(24)]
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int32)
    ci = np.concatenate(rows).astype(np.int32)
    M = B.bmSpMatrix.from_csr(24, nc, rp, ci, np.ones(ci.size, np.float32))
    assert M.nnz / M.block_num < 2.5
    _spmv(B, M, nc)


def _spmv_host(B):
    nr, nc, rp, ci, v = _csr(B)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    xh = torch.from_numpy(B.generators.x_vector(nc)).pin_memory()
    yh = torch.empty(nr).pin_memory()
    for _ in range(3):                # eager, captured as a graph, replayed
        B.bmSparse_SpMV_host(M, xh, yh)
        torch.cuda.synchronize()
    yp = torch.empty(nr)             # pageable: eager only
    B.bmSparse_SpMV_host(M, xh, yp)
    torch.cuda.synchronize()


# ---- SpGEMM ---------------------------------------------------------------------------------------------------------
def _mult(B, shA, a, shB, b, **kw):
    A = B.bmSpMatrix.from_csr(*shA, *a)
    Bt = B.bmSpMatrix.from_csr(*shB, *b, transpose=True)
    B.bmSparse_mult(A, Bt, VERBOSE=True, **kw)
    B.bmSparse_mult(A, Bt, **kw)          # B's packed records and fine index exist now


def _spgemm_poisson(B):
    nr, nc, rp, ci, v = B.generators.poisson5pt(64, 52)
    _mult(B, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))


def _spgemm_fine(B):
    nr, nc, rp, ci, v = B.generators.uniform_random(4096, 16, seed=7)
    _mult(B, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))


def _spgemm_rmat(B):
    nr, nc, rp, ci, v = B.generators.rmat(11)
    _mult(B, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))


def _spgemm_heavy_split(B, monkeypatch):
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", "300")
    _spgemm_rmat(B)


def _spgemm_dense(B):
    nr, nc, rp, ci, v = B.generators.block_clustered(64)
    _mult(B, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))


def _spgemm_mma(B):
    a = random_csr(16, 64, 0.9, seed=5)
    _mult(B, (16, 64), a, (64, 8 * 128 * 17), _strided_b(64, 128, 17, 0.5, seed=6), numeric_path=1)     # shared accumulators
    _mult(B, (16, 64), a, (64, 8 * 1200), random_csr(64, 8 * 1200, 0.5, seed=4), numeric_path=1)        # global accumulators


def _spgemm_plan(B, monkeypatch):
    for heavy in (None, "300"):
        if heavy:
            monkeypatch.setenv("BMSP_SPGEMM_HEAVY", heavy)
        for nr, nc, rp, ci, v in (B.generators.poisson5pt(64, 52), B.generators.rmat(11)):
            A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
            plan = B.bmSparse_mult_plan(A, Bt)
            plan.numeric(); plan.numeric()
            torch.cuda.synchronize()
            plan.close()


CASES = {
    "from_csr_host": _from_csr_host, "from_csr_device": _from_csr_device, "from_coo": _from_coo, "from_mtx": _from_mtx,
    "from_arrays": _from_arrays, "transpose_slice_partition": _transpose_slice_partition, "export_compare": _export_compare,
    "set_values": _set_values, "spmv_palette": _spmv_palette, "spmv_no_palette": _spmv_no_palette, "spmv_per_tile": _spmv_per_tile,
    "spmv_block_parallel": _spmv_block_parallel, "spmv_host": _spmv_host, "spgemm_poisson": _spgemm_poisson,
    "spgemm_fine": _spgemm_fine, "spgemm_rmat": _spgemm_rmat, "spgemm_heavy_split": _spgemm_heavy_split,
    "spgemm_dense": _spgemm_dense, "spgemm_mma": _spgemm_mma, "spgemm_plan": _spgemm_plan,
}


@pytest.mark.parametrize("name", list(CASES))
def test_entry_point_returns_its_memory(B, pool, monkeypatch, tmp_path, name):
    fn = CASES[name]
    extra = {"monkeypatch": monkeypatch, "tmp_path": tmp_path}
    kw = {k: extra[k] for k in inspect.signature(fn).parameters if k != "B"}
    _run(pool, name, lambda: fn(B, **kw))


# ---- validation failures ------------------------------------------------------------------------------------------
def _bad_csr(kind):
    rp = np.array([0, 2, 4, 6], np.int32); ci = np.array([1, 5, 0, 2, 3, 7], np.int32)
    if kind == "row_ptr":
        rp = np.array([0, 4, 2, 6], np.int32)
    elif kind == "unsorted":
        ci = np.array([5, 1, 0, 2, 3, 7], np.int32)
    elif kind == "duplicate":
        ci = np.array([1, 1, 0, 2, 3, 7], np.int32)
    elif kind == "range":
        ci = np.array([1, 5, 0, 2, 3, 9], np.int32)
    return rp, ci, np.ones(6, np.float32)


@pytest.mark.parametrize("kind", ["row_ptr", "unsorted", "duplicate", "range", "set_values_csr_pattern"])
def test_validation_failure_returns_its_memory(B, pool, kind):
    from bmsparse_spgemm_spmv_b200 import _lib as L
    d = lambda a: torch.from_numpy(a).cuda()
    rp, ci, v = _bad_csr("ok")
    M = B.bmSpMatrix.from_csr(3, 8, rp, ci, v)

    def fail():
        with pytest.raises(L.BmspError):
            if kind == "set_values_csr_pattern":
                M.set_values_csr(d(rp), d(np.array([1, 5, 0, 3, 2, 7], np.int32)), d(v))      # same lengths, other pattern
            else:
                B.bmSpMatrix.from_csr(3, 8, *(d(a) for a in _bad_csr(kind)))
    _run(pool, "invalid_" + kind, fail)
    assert np.array_equal(M.download()[3], np.ones(6, np.float16))
