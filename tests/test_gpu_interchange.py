"""GPU: the host-memory forms of the export and compare calls give what their device forms give, and the host COO compare's
handling of entries outside the matrix and of repeated entries."""
import ctypes

import numpy as np
import pytest
import torch

from tests.util import csr_rows, random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if isinstance(a, np.ndarray) else ctypes.c_void_p(a.data_ptr())


def _compare_csr(B, M, rp, ci, v, mem):
    """bmsp_compare_csr with the three arrays in host (numpy) or device (torch) memory"""
    L = B._lib
    out = [ctypes.c_int64(), ctypes.c_int64(), ctypes.c_double(), ctypes.c_double()]
    L.check(B.lib().bmsp_compare_csr(M._h, _p(rp), _p(ci), _p(v), mem, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream),
                                     *(ctypes.byref(x) for x in out)))
    return tuple(x.value for x in out)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("gen", ["random", "poisson"])
def test_to_csr_host_equals_device(B, dtype, gen):
    if gen == "poisson":
        nr, nc, rp, ci, v = B.generators.poisson5pt(70, 53)
    else:
        nr, nc = 1001, 777
        rp, ci, v = random_csr(nr, nc, 0.03, seed=3, empty_block_rows=(1, 5), fp16=False)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=dtype)
    drp, dci, dv = M.to_csr()
    hrp = np.full(nr + 1, -1, np.int32); hci = np.full(ci.size, -1, np.int32); hv = np.full(ci.size, np.nan, np.float32)
    B._lib.check(B.lib().bmsp_to_csr(M._h, _p(hrp), _p(hci), _p(hv), B._lib.HOST, None))
    assert np.array_equal(hrp, drp.cpu().numpy()) and np.array_equal(hci, dci.cpu().numpy())
    assert np.array_equal(hv, dv.cpu().numpy())


@pytest.mark.parametrize("gen", ["random", "poisson"])
def test_compare_csr_host_equals_device(B, gen):
    """the identity case and the two-dropped, one-perturbed case of test_to_csr_and_device_compare, host arrays against device ones"""
    if gen == "poisson":
        nr, nc, rp, ci, v = B.generators.poisson5pt(70, 53)
    else:
        nr, nc = 1001, 777
        rp, ci, v = random_csr(nr, nc, 0.03, seed=3, empty_block_rows=(1, 5))
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    v2 = v.astype(np.float16).astype(np.float32)
    keep = np.ones(ci.size, bool); keep[[3, ci.size // 2]] = False
    rp3 = np.zeros(nr + 1, np.int64); np.cumsum(np.bincount(csr_rows(rp)[keep], minlength=nr), out=rp3[1:])
    v3 = v2[keep].copy(); v3[10] *= 1.5
    for crp, cci, cv, exp_ab in ((rp, ci, v2, (0, 0)), (rp3.astype(np.int32), ci[keep], v3, (2, 0))):
        host = _compare_csr(B, M, crp, cci, cv, B._lib.HOST)
        dev = _compare_csr(B, M, *(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (crp, cci, cv)), B._lib.DEVICE)
        assert host == dev and host[:2] == exp_ab


def test_compare_coo_outside_rows_and_repeated_entries(B):
    rp, ci, v = random_csr(40, 30, 0.2, seed=12)
    M = B.bmSpMatrix.from_csr(40, 30, rp, ci, v)
    r, c = csr_rows(rp), ci
    assert M.compare(r, c, v) == (0, 0, 0.0, 0.0)
    # rows outside [0, 40): only in the COO
    assert M.compare(np.r_[r, -1, 40], np.r_[c, 0, 3], np.r_[v, 1.0, 1.0]) == (0, 2, 0.0, 0.0)
    # entry e twice: the first in input order is the one compared, the other is only in the COO
    e = 5
    rd, cd = np.r_[r, r[e]], np.r_[c, c[e]]
    assert M.compare(rd, cd, np.r_[v, v[e] * 1.5]) == (0, 1, 0.0, 0.0)
    vd = v.copy(); vd[e] *= 1.5
    a, b, mean, mx = M.compare(rd, cd, np.r_[vd, v[e]])
    assert (a, b) == (0, 1) and abs(mx - 1.0 / 3.0) < 1e-6 and abs(mean - (1.0 / 3.0) / ci.size) < 1e-9
