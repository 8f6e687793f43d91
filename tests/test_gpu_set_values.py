"""GPU: new values for an existing matrix (bmSpMatrix.set_values / set_values_csr), the copies of them the library keeps, and the
pattern check that leaves a matrix untouched when the CSR does not match."""
import ctypes

import numpy as np
import pytest
import torch

from tests.test_gpu_spgemm_reuse import _oracle_values
from tests.util import random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _fp32_values(n, seed):
    """values that fp16 cannot hold exactly: the conversion's rounding is part of what is compared"""
    v = np.random.default_rng(seed).uniform(-3, 3, n).astype(np.float32)
    v[v == 0] = 0.3
    return v


@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("device", [False, True])
def test_set_values_csr_matches_from_csr(B, transpose, dtype, device):
    rp, ci, _ = random_csr(203, 171, 0.08, seed=21, empty_block_rows=(2,), fp16=False)
    v1, v2 = _fp32_values(ci.size, 1), _fp32_values(ci.size, 2)
    d = (lambda a: torch.from_numpy(a).cuda()) if device else (lambda a: a)
    M = B.bmSpMatrix.from_csr(203, 171, d(rp), d(ci), d(v1), transpose=transpose, dtype=dtype)
    M.set_values_csr(d(rp), d(ci), d(v2))
    F = B.bmSpMatrix.from_csr(203, 171, rp, ci, v2, transpose=transpose, dtype=dtype)
    assert torch.equal(M.values, F.values)
    # fp16 input values
    h = v1.astype(np.float16)
    M.set_values_csr(d(rp), d(ci), d(h))
    assert torch.equal(M.values, B.bmSpMatrix.from_csr(203, 171, rp, ci, h, transpose=transpose, dtype=dtype).values)


@pytest.mark.parametrize("device", [False, True])
def test_set_values_compact_fp32_to_fp16(B, device):
    rp, ci, v = random_csr(150, 130, 0.1, seed=22)
    M = B.bmSpMatrix.from_csr(150, 130, rp, ci, v, transpose=True)
    new = _fp32_values(M.nnz, 3)
    M.set_values(torch.from_numpy(new).cuda() if device else new)
    torch.cuda.synchronize()
    assert torch.equal(M.values.cpu(), torch.from_numpy(new).half())


@pytest.mark.parametrize("src", [np.float16, np.float32])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("device", [False, True])
def test_set_values_compact_dtype_pairs(B, src, dtype, device):
    """compact values of either dtype into a matrix of either dtype: copied when the dtypes agree, converted when they differ"""
    rp, ci, v = random_csr(150, 130, 0.1, seed=22)
    M = B.bmSpMatrix.from_csr(150, 130, rp, ci, v, dtype=dtype)
    new = _fp32_values(M.nnz, 3).astype(src)
    M.set_values(torch.from_numpy(new).cuda() if device else new)
    torch.cuda.synchronize()
    assert torch.equal(M.values.cpu(), torch.from_numpy(new).to(dtype))


def test_set_values_none_after_in_place_write(B, oracle):
    """a B operand used once (packed records built), its values rewritten through .values, set_values(None), multiplied again"""
    nr, nc, rp, ci, v = B.generators.poisson5pt(40, 36)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    B.bmSparse_mult(A, Bt)
    v2 = _fp32_values(ci.size, 4).astype(np.float16).astype(np.float32)
    Bt.values.copy_(B.bmSpMatrix.from_csr(nr, nc, rp, ci, v2, transpose=True).values)
    Bt.set_values(None)
    C, _ = B.bmSparse_mult(A, Bt)
    _oracle_values(oracle, C, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v2))


@pytest.mark.parametrize("gen", ["poisson_palette", "uniform_block_parallel"])
def test_spmv_after_update(B, gen):
    """SpMV on an updated matrix (its SpMV plan kept) equals SpMV on a fresh handle bit for bit: the streaming kernel with a
    bitmap palette (Poisson) and the block-parallel path (uniform random), as tests/test_gpu_spmv_halo.py picks them"""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(1100, 1003) if gen == "poisson_palette" else G.uniform_random(20000, 16)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    x = torch.from_numpy(G.x_vector(nc)).cuda()
    B.bmSparse_SpMV(M, x)                          # plans
    v2 = _fp32_values(ci.size, 5)
    M.set_values_csr(rp, ci, v2)
    y = B.bmSparse_SpMV(M, x)
    assert torch.equal(y, B.bmSparse_SpMV(B.bmSpMatrix.from_csr(nr, nc, rp, ci, v2), x))


@pytest.mark.parametrize("gen", ["uniform_random", "poisson"])
def test_stale_copies_refreshed(B, oracle, gen):
    """a B operand used once keeps copies of its values (packed records; the fine index too for uniform random): after
    set_values_csr the next product must use the new values"""
    G = B.generators
    nr, nc, rp, ci, v = G.uniform_random(4096, 16, seed=7) if gen == "uniform_random" else G.poisson5pt(48, 40)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    B.bmSparse_mult(A, Bt)
    v2 = _fp32_values(ci.size, 6).astype(np.float16).astype(np.float32)
    Bt.set_values_csr(rp, ci, v2)
    C, _ = B.bmSparse_mult(A, Bt)
    _oracle_values(oracle, C, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v2))


def _mismatches(rp, ci, v, ncols):
    """(name, row_ptr, col_idx, vals): CSRs whose pattern differs from (rp, ci)"""
    n = np.diff(rp)
    r = int(np.flatnonzero((n >= 2) & (np.r_[ci[rp[1:] - 1]] < ncols - 1))[0])   # two entries or more, the last not in the last column
    e, last = int(rp[r]), int(rp[r + 1]) - 1
    out = []
    ci_x = np.insert(ci, last + 1, ci[last] + 1); rp_x = rp.copy(); rp_x[r + 1:] += 1
    out.append(("extra", rp_x, ci_x, np.insert(v, last + 1, 1.0)))
    rp_m = rp.copy(); rp_m[r + 1:] -= 1
    out.append(("missing", rp_m, np.delete(ci, e), np.delete(v, e)))
    ci_w = ci.copy(); ci_w[last] += 1
    out.append(("wrong_column", rp, ci_w, v))
    rp_t = rp.copy(); rp_t[-1] -= 1
    out.append(("row_ptr_total", rp_t, ci, v))
    rp_s = rp.copy(); rp_s[r + 1] -= 1                        # the same total, row r's last entry handed to row r + 1
    out.append(("moved_entry", rp_s, ci, v))
    return out


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("transpose", [False, True])
def test_pattern_mismatch_rejected(B, device, transpose):
    rp, ci, v = random_csr(120, 96, 0.1, seed=23)
    M = B.bmSpMatrix.from_csr(120, 96, rp, ci, v, transpose=transpose)
    before = M.values.clone()
    d = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if device else (lambda a: a)
    for name, rp2, ci2, v2 in _mismatches(rp, ci, v, 96):
        with pytest.raises(B.BmspError) as ex:
            M.set_values_csr(d(rp2), d(ci2), d(v2 * 2))
        assert ex.value.code == 1, name
        assert torch.equal(M.values, before), name
    # the C call itself, with col_idx / vals of the matrix's length: the device check is what rejects these
    from bmsparse_spgemm_spmv_b200 import _lib as L
    for name, rp2, ci2, v2 in _mismatches(rp, ci, v, 96):
        if ci2.size != ci.size:
            continue
        t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (rp2.astype(np.int32), ci2.astype(np.int32), (v2 * 2).astype(np.float32))]
        code = L.lib().bmsp_set_values_csr(M._h, *(ctypes.c_void_p(x.data_ptr()) for x in t), L.F32, L.DEVICE,
                                           ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert code == 1, name
        assert torch.equal(M.values, before), name
