"""GPU: bmSpMatrix.matrix_transpose (bmsp_matrix_transpose), the matrix A^T in either storage form.

The expected arrays are the oracle's conversion of A's own COO with rows and columns swapped, so every array of A^T is compared
bit for bit.  Products built from A^T (SpMV, A * A^T, P^T * A * P) are checked against scipy."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from tests.util import assert_structure_equal, csr_rows, random_csr

pytestmark = pytest.mark.gpu

FORMS = [(False, False), (False, True), (True, False), (True, True)]


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _assert_same_arrays(X, Y):
    for x, y in zip(X.download(), Y.download()):
        assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert X._view().offsets_len == Y._view().offsets_len


def _check_transpose(B, O, nr, nc, rp, ci, v, in_t, out_t, in_dtype=torch.float16, out_dtype=torch.float16):
    """A (nr x nc, form in_t, in_dtype) -> A^T (form out_t, out_dtype) against the oracle's conversion of A's swapped COO"""
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=in_t, dtype=in_dtype)
    At = A.matrix_transpose(dtype=out_dtype, transpose=out_t)
    stored = O.f16_round(v) if in_dtype == torch.float16 else np.asarray(v, np.float32)
    exp = O.coo_to_bmsp(nc, nr, ci, csr_rows(rp), stored, transposed=out_t, f16=(out_dtype == torch.float16))
    what = f"{nr}x{nc} {in_t}->{out_t}"
    assert (At.num_rows, At.num_cols, At.transposed, At.dtype) == (nc, nr, out_t, out_dtype), what
    assert At.nnz == A.nnz and At.block_num == exp.block_num, what
    k, b, o, vals = At.download()
    assert_structure_equal((k, b, o), exp, what)
    assert o.size == exp.offsets.size, what
    assert np.array_equal(vals.astype(np.float32), exp.values), what
    nbr = (nc + 7) // 8
    exp_brp = np.searchsorted(exp.keys >> np.uint64(32), np.arange(nbr + 1, dtype=np.uint64), side="left")
    assert np.array_equal(At.block_row_ptr.cpu().numpy(), exp_brp), what
    assert np.array_equal(At.block_col.cpu().numpy(), (exp.keys & np.uint64(0xFFFFFFFF)).astype(np.int32)), what
    return A, At


@pytest.mark.parametrize("shape", [(24, 24), (61, 29), (100, 7), (7, 300), (257, 513), (1000, 1000)])
@pytest.mark.parametrize("in_t,out_t", FORMS)
def test_bit_exact_vs_oracle(B, oracle, shape, in_t, out_t):
    nr, nc = shape
    rp, ci, v = random_csr(nr, nc, 0.08, seed=nr * 31 + nc, empty_block_rows=(1,) if nr > 24 else ())
    _check_transpose(B, oracle, nr, nc, rp, ci, v, in_t, out_t)


@pytest.mark.parametrize("in_dtype,out_dtype", [(torch.float16, torch.float32), (torch.float32, torch.float16), (torch.float32, torch.float32)])
@pytest.mark.parametrize("in_t,out_t", [(False, False), (True, True), (False, True)])
def test_dtype_pairs(B, oracle, in_dtype, out_dtype, in_t, out_t):
    """fp32 values that fp16 cannot hold: fp32 -> fp16 rounds once, so A^T equals from_csr of the transposed CSR at fp16"""
    nr, nc = 203, 171
    rp, ci, v = random_csr(nr, nc, 0.1, seed=31, empty_block_rows=(2,), fp16=False)
    A, At = _check_transpose(B, oracle, nr, nc, rp, ci, v, in_t, out_t, in_dtype, out_dtype)
    if in_dtype == torch.float32 and out_dtype == torch.float16:
        T = sp.csr_matrix((v, ci, rp), shape=(nr, nc)).T.tocsr()
        T.sort_indices()
        ref = B.bmSpMatrix.from_csr(nc, nr, T.indptr, T.indices, T.data.astype(np.float32), transpose=out_t, dtype=torch.float16)
        _assert_same_arrays(At, ref)


def _coo_csr(nr, nc, r, c, v):
    M = sp.csr_matrix((v, (r, c)), shape=(nr, nc))
    M.sort_indices()
    return M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float32)


@pytest.mark.parametrize("in_t,out_t", FORMS)
def test_wide_matrix_three_digit_sort(B, oracle, in_t, out_t):
    """16 x 560 000: 70 000 block columns (a three-pass radix sort), and its 560 000 x 16 transpose, whose transpose has two block
    rows of tens of thousands of blocks each"""
    rng = np.random.default_rng(7)
    n = 60000
    lin = np.unique(rng.integers(0, 16 * 560000, n))
    r, c = (lin // 560000).astype(np.int32), (lin % 560000).astype(np.int32)
    v = (rng.integers(1, 64, r.size) / 8.0).astype(np.float32)
    rp, ci, vv = _coo_csr(16, 560000, r, c, v)
    _check_transpose(B, oracle, 16, 560000, rp, ci, vv, in_t, out_t)
    rp, ci, vv = _coo_csr(560000, 16, c, r, v)
    _, At = _check_transpose(B, oracle, 560000, 16, rp, ci, vv, in_t, out_t)
    assert At.block_row_ptr.cpu().numpy()[1] > 20000


@pytest.mark.parametrize("in_t,out_t", FORMS)
def test_dense_column_and_rmat(B, oracle, in_t, out_t):
    """a dense column of A is one block row of A^T holding a block of every block row of A; R-MAT has skewed column counts"""
    nr, nc = 3000, 2500
    rp, ci, v = random_csr(nr, nc, 0.004, seed=12)
    r, c = csr_rows(rp), ci
    r = np.concatenate([r, np.arange(nr, dtype=np.int32)]); c = np.concatenate([c, np.full(nr, 1234, np.int32)])
    v = np.concatenate([v, np.full(nr, 0.75, np.float32)])
    keep = np.unique(r.astype(np.int64) * nc + c, return_index=True)[1]
    rp, ci, v = _coo_csr(nr, nc, r[keep], c[keep], v[keep])
    _check_transpose(B, oracle, nr, nc, rp, ci, v, in_t, out_t)
    nr, nc, rp, ci, v = B.generators.rmat(12)
    _check_transpose(B, oracle, nr, nc, rp, ci, v, in_t, out_t)


@pytest.mark.parametrize("in_t,out_t", FORMS)
def test_empty_and_one_by_one(B, oracle, in_t, out_t):
    E = B.bmSpMatrix.from_csr(16, 40, np.zeros(17, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32), transpose=in_t)
    Et = E.matrix_transpose(transpose=out_t)
    assert (Et.num_rows, Et.num_cols, Et.block_num, Et.nnz, Et.transposed) == (40, 16, 0, 0, out_t)
    assert Et.block_row_ptr.cpu().tolist() == [0] * 6
    _check_transpose(B, oracle, 1, 1, np.array([0, 1], np.int32), np.array([0], np.int32), np.array([2.0], np.float32), in_t, out_t)


def _square(B, n=300, density=0.05, seed=21):
    rp, ci, v = random_csr(n, n, density, seed=seed, empty_block_rows=(3,))
    return rp, ci, v


def test_involution_ingested_and_product(B):
    """transposing twice gives A's arrays bit for bit, offsets_len included: an ingested A (offsets_len = block_num) and an fp32
    SpGEMM product (offsets_len = block_num + 1, last entry = nnz)"""
    rp, ci, v = random_csr(257, 513, 0.08, seed=4)
    for t in (False, True):
        A = B.bmSpMatrix.from_csr(257, 513, rp, ci, v, transpose=t)
        for t2 in (False, True):
            _assert_same_arrays(A.matrix_transpose(transpose=t2).matrix_transpose(transpose=t), A)
    rp, ci, v = _square(B)
    A = B.bmSpMatrix.from_csr(300, 300, rp, ci, v); Bt = B.bmSpMatrix.from_csr(300, 300, rp, ci, v, transpose=True)
    C, _ = B.bmSparse_mult(A, Bt)
    assert C.dtype == torch.float32 and C._view().offsets_len == C.block_num + 1
    Ct = C.matrix_transpose()
    assert Ct._view().offsets_len == C.block_num + 1 and int(Ct.download()[2][-1]) == C.nnz
    _assert_same_arrays(Ct.matrix_transpose(), C)


def _dense(M):
    r, c, v = M.generate_coo()
    return sp.csr_matrix((v.astype(np.float64), (r, c)), shape=(M.num_rows, M.num_cols))


def test_spmv_with_transpose(B, oracle):
    nr, nc = 1000, 777
    rp, ci, v = random_csr(nr, nc, 0.03, seed=3, empty_block_rows=(1, 5))
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    x = B.generators.x_vector(nr)
    y = B.bmSparse_SpMV(A.matrix_transpose(), torch.from_numpy(x).cuda()).cpu().numpy().astype(np.float64)
    S = sp.csr_matrix((oracle.f16_round(v).astype(np.float64), ci, rp), shape=(nr, nc))
    ref = S.T @ x.astype(np.float64)
    absref = abs(S).T @ np.abs(x).astype(np.float64)
    assert np.all(np.abs(y - ref) <= 1e-5 * absref + 1e-30)


def test_a_times_a_transpose(B, oracle):
    """A * A^T through bmSparse_mult(A, A.matrix_transpose(transpose=True)): structure bit-exact, values within _mult_check's bound"""
    nr, nc = 400, 257
    rp, ci, v = random_csr(nr, nc, 0.06, seed=8, empty_block_rows=(2,))
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    C, info = B.bmSparse_mult(A, A.matrix_transpose(transpose=True))
    oA = oracle.csr_to_bmsp(nr, nc, rp, ci, v)
    oB = oracle.coo_to_bmsp(nc, nr, ci, csr_rows(rp), v, transposed=True)
    exp = oracle.spgemm(oA, oB)
    k, b, o, vals = C.download()
    assert_structure_equal((k, b, o), exp, "A*A^T")
    assert (C.num_rows, C.num_cols) == (nr, nr) and int(o[-1]) == exp.nnz == C.nnz
    mag = oracle.spgemm(oracle.OracleMatrix(nr, nc, oA.keys, oA.bmps, oA.offsets, np.abs(oA.values)),
                        oracle.OracleMatrix(nc, nr, oB.keys, oB.bmps, oB.offsets, np.abs(oB.values), True)).values
    err = np.abs(vals.astype(np.float64) - exp.values)
    assert np.all(err <= 1e-3 * np.maximum(np.abs(exp.values), 1e-3 * mag) + 1e-30)
    assert np.all(err <= 2e-6 * mag + 1e-30)


def test_galerkin_product(B):
    """P^T (A P) for the 5-point Laplacian on 32 x 32 and a 0/1 aggregation P (2 x 2 node aggregates): integer values, so exact"""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(32, 32)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    node = np.arange(nr)
    agg = ((node // 32) // 2) * 16 + (node % 32) // 2
    na = 256
    P = sp.csr_matrix((np.ones(nr, np.float32), (node, agg)), shape=(nr, na))
    P.sort_indices()
    prp, pci, pv = P.indptr.astype(np.int32), P.indices.astype(np.int32), P.data.astype(np.float32)
    P_plain = B.bmSpMatrix.from_csr(nr, na, prp, pci, pv)
    P_operand = B.bmSpMatrix.from_csr(nr, na, prp, pci, pv, transpose=True)
    plan = B.bmSparse_mult_plan(A, P_operand)
    APt = plan.C.block_transpose(torch.float16)
    RAP, _ = B.bmSparse_mult(P_plain.matrix_transpose(dtype=torch.float16), APt)
    S = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(nr, nc))
    ref = (P.T.astype(np.float64) @ S @ P.astype(np.float64)).tocsr()
    got = _dense(RAP)
    assert (RAP.num_rows, RAP.num_cols) == (na, na)
    assert abs(got - ref).max() == 0.0
    plan.close()


def test_fp32_product_fed_back(B):
    """C = A * A in fp32, then A * C^T with C^T = C.matrix_transpose(dtype=fp16, transpose=True)"""
    n = 300
    rp, ci, v = _square(B, n)
    A = B.bmSpMatrix.from_csr(n, n, rp, ci, v); At = B.bmSpMatrix.from_csr(n, n, rp, ci, v, transpose=True)
    C, _ = B.bmSparse_mult(A, At)
    Ct = C.matrix_transpose(dtype=torch.float16, transpose=True)
    assert Ct.transposed and Ct.dtype == torch.float16 and Ct.nnz == C.nnz
    Cs = _dense(C)
    CtS = _dense(Ct)                                         # the matrix Ct holds: C^T with fp16 values
    assert np.array_equal(CtS.toarray(), Cs.T.toarray().astype(np.float16).astype(np.float64))
    D, _ = B.bmSparse_mult(A, Ct)
    S = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(n, n))
    ref = (S @ CtS).toarray()
    mag = (abs(S) @ abs(CtS)).toarray()
    assert np.all(np.abs(_dense(D).toarray() - ref) <= 2e-6 * mag + 1e-30)


def test_independent_of_source_and_streams(B):
    rp, ci, v = random_csr(257, 513, 0.08, seed=5)
    A = B.bmSpMatrix.from_csr(257, 513, rp, ci, v)
    At = A.matrix_transpose()
    before = At.download()
    A.set_values(torch.full((A.nnz,), 3.0, device="cuda"))
    torch.cuda.synchronize()
    for x, y in zip(At.download(), before):
        assert np.array_equal(x, y)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        A2 = B.bmSpMatrix.from_csr(257, 513, rp, ci, v, stream=s)
        At2 = A2.matrix_transpose(stream=s)
    s.synchronize()
    for x, y in zip(At2.download(), before):
        assert np.array_equal(x, y)
    del A, A2
    scratch = [B.bmSpMatrix.from_csr(257, 513, rp, ci, np.full(ci.size, 5.0, np.float32)) for _ in range(4)]   # reuse freed memory
    torch.cuda.synchronize()
    for x, y in zip(At.download(), before):
        assert np.array_equal(x, y)
    assert B.bmSparse_SpMV(At, torch.ones(257, device="cuda")).shape == (513,)
    del scratch


def test_errors(B):
    from bmsparse_spgemm_spmv_b200 import _lib as L
    A = B.bmSpMatrix.from_csr(8, 8, np.array([0, 1] + [1] * 7, np.int32), np.array([3], np.int32), np.array([1.0], np.float32))
    out = ctypes.c_void_p()
    assert L.lib().bmsp_matrix_transpose(A._h, 7, 0, None, ctypes.byref(out)) == 1
    assert L.lib().bmsp_matrix_transpose(None, L.F16, 0, None, ctypes.byref(out)) == 1
    assert L.lib().bmsp_matrix_transpose(A._h, L.F16, 0, None, None) == 1
    assert not out
