"""GPU: bmSparse_add (bmsp_add), C = alpha*A + beta*B in the block format.

The expected matrix is built in numpy from the two operands' stored entries: the union of their patterns, with entries that cancel
kept (unlike scipy's A + B), and every value fl(fl(alpha*a) + fl(beta*b)) in float32 with a missing entry = 0.  from_csr of that
CSR with fp32 values, in the operands' form and C's dtype, must equal C in all four arrays and offsets_len, bit for bit."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from tests.test_gpu_device_memory import _Pool, _run, pool  # noqa: F401
from tests.util import csr_rows, random_csr

pytestmark = pytest.mark.gpu

F16, F32 = torch.float16, torch.float32
DTYPES = [(ta, tb, tc) for ta in (F16, F32) for tb in (F16, F32) for tc in (F16, F32)]
SCALES = [(1.0, 1.0), (1.0, -1.0), (0.5, 3.0), (0.0, 2.0)]


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _entries(M):
    """M's stored entries as (row * num_cols + col, fp32 value), sorted"""
    r, c, v = M.generate_coo()
    lin = r.astype(np.int64) * M.num_cols + c
    o = np.argsort(lin, kind="stable")
    return lin[o], v[o].astype(np.float32)


def _expected(B, X, Y, alpha, beta, dtype, transpose):
    nr, nc = X.num_rows, X.num_cols
    la, va = _entries(X)
    lb, vb = _entries(Y)
    u = np.union1d(la, lb)
    a = np.zeros(u.size, np.float32); a[np.searchsorted(u, la)] = va
    b = np.zeros(u.size, np.float32); b[np.searchsorted(u, lb)] = vb
    vals = np.float32(alpha) * a + np.float32(beta) * b
    rows = (u // nc).astype(np.int32)
    rp = np.zeros(nr + 1, np.int64)
    np.cumsum(np.bincount(rows, minlength=nr), out=rp[1:])
    return B.bmSpMatrix.from_csr(nr, nc, rp.astype(np.int32), (u % nc).astype(np.int32), vals, transpose=transpose, dtype=dtype)


def _assert_same_arrays(X, Y, what=""):
    for name, x, y in zip(("keys", "bmps", "offsets", "values"), X.download(), Y.download()):
        assert x.dtype == y.dtype and x.size == y.size and np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"{what}: {name} differ"
    assert X._view().offsets_len == Y._view().offsets_len, what
    assert (X.num_rows, X.num_cols, X.transposed, X.dtype) == (Y.num_rows, Y.num_cols, Y.transposed, Y.dtype), what
    assert torch.equal(X.block_row_ptr, Y.block_row_ptr) and torch.equal(X.block_col, Y.block_col), what


def _check(B, X, Y, alpha=1.0, beta=1.0, dtype=None, what=""):
    Cm = B.bmSparse_add(X, Y, alpha, beta, dtype=dtype)
    exp_dtype = dtype or (F32 if F32 in (X.dtype, Y.dtype) else F16)
    assert Cm.dtype == exp_dtype and Cm._view().offsets_len == Cm.block_num, what
    _assert_same_arrays(Cm, _expected(B, X, Y, alpha, beta, exp_dtype, X.transposed), what)
    return Cm


def _mat(B, nr, nc, rp, ci, v, t=False, dtype=F16):
    return B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=t, dtype=dtype)


def _pair(nr, nc, seed, empty_a=(), empty_b=(), density=0.08):
    """two random patterns that overlap in part; fp32 values fp16 cannot hold"""
    return (random_csr(nr, nc, density, seed=seed, empty_block_rows=empty_a, fp16=False),
            random_csr(nr, nc, density, seed=seed + 1000, empty_block_rows=empty_b, fp16=False))


def _unique(r, c, nc, v):
    """(row, col, value) with repeated (row, col) dropped"""
    lin, first = np.unique(r.astype(np.int64) * nc + c, return_index=True)
    return (lin // nc).astype(np.int32), (lin % nc).astype(np.int32), v[first]


def _coo_csr(nr, nc, r, c, v):
    M = sp.csr_matrix((np.asarray(v, np.float32), (r, c)), shape=(nr, nc))
    M.sort_indices()
    return M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float32)


@pytest.mark.parametrize("alpha,beta", SCALES)
@pytest.mark.parametrize("ta,tb,tc", DTYPES)
@pytest.mark.parametrize("t", [False, True])
def test_bit_exact_dtypes_and_scales(B, t, ta, tb, tc, alpha, beta):
    nr, nc = 61, 45
    a, b = _pair(nr, nc, seed=3, empty_a=(2,), empty_b=(2, 4))
    X, Y = _mat(B, nr, nc, *a, t=t, dtype=ta), _mat(B, nr, nc, *b, t=t, dtype=tb)
    _check(B, X, Y, alpha, beta, tc, f"{t} {ta} {tb} {tc} {alpha} {beta}")


@pytest.mark.parametrize("shape", [(1, 1), (7, 300), (100, 7), (257, 513), (1000, 999)])
@pytest.mark.parametrize("t", [False, True])
def test_shapes_and_empty_block_rows(B, shape, t):
    nr, nc = shape
    a, b = _pair(nr, nc, seed=nr + nc, empty_a=(1, 3) if nr > 32 else (), empty_b=(3, 5) if nr > 48 else ())
    X, Y = _mat(B, nr, nc, *a, t=t), _mat(B, nr, nc, *b, t=t, dtype=F32)
    _check(B, X, Y, 0.5, 3.0, F16, f"{shape} {t}")
    _check(B, Y, X, 1.0, -1.0, None, f"{shape} {t} swapped")


@pytest.mark.parametrize("t", [False, True])
def test_explicit_zeros_and_cancellation(B, t):
    """explicit zero entries stay; A - A keeps A's whole pattern with (signed) zeros; A passed as both operands"""
    nr, nc = 130, 77
    rp, ci, v = random_csr(nr, nc, 0.1, seed=9, empty_block_rows=(4,))
    v = v.copy(); v[::5] = 0.0; v[1::7] = -0.0
    X = _mat(B, nr, nc, rp, ci, v, t=t)
    D = _check(B, X, X, 1.0, -1.0, None, "A - A")
    assert D.nnz == X.nnz and D.block_num == X.block_num
    assert np.all(D.download()[3] == 0)
    _check(B, X, X, 1.0, 1.0, None, "A + A")
    _check(B, X, X, 0.0, 0.0, F32, "0A + 0A")
    Y = _mat(B, nr, nc, rp, ci, -np.asarray(v), t=t)
    Z = _check(B, X, Y, 1.0, 1.0, F16, "A + (-A)")
    assert Z.nnz == X.nnz


@pytest.mark.parametrize("t", [False, True])
def test_identical_disjoint_interleaved_empty(B, t):
    nr, nc = 200, 160
    rp, ci, v = random_csr(nr, nc, 0.1, seed=5, fp16=False)
    r = csr_rows(rp)
    X = _mat(B, nr, nc, rp, ci, v, t=t)
    _check(B, X, _mat(B, nr, nc, rp, ci, v[::-1].copy(), t=t), 0.5, 3.0, F32, "identical patterns")
    top, bot = r < 96, r >= 96                                   # disjoint block rows
    _check(B, _mat(B, nr, nc, *_coo_csr(nr, nc, r[top], ci[top], v[top]), t=t),
           _mat(B, nr, nc, *_coo_csr(nr, nc, r[bot], ci[bot], v[bot]), t=t), 1.0, 1.0, None, "disjoint")
    ev, od = (ci // 8) % 2 == 0, (ci // 8) % 2 == 1              # interleaved blocks of every block row
    _check(B, _mat(B, nr, nc, *_coo_csr(nr, nc, r[ev], ci[ev], v[ev]), t=t),
           _mat(B, nr, nc, *_coo_csr(nr, nc, r[od], ci[od], v[od]), t=t), 1.0, -1.0, None, "interleaved")
    inside = (ci % 8) < 4                                        # the same blocks, interleaved cells
    _check(B, _mat(B, nr, nc, *_coo_csr(nr, nc, r[inside], ci[inside], v[inside]), t=t),
           _mat(B, nr, nc, *_coo_csr(nr, nc, r[~inside], ci[~inside], v[~inside]), t=t), 0.5, 3.0, F16, "interleaved cells")
    E = _mat(B, nr, nc, np.zeros(nr + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32), t=t)
    _check(B, X, E, 1.0, 1.0, None, "A + 0")
    _check(B, E, X, 2.0, 0.5, None, "0 + A")
    Z = _check(B, E, E, 1.0, 1.0, F32, "both empty")
    assert (Z.block_num, Z.nnz) == (0, 0) and Z.block_row_ptr.cpu().tolist() == [0] * (nr // 8 + 1)


@pytest.mark.parametrize("t", [False, True])
def test_many_blocks_across_tiles(B, t):
    """about 600 000 blocks per operand, half of B's on A's keys: shared keys straddle merge-tile boundaries"""
    rng = np.random.default_rng(11)
    nr = nc = 40000
    n = 600000
    ra, ca = rng.integers(0, nr, n), rng.integers(0, nc, n)
    take = rng.random(n) < 0.5
    rb = np.where(take, ra, rng.integers(0, nr, n)); cb = np.where(take, (ca // 8) * 8 + rng.integers(0, 8, n), rng.integers(0, nc, n))
    A_ = _coo_csr(nr, nc, *_unique(ra, ca, nc, rng.uniform(-1, 1, n).astype(np.float32)))
    B_ = _coo_csr(nr, nc, *_unique(rb, cb, nc, rng.uniform(-1, 1, n).astype(np.float32)))
    X, Y = _mat(B, nr, nc, *A_, t=t), _mat(B, nr, nc, *B_, t=t)
    assert X.block_num > 500000 and Y.block_num > 500000
    _check(B, X, Y, 1.0, -1.0, None, "many blocks")


@pytest.mark.parametrize("t", [False, True])
def test_two_long_block_rows(B, t):
    """16 rows: two block rows of tens of thousands of blocks each, all in a handful of merge tiles"""
    rng = np.random.default_rng(7)
    nc = 560000
    mats = []
    for s in range(2):
        lin = np.unique(rng.integers(0, 16 * nc, 60000))
        r, c = (lin // nc).astype(np.int32), (lin % nc).astype(np.int32)
        mats.append(_mat(B, 16, nc, *_coo_csr(16, nc, r, c, (rng.integers(1, 64, r.size) / 8.0).astype(np.float32)), t=t))
    Cm = _check(B, mats[0], mats[1], 0.5, 3.0, None, "two long block rows")
    assert Cm.block_row_ptr.cpu().numpy()[1] > 20000


@pytest.mark.parametrize("t", [False, True])
def test_rmat_plus_transpose(B, t):
    """A + A^T for R-MAT(12): skewed rows and columns; A + A^T is symmetric, so its transpose is itself, bit for bit"""
    nr, nc, rp, ci, v = B.generators.rmat(12)
    A = _mat(B, nr, nc, rp, ci, v, t=t)
    S = _check(B, A, A.matrix_transpose(transpose=t), 1.0, 1.0, None, "A + A^T")
    _assert_same_arrays(S.matrix_transpose(transpose=t), S, "(A + A^T)^T")


def test_product_as_operand(B):
    """an fp32 SpGEMM result (offsets_len = block_num + 1) on either side"""
    n = 300
    rp, ci, v = random_csr(n, n, 0.05, seed=21, empty_block_rows=(3,))
    A = _mat(B, n, n, rp, ci, v)
    P, _ = B.bmSparse_mult(A, _mat(B, n, n, rp, ci, v, t=True))
    assert P._view().offsets_len == P.block_num + 1
    _check(B, P, A, 1.0, -0.5, None, "P - A/2")
    _check(B, A, P, 2.0, 1.0, F16, "2A + P")
    _check(B, P, P, 1.0, 1.0, None, "P + P")


def _dense(M):
    r, c, v = M.generate_coo()
    return sp.csr_matrix((v.astype(np.float64), (r, c)), shape=(M.num_rows, M.num_cols))


def test_sum_as_spmv_and_spgemm_operand(B):
    nr = nc = 520
    a, b = _pair(nr, nc, seed=17, empty_a=(5,), density=0.03)
    X, Y = _mat(B, nr, nc, *a), _mat(B, nr, nc, *b)
    Cm = B.bmSparse_add(X, Y, 1.0, -2.0)
    E = _expected(B, X, Y, 1.0, -2.0, F16, False)
    _assert_same_arrays(Cm, E)
    x = torch.from_numpy(B.generators.x_vector(nc)).cuda()
    assert torch.equal(B.bmSparse_SpMV(Cm, x), B.bmSparse_SpMV(E, x))
    Xt, Yt = _mat(B, nr, nc, *a, t=True), _mat(B, nr, nc, *b, t=True)
    Ct = B.bmSparse_add(Xt, Yt, 1.0, -2.0)
    Et = _expected(B, Xt, Yt, 1.0, -2.0, F16, True)
    _assert_same_arrays(Ct, Et)
    P, _ = B.bmSparse_mult(Cm, Ct)
    R, _ = B.bmSparse_mult(E, Et)
    pk, pb, po, pv = P.download()
    rk, rb, ro, rv = R.download()
    assert np.array_equal(pk, rk) and np.array_equal(pb, rb) and np.array_equal(po, ro)
    S = _dense(Cm)
    mag = (abs(S) @ abs(S)).max()
    assert np.abs(pv.astype(np.float64) - rv).max() <= 2e-6 * mag                  # the product's own summation order may differ
    assert abs(_dense(P) - S @ S).max() <= 2e-6 * mag


def test_smoothed_prolongator(B):
    """P = (I - omega D^-1 A) T for the 5-point Laplacian on 32 x 32 and 2 x 2 aggregates, through D^-1 A = Dinv * A,
    S = I - omega D^-1 A (fp16) and S * T; against scipy in float64, within fp16 rounding of S"""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(32, 32)
    n = nr
    A_op = _mat(B, n, n, rp, ci, v, t=True)
    d = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(n, n)).diagonal()
    eye = np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32)
    Dinv = _mat(B, n, n, *eye, (1.0 / d).astype(np.float32))
    I = _mat(B, n, n, *eye, np.ones(n, np.float32))
    omega = 2.0 / 3.0
    DinvA, _ = B.bmSparse_mult(Dinv, A_op)
    S = B.bmSparse_add(I, DinvA, 1.0, -omega, dtype=F16)
    node = np.arange(n)
    agg = ((node // 32) // 2) * 16 + (node % 32) // 2
    T = sp.csr_matrix((np.ones(n, np.float32), (node, agg)), shape=(n, 256))
    T.sort_indices()
    P, _ = B.bmSparse_mult(S, _mat(B, n, 256, T.indptr.astype(np.int32), T.indices.astype(np.int32), T.data, t=True))
    As = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(n, n))
    ref = ((sp.identity(n) - omega * sp.diags(1.0 / d) @ As) @ T.astype(np.float64)).toarray()
    got = _dense(P).toarray()
    assert (P.num_rows, P.num_cols) == (n, 256)
    assert np.abs(got - ref).max() <= 2e-3 * np.abs(ref).max()


def test_independent_of_operands_and_streams(B):
    nr, nc = 257, 513
    a, b = _pair(nr, nc, seed=4)
    X, Y = _mat(B, nr, nc, *a), _mat(B, nr, nc, *b)
    Cm = B.bmSparse_add(X, Y, 0.5, 3.0)
    before = Cm.download()
    again = B.bmSparse_add(X, Y, 0.5, 3.0)                      # two calls: identical arrays
    for x, y in zip(again.download(), before):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    del X, Y, again
    scratch = [B.bmSpMatrix.from_csr(nr, nc, a[0], a[1], np.full(a[1].size, 5.0, np.float32)) for _ in range(4)]   # reuse freed memory
    torch.cuda.synchronize()
    for x, y in zip(Cm.download(), before):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        X2, Y2 = (B.bmSpMatrix.from_csr(nr, nc, *p, stream=s) for p in (a, b))
        C2 = B.bmSparse_add(X2, Y2, 0.5, 3.0, stream=s)
    s.synchronize()
    for x, y in zip(C2.download(), before):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert B.bmSparse_SpMV(Cm, torch.ones(nc, device="cuda")).shape == (nr,)
    del scratch


def test_errors(B):
    from bmsparse_spgemm_spmv_b200 import _lib as L
    lib = L.lib()
    f = ctypes.c_float
    rp, ci, v = random_csr(16, 16, 0.2, seed=1)
    X = _mat(B, 16, 16, rp, ci, v)
    Xt = _mat(B, 16, 16, rp, ci, v, t=True)
    W = _mat(B, 16, 24, np.zeros(17, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    H = _mat(B, 24, 16, np.zeros(25, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    out = ctypes.c_void_p()
    for args in [(X._h, X._h, 7), (X._h, X._h, -1), (None, X._h, L.F16), (X._h, None, L.F16), (X._h, W._h, L.F16),
                 (X._h, H._h, L.F16)]:
        assert lib.bmsp_add(f(1), args[0], f(1), args[1], args[2], None, ctypes.byref(out)) == 1, args
    assert lib.bmsp_add(f(1), X._h, f(1), X._h, L.F16, None, None) == 1
    assert lib.bmsp_add(f(1), X._h, f(1), Xt._h, L.F16, None, ctypes.byref(out)) == 7
    assert not out
    with pytest.raises(L.BmspError) as e:
        B.bmSparse_add(X, Xt)
    assert e.value.code == 7
    with pytest.raises(L.BmspError) as e:
        B.bmSparse_add(X, W)
    assert e.value.code == 1


def _dense_blocks(B, nbr, bc):
    """nbr block rows x 2 block columns, one full block per block row in block column bc: 64 * nbr fp16 values"""
    br = torch.arange(nbr, dtype=torch.int64, device="cuda")
    keys = (br << 32) | bc
    bmps = torch.full((nbr,), -1, dtype=torch.int64, device="cuda")
    offs = br * 64
    vals = torch.ones(nbr * 64, dtype=torch.float16, device="cuda")
    return B.bmSpMatrix.from_arrays(8 * nbr, 16, nbr, keys, bmps, offs, vals)


def test_memory_returns_and_too_large(B, pool):
    """used device memory is back at its baseline after a sum and after every failure; a union of 2^32 values (two disjoint
    operands of 2^31 values each) fails with BMSP_ERR_TOO_LARGE once the counts are read back, before C is allocated"""
    from bmsparse_spgemm_spmv_b200 import _lib as L
    nr = nc = 300
    a, b = _pair(nr, nc, seed=8)

    def ok():
        X, Y = _mat(B, nr, nc, *a), _mat(B, nr, nc, *b, dtype=F32)
        Cm = B.bmSparse_add(X, Y, 1.0, -1.0)
        B.bmSparse_SpMV(Cm, torch.ones(nc, device="cuda"))
        torch.cuda.synchronize()
    _run(pool, "add", ok)
    X, Xt = _mat(B, nr, nc, *a), _mat(B, nr, nc, *a, t=True)
    W = _mat(B, nr, nc + 8, np.zeros(nr + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    for name, args, code in [("shape", (X, W), 1), ("form", (X, Xt), 7)]:
        def fail(args=args, code=code):
            with pytest.raises(L.BmspError) as e:
                B.bmSparse_add(*args)
            assert e.value.code == code
        _run(pool, "add_invalid_" + name, fail)
    del X, Xt, W
    nbr = 1 << 25
    Big0, Big1 = _dense_blocks(B, nbr, 0), _dense_blocks(B, nbr, 1)
    assert Big0.nnz == 1 << 31

    def too_large():
        with pytest.raises(L.BmspError) as e:
            B.bmSparse_add(Big0, Big1)
        assert e.value.code == 6
    _run(pool, "add_too_large", too_large)
