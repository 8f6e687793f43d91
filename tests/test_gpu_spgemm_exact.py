"""Exact values of C = A * B on the SpGEMM paths test_gpu_spgemm_paths.py plans, with fp16 operands that hold small integers.

When every product a_ik * b_kj and every partial sum is an integer below 2^24 (checked per entry: sum_k |a_ik b_kj| < 2^24), fp32
accumulation is exact in any order, scalar or on the tensor cores (mma.sync accumulates in fp32), so C's values must equal scipy's
int64 product bit for bit: a dropped, doubled or misrouted product of any size changes an entry.  The structure is compared with
the oracle by the existing tests; these compare values, including entries that cancel to zero."""
import numpy as np
import pytest
import scipy.sparse as sp

from tests.test_gpu_spgemm_paths import DENSE_MAX_WORDS, MMA_SHARED_CAP, _fine_chosen, _hub_row, _paired_rows, _plan, _strided_b
from tests.util import random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _ints(csr, seed, lo=1, hi=16):
    """the pattern of csr (row_ptr, col_idx, ...) with nonzero integer values lo <= |v| < hi (fp16-exact up to 2048)"""
    rp, ci = csr[0], csr[1]
    rng = np.random.default_rng(seed)
    v = (np.where(rng.random(ci.size) < 0.5, -1.0, 1.0) * rng.integers(lo, hi, ci.size)).astype(np.float32)
    return rp, ci, v


def _scipy(shape, csr, scale=1.0):
    return sp.csr_matrix((csr[2].astype(np.float64) * scale, csr[1], csr[0]), shape=shape)


def _expected(shapeA, a, shapeB, b, scaleA=1.0):
    """A * B in float64 from the integer values (times scaleA, a power of two), after checking the exactness bound"""
    Ai, Bi = _scipy(shapeA, a), _scipy(shapeB, b)
    assert float((abs(Ai) @ abs(Bi)).max()) < 2 ** 24
    R = (Ai.astype(np.int64) @ Bi.astype(np.int64)).astype(np.float64)
    return R * scaleA


def _assert_exact(C, R):
    """C's values (fp32) equal R's at every position of C, and C stores every nonzero of R"""
    r, c, v = C.generate_coo()
    got = sp.csr_matrix((v.astype(np.float64), (r, c)), shape=R.shape)
    d = (got - R).tocoo()
    bad = d.data != 0
    assert not bad.any(), f"{int(bad.sum())} entries differ, first at {list(zip(d.row[bad][:4], d.col[bad][:4]))}: {d.data[bad][:4]}"


def _mult(B, shapeA, a, shapeB, b, scaleA=1.0, **kw):
    A = B.bmSpMatrix.from_csr(*shapeA, a[0], a[1], a[2] * scaleA)
    Bt = B.bmSpMatrix.from_csr(*shapeB, *b, transpose=True)
    C, info = B.bmSparse_mult(A, Bt, None, 0, True, 5, **kw)
    _assert_exact(C, _expected(shapeA, a, shapeB, b, scaleA))
    return C, info


def _square(gen):
    nr, nc, rp, ci, _ = gen
    return (nr, nc), (rp, ci)


# ------------------------------------------------------------------------------------------------------ scalar path (path 0)
@pytest.mark.parametrize("gen,fine", [("uniform_random", True), ("rmat", False), ("hub_row", False), ("paired_rows", False),
                                      ("poisson", False)])
def test_scalar_path(B, gen, fine):
    """the scalar NUMERIC pass: B's fine index (uniform random), the scan of B's block rows (R-MAT), one hub bucket, every block
    in two buckets, and Poisson's class-sorted pair lists"""
    G = B.generators
    src = {"uniform_random": lambda: G.uniform_random(4096, 16, seed=7), "rmat": lambda: G.rmat(12),
           "hub_row": lambda: _hub_row(*G.uniform_random(8192, 8, seed=9)), "paired_rows": lambda: _paired_rows(4096, 8, 10),
           "poisson": lambda: G.poisson5pt(64, 52)}[gen]()
    shape, pat = _square(src)
    p = _plan(shape, pat, shape, pat)
    assert _fine_chosen(p) == fine and p["auto_path"] == 0
    a, b = _ints(pat, 1), _ints(pat, 2)
    C, info = _mult(B, shape, a, shape, b)
    assert info.numeric_path == 0


# ------------------------------------------------------------------------------------------------------ MMA path (path 1)
@pytest.mark.parametrize("n,m,p,density", [(24, 24, 24, 0.2), (61, 45, 29, 0.15), (300, 200, 250, 0.05), (257, 513, 129, 0.3),
                                           (1000, 1000, 1000, 0.004), (64, 64, 64, 0.9)])
def test_mma_forced_random(B, n, m, p, density):
    """path 1 (mma.sync m16n8k8, fp32 accumulation) forced on the random shapes of test_gpu_spgemm.test_random, integer values"""
    a = _ints(random_csr(n, m, density, seed=n * 7 + m, empty_block_rows=(1,) if n > 24 else ()), 3)
    b = _ints(random_csr(m, p, density, seed=m * 13 + p, empty_block_rows=(0, 3) if m > 40 else ()), 4)
    C, info = _mult(B, (n, m), a, (m, p), b, numeric_path=1)
    assert info.numeric_path == 1


def test_mma_dense_block_kernel(B):
    """narrow rows of dense blocks: the dense-block kernel, chosen by the planner"""
    shape, pat = _square(B.generators.block_clustered(64))
    p = _plan(shape, pat, shape, pat)
    assert p["auto_path"] == 1 and p["max_words"] <= DENSE_MAX_WORDS
    C, info = _mult(B, shape, _ints(pat, 5), shape, _ints(pat, 6))
    assert info.numeric_path == 1


@pytest.mark.parametrize("accumulators", ["shared", "global"])
def test_mma_wide_rows(B, accumulators):
    """C rows spanning more than 1024 block columns: the generic MMA pass with the row's accumulators in shared memory (at most
    192 C blocks per row) or in global memory (more)"""
    if accumulators == "shared":
        a, b, sa, sb = random_csr(16, 64, 0.9, seed=5), _strided_b(64, 128, 17, 0.5, seed=6), (16, 64), (64, 8 * 128 * 17)
    else:
        a, b, sa, sb = random_csr(16, 64, 0.9, seed=3), random_csr(64, 8 * 1200, 0.5, seed=4), (16, 64), (64, 8 * 1200)
    p = _plan(sa, a, sb, b)
    assert p["max_words"] > DENSE_MAX_WORDS and (0 < p["max_c_row"] <= MMA_SHARED_CAP) == (accumulators == "shared")
    C, info = _mult(B, sa, _ints(a, 7), sb, _ints(b, 8), numeric_path=1)
    assert info.numeric_path == 1


def test_heavy_row_split(B, monkeypatch):
    """hub rows in their own launch (BMSP_SPGEMM_HEAVY lowered): block-clustered on the MMA path, R-MAT and uniform random on the
    scalar path"""
    G = B.generators
    shape, pat = _square(G.block_clustered(64))
    p = _plan(shape, pat, shape, pat)
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", str(p["max_cand"] // 4))
    assert int((p["cand"] >= p["max_cand"] // 4).sum()) > 0
    C, info = _mult(B, shape, _ints(pat, 9), shape, _ints(pat, 10))
    assert info.numeric_path == 1
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", "300")
    for gen in (G.rmat(11), G.uniform_random(3000, 16)):
        shape, pat = _square(gen)
        assert int((_plan(shape, pat, shape, pat)["cand"] >= 300).sum()) > 0
        C, info = _mult(B, shape, _ints(pat, 11), shape, _ints(pat, 12))
        assert info.numeric_path == 0


@pytest.mark.parametrize("path", [0, 1])
def test_block_row_shards(B, path):
    """brow_range shards: each shard's C holds exactly the rows of the full product it owns"""
    shape, pat = _square(B.generators.uniform_random(1024, 12, seed=11))
    a, b = _ints(pat, 13), _ints(pat, 14)
    A = B.bmSpMatrix.from_csr(*shape, *a)
    Bt = B.bmSpMatrix.from_csr(*shape, *b, transpose=True)
    R = _expected(shape, a, shape, b).tocsr()
    bounds = A.partition_block_rows(3, Bt)
    for i in range(3):
        r0, r1 = int(bounds[i]) * 8, min(int(bounds[i + 1]) * 8, shape[0])
        C, info = B.bmSparse_mult(A, Bt, brow_range=(int(bounds[i]), int(bounds[i + 1])), numeric_path=path)
        assert info.numeric_path == path
        Rs = R.copy()
        keep = np.zeros(shape[0], bool); keep[r0:r1] = True
        Rs = sp.diags(keep.astype(np.float64)) @ Rs
        _assert_exact(C, Rs)


@pytest.mark.parametrize("path", [0, 1])
def test_plan_numeric_after_set_values(B, path):
    """SpGEMMPlan.numeric() after both operands' values changed (set_values_csr): C's values are the new exact product"""
    shape, pat = _square(B.generators.poisson5pt(48, 40))
    a, b = _ints(pat, 15), _ints(pat, 16)
    A = B.bmSpMatrix.from_csr(*shape, *a)
    Bt = B.bmSpMatrix.from_csr(*shape, *b, transpose=True)
    plan = B.bmSparse_mult_plan(A, Bt, numeric_path=path)
    _assert_exact(plan.C, _expected(shape, a, shape, b))
    a2, b2 = _ints(pat, 17, 16, 64), _ints(pat, 18, 16, 64)
    A.set_values_csr(*a2)
    Bt.set_values_csr(*b2)
    plan.numeric()
    import torch
    torch.cuda.synchronize()
    _assert_exact(plan.C, _expected(shape, a2, shape, b2))
    plan.close()


# ------------------------------------------------------------------------------------------------------ value ranges
@pytest.mark.parametrize("path", [0, 1])
def test_subnormal_a_values(B, path):
    """A holds fp16 subnormals k * 2^-24 (k < 1024), B small integers: every product and sum is a multiple of 2^-24 below 1,
    exact in fp32; a tensor-core or conversion step that flushes subnormals to zero would lose them"""
    shape, pat = _square(B.generators.block_clustered(48))
    a, b = _ints(pat, 19, 1, 1024), _ints(pat, 20, 1, 8)
    assert np.all(np.abs(a[2]) < 1024)
    C, info = _mult(B, shape, a, shape, b, scaleA=2.0 ** -24, numeric_path=path)
    assert info.numeric_path == path


@pytest.mark.parametrize("path", [0, 1])
def test_values_near_2048(B, path):
    """A holds integers 2040 .. 2047 and 2048 (the top of fp16's unit-spaced range), B small integers: products up to 14 336"""
    shape, pat = _square(B.generators.block_clustered(48))
    a, b = _ints(pat, 21, 2040, 2049), _ints(pat, 22, 1, 8)
    C, info = _mult(B, shape, a, shape, b, numeric_path=path)
    assert info.numeric_path == path
