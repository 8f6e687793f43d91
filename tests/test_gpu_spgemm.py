"""GPU parity: bmSparse_mult through the C ABI vs the oracle.

Structure (keys, bmps, offsets) must be bit-exact.  Values: fp16 inputs, fp32 accumulation; tolerance as
BASELINE.json states it: <= 1e-3 relative to an exact (float64) product of the same fp16 inputs, with an
absolute floor of 1e-3 * sum|a||b| for cancelling sums."""
import ctypes

import numpy as np
import pytest
import torch

from tests.util import assert_structure_equal, hex_to_u64, load_golden, random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _mult_check(B, O, shapeA, csrA, shapeB, csrB, **kw):
    A = B.bmSpMatrix.from_csr(*shapeA, *csrA)
    Bt = B.bmSpMatrix.from_csr(*shapeB, *csrB, transpose=True)
    oA = O.csr_to_bmsp(*shapeA, *csrA); oB = O.csr_to_bmsp(*shapeB, *csrB, transposed=True)
    C, info = B.bmSparse_mult(A, Bt, None, 0, True, 5, **kw)
    exp = O.spgemm(oA, oB)
    k, b, o, v = C.download()
    assert_structure_equal((k, b, o), exp, "C")
    assert o.size == exp.block_num + 1 and int(o[-1]) == exp.nnz == C.nnz
    assert info.c_blocks == exp.block_num and info.c_nnz == exp.nnz
    mag = O.spgemm(O.OracleMatrix(oA.num_rows, oA.num_cols, oA.keys, oA.bmps, oA.offsets, np.abs(oA.values)),
                   O.OracleMatrix(oB.num_rows, oB.num_cols, oB.keys, oB.bmps, oB.offsets, np.abs(oB.values), True)).values
    err = np.abs(v.astype(np.float64) - exp.values)
    assert np.all(err <= 1e-3 * np.maximum(np.abs(exp.values), 1e-3 * mag) + 1e-30), f"max err {err.max()}"
    # tighter: fp32 accumulation of exact products
    assert np.all(err <= 2e-6 * mag + 1e-30)
    return C, info, exp


def test_pair_bitmap_kernel(B, oracle):
    rng = np.random.default_rng(0)
    n = 4096
    a = rng.integers(0, 2**64, n, dtype=np.uint64) & rng.integers(0, 2**64, n, dtype=np.uint64)
    bt = rng.integers(0, 2**64, n, dtype=np.uint64) & rng.integers(0, 2**64, n, dtype=np.uint64) & rng.integers(0, 2**64, n, dtype=np.uint64)
    a[:4] = [0, 2**64 - 1, 1, 2**63]; bt[:4] = [2**64 - 1, 2**64 - 1, 2**63, 1]
    # sparse A blocks (<= 8 cells) take the per-cell evaluation, the others the row-wise one
    for i in range(8, n // 2):
        k = int(rng.integers(1, 9))
        a[i] = np.bitwise_or.reduce(np.uint64(1) << rng.integers(0, 64, k).astype(np.uint64))
    out = np.empty(n, np.uint64)
    p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
    from bmsparse_spgemm_spmv_b200 import _lib as L
    L.check(L.lib().bmsp_debug_pair_bitmap(ctypes.c_int64(n), p(a), p(bt), p(out)))
    exp = np.array([oracle.pair_bitmap(int(x), int(y)) for x, y in zip(a, bt)], dtype=np.uint64)
    assert np.array_equal(out, exp)


def test_fixture_exact(B):
    g = load_golden("ragusa16.json")
    A = B.bmSpMatrix.from_coo(24, 24, g["A"]["rows"], g["A"]["cols"], g["A"]["vals"])
    Bt = B.bmSpMatrix.from_coo(24, 24, g["B"]["rows"], g["B"]["cols"], g["B"]["vals"], transpose=True)
    C, info = B.bmSparse_mult(A, Bt)
    k, b, o, v = C.download()
    assert np.array_equal(k, hex_to_u64(g["C_keys"]))
    assert np.array_equal(b, hex_to_u64(g["survey_C_bmps"]))
    assert o.tolist() == g["survey_C_offsets"] and C.nnz == 255 and C.block_num == 9
    r, c, vals = C.generate_coo()
    got = {(int(x), int(y)): float(z) for x, y, z in zip(r, c, vals)}
    exp = {(x, y): z for x, y, z in zip(g["C_coo"]["rows"], g["C_coo"]["cols"], g["C_coo"]["vals"])}
    assert got == exp


@pytest.mark.parametrize("path", [0, 1])
@pytest.mark.parametrize("n,m,p,density", [(24, 24, 24, 0.2), (61, 45, 29, 0.15), (300, 200, 250, 0.05), (257, 513, 129, 0.3),
                                           (1000, 1000, 1000, 0.004), (64, 64, 64, 0.9)])
def test_random(B, oracle, n, m, p, density, path):
    """path 0 = scalar lanes, path 1 = mma.sync m16n8k8 (forced on every density, also the sparse ones)"""
    a = random_csr(n, m, density, seed=n * 7 + m, empty_block_rows=(1,) if n > 24 else ())
    b = random_csr(m, p, density, seed=m * 13 + p, empty_block_rows=(0, 3) if m > 40 else ())
    C, info, exp = _mult_check(B, oracle, (n, m), a, (m, p), b, numeric_path=path)
    assert info.numeric_path == path


def test_generators_square(B, oracle):
    G = B.generators
    for gen in (lambda: G.poisson5pt(40, 36), lambda: G.block_clustered(96), lambda: G.uniform_random(2048, 16),
                lambda: G.rmat(10)):
        nr, nc, rp, ci, v = gen()
        C, info, exp = _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
        assert info.surviving_pairs <= info.candidate_pairs
        _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v), numeric_path=1 - info.numeric_path)


def test_poisson256_counts(B):
    """BASELINE config 1 shape on the GPU path: 88 260 C blocks / 846 852 nnz (SURVEY Appendix D)."""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(256, 256)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    C, info = B.bmSparse_mult(A, Bt)
    assert C.block_num == 88260 and C.nnz == 846852 and info.candidate_pairs == 199624
    # values: A*A of the 5-point stencil has integer entries -> exact
    import scipy.sparse as sp
    S = sp.csr_matrix((v, ci, rp), shape=(nr, nc)); R = (S @ S).tocoo()
    assert C.compare(R.row, R.col, R.data) == (0, 0, 0.0, 0.0)


def test_row_range_shards_concatenate(B, oracle):
    nr, nc, rp, ci, v = B.generators.uniform_random(1024, 12, seed=11)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    full = B.bmSparse_mult(A, Bt)[0].download()
    bounds = A.partition_block_rows(3, Bt)
    assert bounds[0] == 0 and bounds[-1] == A.num_block_rows and np.all(np.diff(bounds) >= 0)
    ks, bs, vs, offs, base = [], [], [], [], 0
    for i in range(3):
        k, b, o, v_ = B.bmSparse_mult(A, Bt, brow_range=(int(bounds[i]), int(bounds[i + 1])))[0].download()
        ks.append(k); bs.append(b); vs.append(v_); offs.append(o[:-1] + np.uint64(base)); base += int(o[-1])
    assert np.array_equal(np.concatenate(ks), full[0]) and np.array_equal(np.concatenate(bs), full[1])
    assert np.array_equal(np.concatenate(offs), full[2][:-1]) and base == int(full[2][-1])
    assert np.allclose(np.concatenate(vs), full[3], rtol=1e-6, atol=1e-7)


def test_chained_product_via_block_transpose(B, oracle):
    """(A*A)*A with the fp32 product turned into the next fp16 operand on the device"""
    nr, nc, rp, ci, v = B.generators.poisson5pt(24, 20)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); At = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    C1, _ = B.bmSparse_mult(A, At)
    # plain fp32 -> plain fp16 (two transposes), then multiply by A again
    C1h = C1.block_transpose(torch.float16).block_transpose(torch.float16)
    C2, _ = B.bmSparse_mult(C1h, At)
    import scipy.sparse as sp
    S = sp.csr_matrix((v, ci, rp), shape=(nr, nc)); R = (S @ S @ S).tocoo()
    a, b, mean, mx = C2.compare(R.row, R.col, R.data)
    assert (a, b) == (0, 0) and mx == 0.0      # integers up to 6*4^2.. exact in fp16/fp32


def test_heavy_row_split(B, oracle, monkeypatch):
    """hub rows run in their own launch (1024-thread CTAs on a side stream, heaviest first): same structure bit for bit,
    values within the fp32-accumulation tolerance.  The threshold is lowered so that small inputs exercise the split."""
    G = B.generators
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", "300")
    for gen in (lambda: G.rmat(11), lambda: G.uniform_random(3000, 16), lambda: G.poisson5pt(40, 40)):
        nr, nc, rp, ci, v = gen()
        C, info, exp = _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
        # sharded range with the split active
        A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
        nbr = A.num_block_rows
        C2, _ = B.bmSparse_mult(A, Bt, brow_range=(nbr // 3, nbr))
        k, b, o, vals = C.download(); k2, b2, o2, vals2 = C2.download()
        first = int(np.searchsorted(k >> np.uint64(32), nbr // 3))
        assert np.array_equal(k[first:], k2) and np.array_equal(b[first:], b2)


def test_full_size_u1m_properties(B):
    """BASELINE config 3 at full size (uniform-random 1M x 1M, 16 nnz/row, A*A): size-independent properties.
    (i) the structure counts the reference's own CUDA operator produced on the same input (profiles/r1_compare_baselines.json);
    (ii) sum of all C entries = (1^T A)(A 1), evaluated in fp64 from A alone;  (iii) C x = A (A x) with both sides through the
    SpMV kernels (C is an fp32 bmSparse matrix, A fp16) -- ties the two operators together;  (iv) keys strictly ascending and
    offsets = exclusive scan of popcount(bitmaps)."""
    G = B.generators
    nr, nc, rp, ci, v = G.uniform_random(1_000_000, 16, seed=2)
    d = lambda a: torch.from_numpy(a).cuda()
    A = B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v)); Bt = B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v), transpose=True)
    C, info = B.bmSparse_mult(A, Bt)
    assert (C.block_num, C.nnz) == (253900089, 255969153)
    assert info.candidate_pairs == 2045965407 and info.surviving_pairs == 255971715
    # (ii)
    v64 = v.astype(np.float64)
    rowsum = np.add.reduceat(v64, rp[:-1].astype(np.int64))
    colsum = np.bincount(ci, weights=v64, minlength=nc)
    exact = float(colsum @ rowsum)
    scale = float(np.bincount(ci, weights=np.abs(v64), minlength=nc) @ np.add.reduceat(np.abs(v64), rp[:-1].astype(np.int64)))
    got = float(C.values.sum(dtype=torch.float64).item())
    assert abs(got - exact) <= 1e-6 * scale, (got, exact, scale)
    # (iv)
    k = C.keys
    assert bool((k[1:] > k[:-1]).all())
    bm = C.bmps
    pc = torch.zeros_like(bm)
    t = bm.clone()
    for _ in range(64):          # popcount of int64 bit patterns without uint64 support
        pc += t & 1
        t = (t >> 1) & 0x7FFFFFFFFFFFFFFF
    off = C.offsets
    assert int(off[0]) == 0 and int(off[-1]) == C.nnz and torch.equal(off[1:] - off[:-1], pc)
    del pc, t
    # (iii)
    x = d(G.x_vector(nc))
    y1 = B.bmSparse_SpMV(A, B.bmSparse_SpMV(A, x))
    y2 = B.bmSparse_SpMV(C, x)
    tol = 1e-4 * float(y1.abs().max())
    assert float((y1 - y2).abs().max()) <= tol


def test_empty_block_row_range_multiplies_nothing(B):
    """ADVICE r1: brow_range=(0, 0) -- a shard that owns no block rows -- used to mean "all rows"."""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(48, 40)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    full, _ = B.bmSparse_mult(A, Bt)
    for rng_ in ((0, 0), (5, 5), (A.num_block_rows, A.num_block_rows)):
        C, info = B.bmSparse_mult(A, Bt, brow_range=rng_)
        assert C.block_num == 0 and C.nnz == 0 and info.c_blocks == 0
        assert C.download()[2].tolist() == [0]
    C, _ = B.bmSparse_mult(A, Bt, brow_range=None)
    assert C.block_num == full.block_num > 0
