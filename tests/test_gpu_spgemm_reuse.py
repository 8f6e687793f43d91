"""GPU: SpGEMM plans (bmSparse_mult_plan) recompute C's values after the operands' values change.

Every case is built like tests/test_gpu_spgemm_paths.py and asserts first, in numpy, that it takes the kernel path it is named for.
Then: plan on values v1, new values v2 on A and B through set_values_csr, plan.numeric().  C's structure must be bit-identical to
what the plan made and to a fresh bmSparse_mult on v2; C's values must match the oracle with _mult_check's tolerances and the fresh
product within 2e-6 * sum|a||b| (bit for bit on the dense-block kernel, whose accumulators are lane-private); a second numeric()
with nothing changed must leave them there."""
import numpy as np
import pytest
import torch

from tests.test_gpu_spgemm_paths import DENSE_MAX_WORDS, MMA_SHARED_CAP, _fine_chosen, _plan, _strided_b
from tests.util import assert_structure_equal, random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _new_values(n, seed):
    v = np.random.default_rng(seed).uniform(-1, 1, n).astype(np.float16).astype(np.float32)
    v[v == 0] = 0.25
    return v


def _structure(B, C):
    """keys, bitmaps, offsets, block_row_ptr, block_col and block_row_val of C, on the host"""
    from bmsparse_spgemm_spmv_b200.matrix import _alias
    v = C._view()
    rvb = _alias(v.block_row_val, v.num_block_rows + 1, "<i4", torch.int32, C)
    k, b, o, _ = C.download()
    return [k, b, o, C.block_row_ptr.cpu().numpy(), C.block_col.cpu().numpy(), rvb.cpu().numpy()]


def _same_structure(s1, s2):
    return all(np.array_equal(x, y) for x, y in zip(s1, s2))


def _oracle_values(O, C, shapeA, csrA, shapeB, csrB):
    """C against the oracle product of the CSR inputs, with _mult_check's tolerances; returns sum|a||b| per value"""
    oA = O.csr_to_bmsp(*shapeA, *csrA); oB = O.csr_to_bmsp(*shapeB, *csrB, transposed=True)
    exp = O.spgemm(oA, oB)
    k, b, o, v = C.download()
    assert_structure_equal((k, b, o), exp, "C")
    mag = O.spgemm(O.OracleMatrix(oA.num_rows, oA.num_cols, oA.keys, oA.bmps, oA.offsets, np.abs(oA.values)),
                   O.OracleMatrix(oB.num_rows, oB.num_cols, oB.keys, oB.bmps, oB.offsets, np.abs(oB.values), True)).values
    err = np.abs(v.astype(np.float64) - exp.values)
    assert np.all(err <= 1e-3 * np.maximum(np.abs(exp.values), 1e-3 * mag) + 1e-30), f"max err {err.max()}"
    assert np.all(err <= 2e-6 * mag + 1e-30)
    return mag


def _reuse_check(B, O, shapeA, a, shapeB, b, exact=False, brow_range=None, **kw):
    """the checks of the module docstring; returns the plan (already updated to v2)"""
    A = B.bmSpMatrix.from_csr(*shapeA, *a)
    Bt = B.bmSpMatrix.from_csr(*shapeB, *b, transpose=True)
    plan = B.bmSparse_mult_plan(A, Bt, VERBOSE=True, brow_range=brow_range, **kw)
    C = plan.C
    s1 = _structure(B, C)
    a2 = (a[0], a[1], _new_values(a[1].size, 101)); b2 = (b[0], b[1], _new_values(b[1].size, 202))
    A.set_values_csr(*a2); Bt.set_values_csr(*b2)
    plan.numeric()
    torch.cuda.synchronize()
    fresh, info = B.bmSparse_mult(A, Bt, brow_range=brow_range, **kw)
    assert info.numeric_path == plan.info.numeric_path
    s2 = _structure(B, C)
    assert _same_structure(s1, s2), "numeric() changed C's structure"
    assert _same_structure(s2, _structure(B, fresh)), "C's structure differs from a fresh product's"
    got = C.values.cpu().numpy().astype(np.float64); ref = fresh.values.cpu().numpy().astype(np.float64)
    if brow_range is None:
        mag = _oracle_values(O, C, shapeA, a2, shapeB, b2)
    else:       # a shard: the oracle's full product has other rows; the bound's scale from the fresh shard's own magnitudes
        mag = np.abs(ref) + 1.0
    if exact:
        assert np.array_equal(got, ref)
    assert np.all(np.abs(got - ref) <= 2e-6 * mag + 1e-30)
    plan.numeric()
    torch.cuda.synchronize()
    again = C.values.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(again - ref) <= 2e-6 * mag + 1e-30)
    assert _same_structure(s1, _structure(B, C))
    return plan


def _poisson(B):
    nr, nc, rp, ci, v = B.generators.poisson5pt(64, 52)
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    assert p["avg_cand"] <= 96 and 16 * p["max_words"] <= 8192 and p["dA"] >= 4.0 and p["auto_path"] == 0
    return (nr, nc), (rp, ci, v)


def _rmat_split(B, monkeypatch):
    nr, nc, rp, ci, v = B.generators.rmat(11)
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    heavy = 300
    assert p["max_cand"] >= 4 * heavy and int((p["cand"] >= heavy).sum()) > 0       # the split is active
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", str(heavy))
    return (nr, nc), (rp, ci, v)


def test_poisson_class_sorted(B, oracle):
    """row groups, FILL's class-sorted pair list, scalar NUMERIC with 8 lanes per pair: the plan keeps the pair list"""
    sh, a = _poisson(B)
    plan = _reuse_check(B, oracle, sh, a, sh, a)
    assert plan.info.numeric_path == 0 and plan.nbytes >= 8 * plan.info.surviving_pairs


def test_uniform_random_fine_index(B, oracle):
    """B's fine index: the plan keeps no pair list"""
    nr, nc, rp, ci, v = B.generators.uniform_random(4096, 16, seed=7)
    assert _fine_chosen(_plan((nr, nc), (rp, ci), (nr, nc), (rp, ci)))
    plan = _reuse_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
    assert plan.info.numeric_path == 0 and plan.nbytes < 8 * plan.info.surviving_pairs


def test_rmat_scan(B, oracle):
    """R-MAT: the fine index is refused, the scalar pass walks the candidate scan's pair list, which the plan keeps"""
    nr, nc, rp, ci, v = B.generators.rmat(12)
    assert not _fine_chosen(_plan((nr, nc), (rp, ci), (nr, nc), (rp, ci)))
    plan = _reuse_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
    assert plan.info.numeric_path == 0 and plan.nbytes >= 8 * plan.info.surviving_pairs


def test_block_clustered_dense_kernel(B, oracle):
    """narrow rows of dense blocks: the dense-block kernel, lane-private accumulators -- bit-identical to a fresh product"""
    nr, nc, rp, ci, v = B.generators.block_clustered(64)
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    assert p["auto_path"] == 1 and p["max_words"] <= DENSE_MAX_WORDS
    plan = _reuse_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v), exact=True)
    assert plan.info.numeric_path == 1 and plan.nbytes < 8 * plan.info.surviving_pairs


def test_mma_wide_rows_shared(B, oracle):
    """the generic MMA pass with the row's accumulators in shared memory"""
    a = random_csr(16, 64, 0.9, seed=5)
    b = _strided_b(64, 128, 17, 0.5, seed=6)
    sa, sb = (16, 64), (64, 8 * 128 * 17)
    p = _plan(sa, a, sb, b)
    assert p["max_words"] > DENSE_MAX_WORDS and 0 < p["max_c_row"] <= MMA_SHARED_CAP
    plan = _reuse_check(B, oracle, sa, a, sb, b, numeric_path=1)
    assert plan.nbytes < 8 * plan.info.surviving_pairs


def test_mma_global_fallback(B, oracle):
    """more than 192 C blocks in a row: the MMA pass accumulates in global memory, and every numeric() zeroes C first"""
    a = random_csr(16, 64, 0.9, seed=3)
    b = random_csr(64, 8 * 1200, 0.5, seed=4)
    p = _plan((16, 64), a, (64, 8 * 1200), b)
    assert p["max_words"] > DENSE_MAX_WORDS and p["max_c_row"] > MMA_SHARED_CAP
    _reuse_check(B, oracle, (16, 64), a, (64, 8 * 1200), b, numeric_path=1)


def test_heavy_row_split(B, oracle, monkeypatch):
    """hub rows on the plan's side stream, light rows on the caller's"""
    sh, a = _rmat_split(B, monkeypatch)
    _reuse_check(B, oracle, sh, a, sh, a)


def test_empty_block_rows(B, oracle):
    a = random_csr(300, 200, 0.05, seed=300 * 7 + 200, empty_block_rows=(1,))
    b = random_csr(200, 250, 0.05, seed=200 * 13 + 250, empty_block_rows=(0, 3))
    for path in (0, 1):
        _reuse_check(B, oracle, (300, 200), a, (200, 250), b, numeric_path=path)


@pytest.mark.parametrize("rng_", ["shard", "empty"])
def test_brow_range(B, oracle, rng_):
    nr, nc, rp, ci, v = B.generators.uniform_random(1024, 12, seed=11)
    nbr = (nr + 7) // 8
    r = (nbr // 3, nbr) if rng_ == "shard" else (5, 5)
    plan = _reuse_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v), brow_range=r)
    assert (plan.C.block_num == 0) == (rng_ == "empty")


@pytest.mark.parametrize("case", ["poisson", "heavy_split"])
def test_cuda_graph_replay(B, oracle, monkeypatch, case):
    """numeric() captured into a CUDA graph; new values; replay"""
    sh, a = _poisson(B) if case == "poisson" else _rmat_split(B, monkeypatch)
    A = B.bmSpMatrix.from_csr(*sh, *a); Bt = B.bmSpMatrix.from_csr(*sh, *a, transpose=True)
    plan = B.bmSparse_mult_plan(A, Bt)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())      # the plan's first NUMERIC pass, enqueued by its creation, makes C's offsets absolute
    with torch.cuda.stream(s):
        plan.numeric()
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        plan.numeric()
    a2 = (a[0], a[1], _new_values(a[1].size, 303))
    A.set_values_csr(*a2); Bt.set_values_csr(*a2)
    g.replay()
    torch.cuda.synchronize()
    _oracle_values(oracle, plan.C, sh, a2, sh, a2)


def test_spmv_on_reused_product(B, oracle):
    """an SpMV planned on C before numeric() gives what an SpMV on a fresh product gives (dense-block kernel: C bit-identical)"""
    nr, nc, rp, ci, v = B.generators.block_clustered(64)
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v); Bt = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, transpose=True)
    plan = B.bmSparse_mult_plan(A, Bt)
    x = torch.from_numpy(B.generators.x_vector(nc)).cuda()
    B.bmSparse_SpMV(plan.C, x)                     # builds C's SpMV plan
    v2 = _new_values(ci.size, 404)
    A.set_values_csr(rp, ci, v2); Bt.set_values_csr(rp, ci, v2)
    plan.numeric()
    y = B.bmSparse_SpMV(plan.C, x)
    fresh, _ = B.bmSparse_mult(A, Bt)
    assert torch.equal(y, B.bmSparse_SpMV(fresh, x))
