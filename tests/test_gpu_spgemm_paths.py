"""GPU parity of the SpGEMM kernel paths that the planner in spgemm.cu selects from the operands.

Every case first evaluates the planner's own rules in numpy, from the CSR inputs, and asserts that the case takes the path it is
named for; then it runs the product through the same check as tests/test_gpu_spgemm.py (structure bit-exact against the oracle,
values within the fp32-accumulation tolerance)."""
import numpy as np
import pytest
import scipy.sparse as sp

from tests.test_gpu_spgemm import _mult_check
from tests.util import random_csr

pytestmark = pytest.mark.gpu

MMA_SHARED_CAP = 192      # C blocks per row that the generic MMA pass accumulates in shared memory
DENSE_MAX_WORDS = 32      # the dense-block kernel takes rows whose bit set spans at most 32 words (1024 block columns)


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _blocks(shape, csr):
    """block row, block column and kmask (inner rows present, one bit each) of every 8x8 block, in key order"""
    rp, ci = csr[0], csr[1]
    r = np.repeat(np.arange(shape[0], dtype=np.int64), np.diff(rp))
    nbc = (shape[1] + 7) // 8
    key = (r // 8) * nbc + ci.astype(np.int64) // 8
    u, inv = np.unique(key, return_inverse=True)
    kmask = np.zeros(u.size, np.int64)
    np.bitwise_or.at(kmask, inv, np.int64(1) << (r % 8))
    return u // nbc, u % nbc, kmask


def _plan(shapeA, csrA, shapeB, csrB):
    """the quantities bmsp_spgemm plans from, for C = A * B"""
    abr, abc, _ = _blocks(shapeA, csrA)
    bbr, bbc, bkm = _blocks(shapeB, csrB)
    nbrA, nbrB = (shapeA[0] + 7) // 8, (shapeB[0] + 7) // 8
    cnt = np.bincount(bbr, minlength=nbrB)
    jmin = np.full(nbrB, np.iinfo(np.int64).max); np.minimum.at(jmin, bbr, bbc)
    jmax = np.full(nbrB, -1, np.int64); np.maximum.at(jmax, bbr, bbc)
    # per A block row: candidate pairs and the span of its C bit set, over the B block rows its A blocks touch
    live = cnt[abc] > 0
    cand = np.bincount(abr, weights=cnt[abc], minlength=nbrA).astype(np.int64)
    rmin = np.full(nbrA, np.iinfo(np.int64).max); np.minimum.at(rmin, abr[live], jmin[abc[live]])
    rmax = np.full(nbrA, -1, np.int64); np.maximum.at(rmax, abr[live], jmax[abc[live]])
    has = rmax >= 0
    words = np.where(has, ((rmax - (np.where(has, rmin, 0) & ~31)) >> 5) + 1, 0)
    # C's blocks: the boolean product of the patterns
    pat = lambda shape, csr: sp.csr_matrix((np.ones(csr[1].size), csr[1], csr[0]), shape=shape)
    Cp = (pat(shapeA, csrA) @ pat(shapeB, csrB)).tocoo()
    nbcC = (shapeB[1] + 7) // 8
    cblk = np.unique((Cp.row.astype(np.int64) // 8) * nbcC + Cp.col // 8)
    c_row = np.bincount(cblk // nbcC, minlength=nbrA)
    dA = csrA[1].size / max(abr.size, 1); dB = csrB[1].size / max(bbr.size, 1)
    # fine index of B: bucket (k, t) = the blocks of B's block row k that have a value in inner row 8k + t
    per_row = np.zeros(nbrB * 8, np.int64)
    for t in range(8):
        np.add.at(per_row, bbr * 8 + t, (bkm >> t) & 1)
    total = int(per_row.sum())
    return dict(cand=cand, max_cand=int(cand.max(initial=0)), max_words=int(words.max(initial=0)), words=words,
                max_c_row=int(c_row.max(initial=0)), c_row=c_row, dA=dA, dB=dB,
                avg_cand=(abr.size / max(nbrA, 1)) * (bbr.size / max(nbrB, 1)),
                auto_path=int(dA * dB / 8.0 >= 40.0),
                fine_total=total, fine_longest=int(per_row.max(initial=0)), fine_mean=total / max(nbrB * 8, 1), b_nblk=int(bbr.size))


def _fine_chosen(p):
    """spgemm.cu's automatic rule for building B's fine index"""
    if not (p["dB"] <= 2.0 and p["dA"] <= 4.0):
        return False
    even = p["fine_longest"] <= 32.0 * max(p["fine_mean"], 1.0) or p["fine_longest"] <= 512
    return p["fine_total"] <= 1.5 * p["b_nblk"] and even


def _strided_b(rows, nbc, stride, density, seed):
    """rows x (8 * nbc * stride) columns whose values sit in every stride-th block column only"""
    rp, ci, v = random_csr(rows, 8 * nbc, density, seed=seed)
    return rp, ((ci // 8) * stride * 8 + ci % 8).astype(np.int32), v


def test_mma_path_wide_rows_shared_accumulators(B, oracle):
    """C rows spanning more than 1024 block columns with at most 192 C blocks each: the generic MMA pass, with the row's
    dense accumulators in shared memory"""
    a = random_csr(16, 64, 0.9, seed=5)
    b = _strided_b(64, 128, 17, 0.5, seed=6)
    sa, sb = (16, 64), (64, 8 * 128 * 17)
    p = _plan(sa, a, sb, b)
    assert p["max_words"] > DENSE_MAX_WORDS and 0 < p["max_c_row"] <= MMA_SHARED_CAP
    C, info, exp = _mult_check(B, oracle, sa, a, sb, b, numeric_path=1)
    assert info.numeric_path == 1


def test_mma_path_wide_rows_fall_back(B, oracle):
    """a block row of C with more blocks than the dense-accumulator cap (192) must take the global fallback"""
    a = random_csr(16, 64, 0.9, seed=3)
    b = random_csr(64, 8 * 1200, 0.5, seed=4)
    p = _plan((16, 64), a, (64, 8 * 1200), b)
    assert p["max_words"] > DENSE_MAX_WORDS and p["max_c_row"] > MMA_SHARED_CAP
    _mult_check(B, oracle, (16, 64), a, (64, 8 * 1200), b, numeric_path=1)


def test_mma_path_heavy_row_split(B, oracle, monkeypatch):
    """narrow rows of dense blocks go to the dense-block kernel, except when the heavy-row split is active: then the generic MMA
    pass runs"""
    nr, nc, rp, ci, v = B.generators.block_clustered(64)
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    assert p["auto_path"] == 1 and p["max_words"] <= DENSE_MAX_WORDS
    heavy = p["max_cand"] // 4
    assert heavy > 0 and int((p["cand"] >= heavy).sum()) > 0
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", str(heavy))
    C, info, exp = _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
    assert info.numeric_path == 1


def _hub_row(n, nc, rp, ci, v):
    """a square CSR matrix with row 0 replaced by one value in every block column: one bucket of n / 8 entries"""
    rows = [np.arange(0, nc, 8, dtype=np.int32)] + [ci[rp[i]:rp[i + 1]] for i in range(1, n)]
    rp2 = np.zeros(n + 1, np.int64); np.cumsum([r.size for r in rows], out=rp2[1:])
    return n, nc, rp2.astype(np.int32), np.concatenate(rows), np.resize(v, int(rp2[-1]))


def _paired_rows(n, k, seed):
    """rows 2p and 2p + 1 hold the same k columns, and the four pairs of a block row use disjoint block columns (j = 4r + p % 4):
    every block has exactly two values, in two inner rows -- each block sits in two buckets"""
    rng = np.random.default_rng(seed)
    nbc = n // 8
    rows = []
    for p in range(n // 2):
        j = 4 * np.sort(rng.choice(nbc // 4, k, replace=False)) + p % 4
        c = (8 * j + rng.integers(0, 8, k)).astype(np.int32)
        rows += [c, c]
    rp = np.zeros(n + 1, np.int64); np.cumsum([r.size for r in rows], out=rp[1:])
    v = rng.uniform(-1, 1, int(rp[-1])).astype(np.float16).astype(np.float32)
    v[v == 0] = 0.25
    return n, n, rp.astype(np.int32), np.concatenate(rows), v


@pytest.mark.parametrize("gen,fine", [("uniform_random", True), ("rmat", False), ("hub_row", False), ("paired_rows", False)])
def test_fine_index_rule(B, oracle, gen, fine):
    """B's fine index is built exactly when the automatic rule says so; both walks give the oracle's product.  The cases that do
    not build it each fail one part of the rule: values per block (R-MAT), bucket evenness (one hub bucket), replication (every
    block in two buckets)"""
    G = B.generators
    nr, nc, rp, ci, v = {"uniform_random": lambda: G.uniform_random(4096, 16, seed=7), "rmat": lambda: G.rmat(12),
                         "hub_row": lambda: _hub_row(*G.uniform_random(8192, 8, seed=9)), "paired_rows": lambda: _paired_rows(4096, 8, 10)}[gen]()
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    dense_ok = p["dB"] <= 2.0 and p["dA"] <= 4.0
    even = p["fine_longest"] <= 32.0 * max(p["fine_mean"], 1.0) or p["fine_longest"] <= 512
    replicates = p["fine_total"] > 1.5 * p["b_nblk"]
    if gen == "uniform_random":
        assert dense_ok and even and not replicates
    elif gen == "rmat":                       # R-MAT's hub blocks: more than two values per block of B on average
        assert not dense_ok
    elif gen == "hub_row":                    # one bucket of 1024 entries against a mean of about 8
        assert dense_ok and not even and not replicates
    else:
        assert dense_ok and even and replicates
    assert _fine_chosen(p) == fine
    C, info, exp = _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
    assert info.numeric_path == 0 and info.surviving_pairs <= info.candidate_pairs == int(p["cand"].sum())


def test_poisson_row_groups_class_sorted(B, oracle):
    """a stencil product: 16 block rows per work item, and FILL leaves each group's pair list sorted by pair class for the
    8-lanes-per-pair NUMERIC pass"""
    nr, nc, rp, ci, v = B.generators.poisson5pt(64, 52)
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    assert p["avg_cand"] <= 96 and 16 * p["max_words"] <= 8192           # groups of 16 rows, 128 threads per CTA
    assert p["dA"] >= 4.0 and p["auto_path"] == 0                           # 8 lanes per pair, scalar NUMERIC: the class sort is on
    grp = np.add.reduceat(p["cand"], np.arange(0, p["cand"].size, 16))
    assert grp.max() <= 4 * 128                                               # every group's pairs fit the sort's registers
    C, info, exp = _mult_check(B, oracle, (nr, nc), (rp, ci, v), (nr, nc), (rp, ci, v))
    assert info.numeric_path == 0 and info.candidate_pairs == int(p["cand"].sum())
