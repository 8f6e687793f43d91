"""GPU parity of the streaming SpMV kernel's bitmap palette (matrices with at most 256 distinct bitmaps) and of its fallback.

Every case is checked against the oracle with the tolerance of test_gpu_spmv._spmv_check, and bit for bit against the one-CTA-per-tile
kernel on the same matrix (BMSP_SPMV_KERNEL=1, read when a matrix is planned): both run the same per-half arithmetic in the same order.
Each input states in numpy which path it takes: its number of distinct bitmaps, and light rows (the row-tiled path, 64-block-row tiles,
which is the streaming kernel's)."""
import numpy as np
import pytest
import torch

from tests.test_gpu_spmv import _spmv_check

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _distinct_bitmaps(oracle, nr, nc, rp, ci, v):
    return np.unique(oracle.csr_to_bmsp(nr, nc, rp, ci, v).bmps).size


def _assert_light_rows(oracle, nr, nc, rp, ci, v):
    """the plan's choice (spmv.cu plan_spmv / plan_tiles): >= 2.5 values per block is the row-tiled path, and an average block
    row under 320 bytes (bitmaps, x offsets, ~x lines, fp16 values) gives 64-block-row tiles, which run the streaming kernel"""
    m = oracle.csr_to_bmsp(nr, nc, rp, ci, v)
    nblk, nnz, nbr = m.bmps.size, int(rp[-1]), (nr + 7) // 8
    assert nnz / nblk >= 2.5
    assert (nblk * 26 + nnz * 2) / nbr + 8 <= 320


def _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x, dtype=torch.float16, x_half=False):
    xt = torch.tensor(x, device="cuda")
    if x_half:
        xt = xt.half()
    M = _spmv_check(B, oracle, nr, nc, rp, ci, v, x, dtype=dtype, x_half=x_half)
    y_stream = B.bmSparse_SpMV(M, xt)
    with monkeypatch.context() as mp:
        mp.setenv("BMSP_SPMV_KERNEL", "1")
        T = _spmv_check(B, oracle, nr, nc, rp, ci, v, x, dtype=dtype, x_half=x_half)
        y_tile = B.bmSparse_SpMV(T, xt)
    torch.cuda.synchronize()
    assert torch.equal(y_stream, y_tile)


def _diagonals_csr(n, offsets, seed):
    """n x n matrix with the given diagonals (fp16-exact values)"""
    rows, cols = [], []
    for d in offsets:
        r = np.arange(max(0, -d), min(n, n - d))
        rows.append(r); cols.append(r + d)
    r = np.concatenate(rows); c = np.concatenate(cols)
    o = np.lexsort((c, r)); r, c = r[o], c[o]
    v = np.random.default_rng(seed).uniform(-1, 1, r.size).astype(np.float16).astype(np.float32)
    v[v == 0] = 0.5
    rp = np.zeros(n + 1, np.int64); np.cumsum(np.bincount(r, minlength=n), out=rp[1:])
    return n, n, rp.astype(np.int32), c.astype(np.int32), v


def _patterned_blocks_csr(nbr, npat, seed):
    """nbr block rows of two blocks each: a diagonal block and a block 3 block columns to the right (wrapping) whose bitmap is pattern
    i % npat of npat distinct 64-bit masks of 12 cells -- npat + 1 distinct bitmaps"""
    rng = np.random.default_rng(seed)
    pats = set()
    while len(pats) < npat:
        cells = tuple(sorted(rng.choice(64, 12, replace=False).tolist()))
        if cells != tuple(9 * i for i in range(8)):
            pats.add(cells)
    pats = sorted(pats)
    n = nbr * 8
    rows, cols = [np.arange(n)], [np.arange(n)]
    for br in range(nbr):
        cells = np.array(pats[br % npat])
        bc = (br + 3) % nbr
        rows.append(br * 8 + cells // 8); cols.append(bc * 8 + cells % 8)
    r = np.concatenate(rows); c = np.concatenate(cols)
    o = np.lexsort((c, r)); r, c = r[o], c[o]
    v = rng.uniform(-1, 1, r.size).astype(np.float16).astype(np.float32)
    v[v == 0] = 0.5
    rp = np.zeros(n + 1, np.int64); np.cumsum(np.bincount(r, minlength=n), out=rp[1:])
    return n, n, rp.astype(np.int32), c.astype(np.int32), v


def test_poisson_not_a_tile_multiple(B, oracle, monkeypatch):
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(300, 221)          # 66300 rows: 8287.5 block rows, 129.5 tiles; m = 300 is no multiple of 8
    assert nr % (64 * 8) != 0
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) <= 256
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, G.x_vector(nc))


def test_band_generic_shapes(B, oracle, monkeypatch):
    """diagonals -2, 0, +3, +11: no half of any block is a diagonal, a tridiagonal or a single cell everywhere -- the bit walk"""
    nr, nc, rp, ci, v = _diagonals_csr(50000, (-2, 0, 3, 11), seed=3)
    nd = _distinct_bitmaps(oracle, nr, nc, rp, ci, v)
    assert 4 <= nd <= 16
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    x = np.random.default_rng(2).uniform(-1, 1, nc).astype(np.float32)
    _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x)


@pytest.mark.parametrize("npat", [255, 256])
def test_palette_limit(B, oracle, monkeypatch, npat):
    """256 distinct bitmaps: the largest palette; 257: more than a palette holds, the streaming kernel's bitmap layout"""
    nr, nc, rp, ci, v = _patterned_blocks_csr(3000, npat, seed=npat)
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) == npat + 1
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    x = np.random.default_rng(4).uniform(-1, 1, nc).astype(np.float32)
    _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x)


def test_fp32_values_and_fp16_x(B, oracle, monkeypatch):
    G = B.generators
    for nr, nc, rp, ci, v in (G.poisson5pt(200, 136), _diagonals_csr(20000, (-2, 0, 3, 11), seed=5)):
        assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) <= 256
        _assert_light_rows(oracle, nr, nc, rp, ci, v)
        x = G.x_vector(nc)
        _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x, dtype=torch.float32)
        _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x, x_half=True)
        _check_both_kernels(B, oracle, monkeypatch, nr, nc, rp, ci, v, x, dtype=torch.float32, x_half=True)


def test_host_pipeline_on_palette_matrix(B, oracle):
    """bmsp_spmv_host (row-range launches of the streaming kernel, chunked) == bmsp_spmv bit for bit"""
    nr, nc, rp, ci, v = _diagonals_csr(400000, (-2, 0, 3, 11), seed=6)
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) <= 256
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    for xdt in (torch.float32, torch.float16):
        xh = torch.from_numpy(B.generators.x_vector(nc)).to(xdt).pin_memory()
        ref = B.bmSparse_SpMV(M, xh.cuda()).cpu()
        yh = torch.full((nr,), 7.0).pin_memory()
        for it in range(3):           # eager, captured as a graph, replayed
            yh.fill_(7.0)
            B.bmSparse_SpMV_host(M, xh, yh)
            torch.cuda.synchronize()
            assert torch.equal(yh, ref), (xdt, it)
