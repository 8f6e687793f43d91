"""Row shapes of the streaming SpMV kernel (spmv.cu, shape_scan_kernel): palette matrices whose staged block rows have at most
SHAPE_MAX distinct block-word sequences stream no per-block words.  Every case asserts the layout the plan chose through
bmsp_debug_spmv_shapes and runs in exact arithmetic (integer values and x, test_gpu_spmv_exact's harness: y == scipy's float64
product bit for bit, nothing written around y), on the streaming kernel and on the one-CTA-per-tile kernel (BMSP_SPMV_KERNEL=1),
which runs the same per-row arithmetic and must give the same y."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_gpu_device_memory import _run as _pool_run, pool  # noqa: F401  (pool is a fixture)
from tests.test_gpu_spmv_exact import (DT_IDS, DTYPES, _band, _band_plus_heavy_row, _buffers, _csr, _exact,
                                       _from_blocks, _poisson, _random_bitmaps, _reference, _scattered, _values, _x, plan_info)
from tests.test_gpu_spmv_halo import _check_halo, _shapes

pytestmark = pytest.mark.gpu

SHAPE_MAX = 128          # distinct shapes per matrix (spmv.cu)


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def shapes(M):
    """(shapes, table words) of M's plan; (-1, -1) when it streams block words or runs another kernel"""
    from bmsparse_spgemm_spmv_b200 import _lib as L
    from bmsparse_spgemm_spmv_b200.matrix import _stream_ptr
    n, w = C.c_int32(), C.c_int32()
    L.check(L.lib().bmsp_debug_spmv_shapes(M._h, C.byref(n), C.byref(w), _stream_ptr()))
    return n.value, w.value


def _streaming_palette(M):
    i = plan_info(M)
    assert i.path == 0 and i.kernel == 0 and i.tile_rows == 64 and i.npal > 0
    return i


def _both_kernels(B, monkeypatch, csr, vdt, xdt, x, use_shapes):
    """csr (integer values) on the streaming kernel -- with row shapes or without, as use_shapes says -- and on the per-tile kernel:
    both exact, so both the same; returns the streaming kernel's matrix"""
    nr, nc, rp, ci, v = csr
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=vdt)
    _streaming_palette(M)
    ns, nw = shapes(M)
    if use_shapes:
        assert 0 < ns <= SHAPE_MAX and ns <= nw <= 1024 and nw % 4 == 0, (ns, nw)
    else:
        assert (ns, nw) == (-1, -1)
    y = _exact(B, M, csr, x, xdt)
    with monkeypatch.context() as mp:
        mp.setenv("BMSP_SPMV_KERNEL", "1")
        T = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=vdt)
        assert plan_info(T).kernel == 1 and shapes(T) == (-1, -1)
    assert np.array_equal(_exact(B, T, csr, x, xdt), y)
    return M


def _stencil3d(nx, ny, nz):
    """7-point stencil on an nx x ny x nz grid (no wrap-around neighbours)"""
    n = nx * ny * nz
    i = np.arange(n)
    x, y, z = i % nx, (i // nx) % ny, i // (nx * ny)
    rows, cols = [i], [i]
    for ok, d in ((x > 0, -1), (x < nx - 1, 1), (y > 0, -nx), (y < ny - 1, nx), (z > 0, -nx * ny), (z < nz - 1, nx * ny)):
        rows.append(i[ok]); cols.append(i[ok] + d)
    return (n, n) + _csr(n, np.concatenate(rows), np.concatenate(cols))


def _with_values(pat, vdt, seed, const=None):
    """pat with random integer values for vdt, or with Poisson's constant coefficients (4 on the diagonal, -1 elsewhere)"""
    nr, nc, rp, ci = pat
    if const is None:
        v = _values(ci.size, vdt, np.random.default_rng(seed))
    else:
        v = np.where(ci == np.repeat(np.arange(nr), np.diff(rp)), 4.0, -1.0).astype(np.float32)
    return nr, nc, rp, ci, v


# ---------------------------------------------------------------------------------------------------------------- structured matrices
# grid widths: no multiple of 8 (the +-m neighbours fall into two block columns), a multiple of 8 but not of 32, tiles that end
# mid grid row in different ways; rows not a multiple of 8 or of 512 (a partial last tile)
GRIDS = [(300, 221), (1001, 67), (520, 131), (37, 1800)]


@pytest.mark.parametrize("const", [True, False], ids=["const", "random"])
@pytest.mark.parametrize("grid", GRIDS, ids=[f"{m}x{n}" for m, n in GRIDS])
@pytest.mark.parametrize("xdt", [torch.float16, torch.float32], ids=["x16", "x32"])
def test_poisson(B, monkeypatch, grid, const, xdt):
    """fp16 values (fp32 values make Poisson's block rows heavier than the streaming kernel's 64-row tiles take)"""
    pat = _poisson(*grid)
    csr = _with_values(pat, torch.float16, seed=grid[0], const=const or None)
    _both_kernels(B, monkeypatch, csr, torch.float16, xdt, _x(csr[1], torch.float16, np.random.default_rng(1)), True)


@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_band(B, monkeypatch, vdt, xdt):
    """diagonals -1, 0, 1, 2, 16: tridiagonal, shifted and diagonal halves, generic walks; every value / x dtype pair (light enough
    with fp32 values for the streaming kernel)"""
    csr = _with_values(_band(70001, (-1, 0, 1, 2, 16)), vdt, seed=5)
    _both_kernels(B, monkeypatch, csr, vdt, xdt, _x(csr[1], vdt, np.random.default_rng(2)), True)


@pytest.mark.parametrize("xdt", [torch.float16, torch.float32], ids=["x16", "x32"])
def test_stencil_3d(B, monkeypatch, xdt):
    """fp16 values (with fp32 values its block rows are too heavy for the streaming kernel)"""
    csr = _with_values(_stencil3d(32, 24, 83), torch.float16, seed=7)
    _both_kernels(B, monkeypatch, csr, torch.float16, xdt, _x(csr[1], torch.float16, np.random.default_rng(3)), True)


# ---------------------------------------------------------------------------------------------------------------- limits and fallbacks
@pytest.mark.parametrize("k", [SHAPE_MAX, SHAPE_MAX + 1])
def test_shape_limit(B, monkeypatch, k):
    """one diagonal block per block row whose bitmap is pattern r % k of k distinct ones: exactly k shapes (the diagonal block's x
    offset is the same relative to every row).  SHAPE_MAX shapes is the largest table; one more keeps the block words."""
    rng = np.random.default_rng(k)
    pats = np.unique(_random_bitmaps(4 * k, rng, (4, 13)))[:k]
    rng.shuffle(pats)
    assert pats.size == k
    nbr = 64 * 23
    br = np.arange(nbr)
    pat = _from_blocks(nbr * 8, nbr * 8, br, br, pats[br % k])
    csr = _with_values(pat, torch.float16, seed=k)
    M = _both_kernels(B, monkeypatch, csr, torch.float16, torch.float32, _x(csr[1], torch.float16, rng), k <= SHAPE_MAX)
    assert plan_info(M).npal == k
    if k <= SHAPE_MAX:
        assert shapes(M) == (k, k)


def test_scattered_palette_matrix_keeps_words(B, monkeypatch):
    """eight bitmaps over random block columns: a palette, but nearly every row is a shape of its own"""
    csr = _with_values(_scattered(3000, 8 * 20000 + 5, 3, seed=11, distinct=False), torch.float16, seed=11)
    _both_kernels(B, monkeypatch, csr, torch.float16, torch.float32, _x(csr[1], torch.float16, np.random.default_rng(4)), False)


def test_negative_relative_offsets(B, monkeypatch):
    """the last block row of every tile but the first also touches the x line eight block columns before the tile: that line comes
    first in the tile's staged lines, so the row's offset relative to 8 * 63 is negative"""
    nbr = 64 * 30 + 9
    tri = np.uint64(0xC0E070381C0E0703)
    br, bc, bm = list(range(nbr)), list(range(nbr)), [tri] * nbr
    for t0 in range(64, nbr, 64):
        if t0 + 63 < nbr:
            br.append(t0 + 63); bc.append(t0 - 8); bm.append(np.uint64(0x8001000000000081))
    br, bc, bm = np.array(br), np.array(bc), np.array(bm, np.uint64)
    o = np.lexsort((bc, br))
    pat = _from_blocks(nbr * 8 - 5, nbr * 8 - 5, br[o], bc[o], bm[o])
    for vdt, xdt in DTYPES:
        csr = _with_values(pat, vdt, seed=9)
        _both_kernels(B, monkeypatch, csr, vdt, xdt, _x(csr[1], vdt, np.random.default_rng(5)), True)


def test_empty_rows_and_over_capacity_tile(B, monkeypatch):
    """a band of diagonal blocks with every seventh block row empty and a partial last tile, and one tile above the capacities
    (read from global memory, its 1000-block row is no shape) among the shape rows"""
    nr, nc, rp, ci = _band_plus_heavy_row(6000 + 17, 8 * 4 * 3000, 2500, 1000, 1000, seed=8, distinct=False)
    rows = np.repeat(np.arange(nr), np.diff(rp))
    keep = ((rows // 8) % 7 != 3) | (rows // 8 == 2500)
    rp2, ci2 = _csr(nr, rows[keep], ci[keep])
    csr = _with_values((nr, nc, rp2, ci2), torch.float16, seed=8)
    M = _both_kernels(B, monkeypatch, csr, torch.float16, torch.float32, _x(nc, torch.float16, np.random.default_rng(6)), True)
    i = plan_info(M)
    assert i.over_cap_tiles == 1 and i.unplanned_tiles == 0


# ---------------------------------------------------------------------------------------------------------------- other callers
def test_halo_variant(B):
    """bmsp_spmv_halo with the rank as its own peer on a shape matrix (the fused halo variant of the streaming kernel)"""
    csr = _with_values(_poisson(1003, 91), torch.float16, seed=12)
    nr, nc, rp, ci, v = csr
    assert nr % 4 != 0
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=torch.float16)
    _streaming_palette(M)
    assert shapes(M)[0] > 0
    x = _x(nc, torch.float16, np.random.default_rng(7))
    xs, _ = _buffers(csr, x, torch.float32)
    case = (M, csr, xs, _reference(csr, x), 512)
    ranges = _shapes(nr, 512)
    for name in ("tile_edges", "all_gather_7", "tail", "mid_quad"):
        _check_halo(B, case, ranges[name])


def test_host_pipeline(B):
    """bmsp_spmv_host (row-range launches over chunks of tiles, eager and as a graph) == bmsp_spmv, bit for bit"""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(700, 401)
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, G.values_fp16(3, ci.size))
    assert shapes(M)[0] > 0
    for xdt in (torch.float32, torch.float16):
        xh = torch.from_numpy(G.x_vector(nc)).to(xdt).pin_memory()
        ref = B.bmSparse_SpMV(M, xh.cuda()).cpu()
        yh = torch.full((nr,), 7.0).pin_memory()
        for it in range(3):
            yh.fill_(7.0)
            B.bmSparse_SpMV_host(M, xh, yh)
            torch.cuda.synchronize()
            assert torch.equal(yh, ref), (xdt, it)


def test_chained_products(B):
    """x <- A x four times with Poisson's coefficients on a grid of 2^17 rows: every product exact (|x| grows at most 8x a step)"""
    import scipy.sparse as sp
    csr = _with_values(_poisson(517, 254), torch.float16, seed=0, const=True)
    nr, nc, rp, ci, v = csr
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    assert shapes(M)[0] > 0
    S = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(nr, nc))
    x = np.random.default_rng(8).integers(-20, 21, nc).astype(np.float64)
    xt = torch.from_numpy(x.astype(np.float32)).cuda()
    for step in range(4):
        x = S @ x
        xt = B.bmSparse_SpMV(M, xt)
        assert np.array_equal(xt.cpu().numpy().astype(np.float64), x), step


def test_device_memory_back_to_baseline(B, pool):  # noqa: F811
    """a shape plan (palette + table, row words) and the scan's scratch are all freed with the matrix"""
    def fn():
        nr, nc, rp, ci, v = B.generators.poisson5pt(300, 221)
        M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
        assert shapes(M)[0] > 0
        B.bmSparse_SpMV(M, torch.ones(nc, device="cuda"))
        torch.cuda.synchronize()
    _pool_run(pool, "spmv_shapes", fn)
