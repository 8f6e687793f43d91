"""Exact-arithmetic tests of every SpMV kernel branch (spmv.cu), each with the plan's choice asserted through bmsp_debug_spmv_plan.

With integer values, integer x and sum_j |a_ij x_j| < 2^24 for every row, every fp32 partial sum is an integer below 2^24 and
therefore exact -- fused or not, in any order.  y must then equal the float64 product bit for bit: a dropped, doubled or misplaced
cell of any size, a wrong x element, a stale staged tile or an fp16 rounding of an fp32 value all change an integer result, where
the tolerance of test_gpu_spmv.py (1e-5 * sum |a x| per row) would let a small one through.

The reference is scipy's float64 product of the same CSR, independent of oracle/.  x is a slice of a buffer filled with NaN and y a
slice of a buffer filled with a sentinel, so a read past x's ends and a write past y's ends show up too.  fp32-valued matrices hold
odd integers in 2049 .. 4095, which fp16 cannot represent: a value rounded to fp16 anywhere changes the result.  Unless a case says
otherwise it runs the four combinations of value dtype and x dtype (fp16, fp32)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

PLAN_MAXB = 2048        # blocks per tile the planner sorts (spmv.cu)
XL_MAX = 1900           # x lines per tile the planner offsets (spmv.cu)
STREAM_CTAS = 7         # streaming-kernel CTAs per SM (spmv.cu)
SENTINEL = -12345.5
PAD = 64                # elements in front of and behind x and y (keeps both 16-byte aligned)
DTYPES = [(vd, xd) for vd in (torch.float16, torch.float32) for xd in (torch.float16, torch.float32)]
DT_IDS = [f"{'v16' if vd == torch.float16 else 'v32'}-{'x16' if xd == torch.float16 else 'x32'}" for vd, xd in DTYPES]


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


class PlanInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("path", "kernel", "tile_rows", "npal", "cap_blk", "cap_val", "cap_lines", "ntiles",
                                          "empty_tiles", "unplanned_tiles", "unplanned_blocks", "unplanned_lines",
                                          "over_cap_tiles", "tail_line_tiles")] + \
              [("runs", C.c_int32 * 4)] + [(n, C.c_int32) for n in ("n_work", "n_bundles", "n_split_rows")]


def plan_info(M):
    from bmsparse_spgemm_spmv_b200 import _lib as L
    from bmsparse_spgemm_spmv_b200.matrix import _stream_ptr
    info = PlanInfo()
    L.check(L.lib().bmsp_debug_spmv_plan(M._h, C.byref(info), _stream_ptr()))
    return info


# ---------------------------------------------------------------------------------------------------------------- inputs
def _values(n, vdt, rng):
    """nonzero integers: |v| <= 63 for fp16 matrices, odd 2049 .. 4095 (not fp16-representable) for fp32 ones"""
    sign = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    mag = rng.integers(1, 64, n) if vdt == torch.float16 else 2049 + 2 * rng.integers(0, 1024, n)
    return (sign * mag).astype(np.float32)


def _x(nc, vdt, rng):
    """nonzero integers small enough for the exactness bound: |x| <= 100 against fp16 values, <= 3 against fp32 values"""
    hi = 101 if vdt == torch.float16 else 4
    return (np.where(rng.random(nc) < 0.5, -1.0, 1.0) * rng.integers(1, hi, nc)).astype(np.float32)


def _csr(nr, rows, cols):
    o = np.lexsort((cols, rows))
    rows, cols = rows[o], cols[o]
    rp = np.zeros(nr + 1, np.int64)
    np.cumsum(np.bincount(rows, minlength=nr), out=rp[1:])
    return rp.astype(np.int32), cols.astype(np.int32)


def _from_blocks(nr, nc, br, bc, bmps):
    """the pattern of 8x8 blocks (block row, block column, MSB-first bitmap: bit 63 - (8 r + c) is cell (r, c)); cells outside
    the matrix are dropped"""
    br = np.asarray(br, np.int64); bc = np.asarray(bc, np.int64); bmps = np.asarray(bmps, np.uint64)
    key = br * ((nc + 7) // 8) + bc
    assert np.unique(key).size == key.size, "one block per (block row, block column)"
    k = np.arange(64, dtype=np.uint64)
    bits = ((bmps[:, None] >> (np.uint64(63) - k[None, :])) & np.uint64(1)).astype(bool)
    b, cell = np.nonzero(bits)
    rows = br[b] * 8 + cell // 8
    cols = bc[b] * 8 + cell % 8
    keep = (rows < nr) & (cols < nc)
    return (nr, nc) + _csr(nr, rows[keep], cols[keep])


def _poisson(m, n):
    import bmsparse_spgemm_spmv_b200 as B
    nr, nc, rp, ci, _ = B.generators.poisson5pt(m, n)
    return nr, nc, rp, ci


def _band(nr, offsets):
    rows, cols = [], []
    for d in offsets:
        r = np.arange(max(0, -d), min(nr, nr - d))
        rows.append(r); cols.append(r + d)
    return (nr, nr) + _csr(nr, np.concatenate(rows), np.concatenate(cols))


def _random_bitmaps(n, rng, cells=(3, 13)):
    k = rng.integers(*cells, n)
    out = np.zeros(n, np.uint64)
    for i in range(n):
        out[i] = np.bitwise_or.reduce(np.uint64(1) << rng.choice(64, int(k[i]), replace=False).astype(np.uint64))
    return out


def _scattered(nbr, nc, per_row, seed, distinct):
    """per_row blocks per block row at random block columns: the tiles' x lines form far more than three runs.  distinct = False:
    every bitmap is one of eight patterns of 4 .. 12 cells; True: more than 256 distinct bitmaps"""
    rng = np.random.default_rng(seed)
    nbc = (nc + 7) // 8
    br = np.repeat(np.arange(nbr), per_row)
    bc = np.concatenate([np.sort(rng.choice(nbc, per_row, replace=False)) for _ in range(nbr)])
    pats = _random_bitmaps(8, rng, (4, 13))
    bm = _random_bitmaps(br.size, rng) if distinct else pats[rng.integers(0, 8, br.size)]
    return _from_blocks(nbr * 8 - 3, nc, br, bc, bm)


def _band_plus_heavy_row(nbr, nc, heavy_br, nblocks, nlines, seed, distinct):
    """a block-diagonal band (one diagonal block of 8 cells per block row: 64 blocks and 16 x lines per tile) and one block row of
    nblocks blocks spread over nlines x lines that none of its tile's band blocks touch, two cells each in different rows;
    distinct: the heavy row's bitmaps are random (more than 256 distinct), else one of eight patterns that cover every row
    equally (a row's sum stays within the exactness bound)"""
    rng = np.random.default_rng(seed)
    t0 = heavy_br // 64 * 64
    band_lines = set(range(t0 // 4, (t0 + 64) // 4 + 1))
    free = np.array([l for l in range((nc // 8 - 1) // 4) if l not in band_lines])
    lines = np.sort(rng.choice(free, nlines, replace=False))
    bcs = (lines[:, None] * 4 + np.arange(4)[None, :]).ravel()
    bc_heavy = np.sort(np.concatenate([lines * 4, rng.choice(np.setdiff1d(bcs, lines * 4), nblocks - nlines, replace=False)]))
    pats = np.array([(1 << (63 - 9 * p)) | (1 << (63 - 8 * ((p + 3) % 8) - (7 - p))) for p in range(8)], np.uint64)
    bm_heavy = _random_bitmaps(nblocks, rng, (2, 3)) if distinct else pats[np.arange(nblocks) % 8]
    diag = np.uint64(0x8040201008040201)
    br = np.concatenate([np.arange(nbr), np.full(nblocks, heavy_br)])
    bc = np.concatenate([np.arange(nbr), bc_heavy])
    bm = np.concatenate([np.full(nbr, diag), bm_heavy])
    return _from_blocks(nbr * 8, nc, br, bc, bm)


# ---------------------------------------------------------------------------------------------------------------- harness
def _matrix(B, pat, vdt, seed):
    """the matrix of pattern pat with integer values for vdt; the CSR with those values; fp32 values come back unchanged"""
    nr, nc, rp, ci = pat
    v = _values(ci.size, vdt, np.random.default_rng(seed))
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=vdt)
    if vdt == torch.float32:
        rows = np.repeat(np.arange(nr), np.diff(rp))
        order = np.lexsort((ci % 8, rows % 8, ci // 8, rows // 8))       # block order, then MSB-first bit order
        assert np.array_equal(M.download()[3], v[order]), "fp32 values must be stored as given"
    return M, (nr, nc, rp, ci, v)


def _reference(csr, x):
    """scipy float64 product, after checking the exactness precondition: integers, sum_j |a_ij x_j| < 2^24 per row"""
    nr, nc, rp, ci, v = csr
    S = sp.csr_matrix((v.astype(np.float64), ci, rp), shape=(nr, nc))
    xf = np.asarray(x, np.float64)
    fin = np.isfinite(xf)
    assert np.all(v == np.round(v)) and np.all(xf[fin] == np.round(xf[fin]))
    assert float((abs(S) @ np.abs(np.where(fin, xf, 0))).max(initial=0)) < 2 ** 24
    return S @ xf


def _buffers(csr, x, xdt):
    """x inside a NaN-filled buffer, a NaN-filled y inside a sentinel-filled buffer (both 16-byte aligned), on the current stream"""
    nr, nc = csr[0], csr[1]
    xbuf = torch.full((nc + 2 * PAD,), float("nan"), dtype=xdt, device="cuda")
    xs = xbuf[PAD:PAD + nc]
    xs.copy_(torch.from_numpy(np.asarray(x, np.float32)).to(xdt))
    ybuf = torch.full((nr + 2 * PAD,), SENTINEL, device="cuda")
    ybuf[PAD:PAD + nr] = float("nan")
    return xs, ybuf


def _check(ref, ybuf, equal_nan=False):
    """y equals the float64 product exactly (NaN where it is NaN, with equal_nan) and the sentinels around it are untouched"""
    yb = ybuf.cpu().numpy()
    got = yb[PAD:PAD + ref.size].astype(np.float64)
    bad = ~((got == ref) | (equal_nan & np.isnan(got) & np.isnan(ref)))
    assert not bad.any(), f"{int(bad.sum())} rows differ, first {np.flatnonzero(bad)[:8].tolist()}: {got[bad][:4]} vs {ref[bad][:4]}"
    assert np.all(yb[:PAD] == SENTINEL) and np.all(yb[PAD + ref.size:] == SENTINEL), "y's neighbours were written"
    return got


def _exact(B, M, csr, x, xdt, equal_nan=False):
    """one product y = A x (see _buffers) checked against the float64 product (_check); returns y on the host"""
    ref = _reference(csr, x)
    xs, ybuf = _buffers(csr, x, xdt)
    B.bmSparse_SpMV(M, xs, ybuf[PAD:PAD + csr[0]])
    return _check(ref, ybuf, equal_nan)


def _run(B, pat, vdt, xdt, seed, check_plan, monkeypatch=None, per_tile=False):
    """build the matrix (per_tile: behind the one-CTA-per-tile kernel), assert its plan, run one exact product"""
    if per_tile:
        monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
    M, csr = _matrix(B, pat, vdt, seed)
    info = plan_info(M)
    if per_tile:
        monkeypatch.delenv("BMSP_SPMV_KERNEL")
    check_plan(info)
    _exact(B, M, csr, _x(csr[1], vdt, np.random.default_rng(seed + 1)), xdt)
    return M, csr, info


def _streaming(info, palette):
    assert info.path == 0 and info.kernel == 0 and info.tile_rows == 64
    assert (info.npal > 0) == palette, info.npal


# ---------------------------------------------------------------------------------------------------------------- streaming kernel
@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_poisson_runs_and_tail_line(B, vdt, xdt):
    """Poisson with 66 300 rows and columns (not a multiple of 8 or 32): x lines in two and in three runs, and a last x line that
    reaches past the last column (hand-loaded by the streaming kernel, a guarded gather in the per-tile kernel).  fp16 values: the
    streaming kernel with a palette; fp32 values make an average block row heavier than 320 bytes: the per-tile kernel at 32-row
    tiles.  Poisson's own values are 4 and -1; random integers on its pattern catch misplaced cells."""
    def plan(i):
        if vdt == torch.float16:
            _streaming(i, palette=True)
        else:
            assert i.path == 0 and i.kernel == 1 and i.tile_rows == 32
        assert i.unplanned_tiles == 0 and i.over_cap_tiles == 0 and i.runs[0] == 0 and i.runs[1] == 0
        assert i.runs[2] > 0 and i.runs[3] > 0 and i.tail_line_tiles > 0
    pat = _poisson(2210, 30)
    assert pat[0] % 8 and pat[0] % 32
    _run(B, pat, vdt, xdt, 1, plan)


@pytest.mark.parametrize("distinct", [False, True], ids=["palette", "no_palette"])
@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_scattered_lines(B, vdt, xdt, distinct):
    """Streaming kernel, x lines scattered over the columns (nruns = 0: one bulk copy per line, all lanes of the producer), with
    and without a palette; some tiles also have the hand-loaded last line.  No existing test checks this branch against a
    reference."""
    def plan(i):
        _streaming(i, palette=not distinct)
        assert i.unplanned_tiles == 0 and i.over_cap_tiles == 0
        assert i.runs[0] == i.ntiles - i.empty_tiles and i.tail_line_tiles > 0
    _run(B, _scattered(3000, 8 * 20000 + 5, 3, seed=11, distinct=distinct), vdt, xdt, 2, plan)


# (heavy-row blocks, their x lines, how the tile is read): one tile of a light band above a shared-memory capacity, above XL_MAX
# distinct x lines, above PLAN_MAXB blocks
HEAVY = {"over_caps": (1000, 1000), "xl_max": (1950, 1950), "plan_maxb": (2500, 640)}


@pytest.mark.parametrize("distinct", [False, True], ids=["palette", "no_palette"])
@pytest.mark.parametrize("case", list(HEAVY))
@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_unstaged_tile_in_streaming_kernel(B, vdt, xdt, case, distinct):
    """Streaming kernel, one tile read from global memory (half_block_row) among staged ones: over the capacities plan_tiles
    derives from the averages, unplanned because of XL_MAX lines, unplanned because of PLAN_MAXB blocks.  test_gpu_spmv's
    test_tile_overflow_falls_back_to_global has heavy rows and runs the per-tile kernel instead."""
    nblocks, nlines = HEAVY[case]

    def plan(i):
        _streaming(i, palette=not distinct)
        if case == "over_caps":
            assert i.unplanned_tiles == 0 and i.over_cap_tiles == 1
        else:
            assert i.unplanned_tiles == 1 and i.over_cap_tiles == 0
            assert (i.unplanned_lines, i.unplanned_blocks) == ((1, 0) if case == "xl_max" else (0, 1))
    _run(B, _band_plus_heavy_row(6000, 8 * 4 * 3000, 2500, nblocks, nlines, seed=len(case), distinct=distinct), vdt, xdt, 3, plan)


# the 32-bit halves tile_half_row and build_palette classify: genuine diagonal / tridiagonal shapes of half 0 (rows 0-3) and half 1
# (rows 4-7), and near misses that must take the generic walk -- each half's constants in the other half, shifted by a column,
# one cell short
DIAG = (0x80402010, 0x08040201)
TRI = (0xC0E07038, 0x1C0E0703)
NEAR = [DIAG[1], TRI[1], DIAG[0] >> 1, TRI[0] >> 1, DIAG[0] & ~0x10, TRI[0] & ~0x08,        # candidates for half 0
        DIAG[0], TRI[0], DIAG[1] << 1, (TRI[1] << 1) & 0xFFFFFFFF, DIAG[1] & ~0x01, TRI[1] & ~0x01]   # for half 1


def _halves_matrix(nbr, seed, distinct):
    """three blocks per block row (the diagonal block, its right neighbour, one more at distance 5); each bitmap joins a half-0 word
    and a half-1 word drawn from the genuine shapes, the near misses, single cells and empty halves.  distinct: one block in four
    gets a random bitmap (more than 256 distinct)."""
    rng = np.random.default_rng(seed)
    h0 = [DIAG[0], TRI[0], 0x00800000, 0] + NEAR[:6]
    h1 = [DIAG[1], TRI[1], 0x00000100, 0] + NEAR[6:]
    words = sorted({(a << 32) | b for a in h0 for b in h1 if a | b})
    words = np.array(words, np.uint64)
    assert words.size <= 256
    br = np.repeat(np.arange(nbr), 3)
    bc = (br + np.tile([0, 1, 5], nbr)) % nbr
    bm = words[rng.integers(0, words.size, br.size)]
    if distinct:
        sel = rng.random(br.size) < 0.25
        bm[sel] = _random_bitmaps(int(sel.sum()), rng)
    # the near misses themselves, each next to both genuine shapes, at fixed places
    for j, w in enumerate(NEAR[:6]):
        bm[3 * j] = (w << 32) | DIAG[1]; bm[3 * j + 1] = (w << 32) | TRI[1]
    for j, w in enumerate(NEAR[6:]):
        bm[3 * (6 + j)] = (DIAG[0] << 32) | w; bm[3 * (6 + j) + 1] = (TRI[0] << 32) | w
    return _from_blocks(nbr * 8 - 5, nbr * 8 - 5, br, bc, bm)


@pytest.mark.parametrize("kernel", ["stream_palette", "stream_bitmaps", "per_tile"])
@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_near_miss_halves(B, monkeypatch, vdt, xdt, kernel):
    """Bitmap halves that resemble a diagonal or tridiagonal shape but are not that half's shape: a lower half holding the upper
    half's tridiagonal constant 0xC0E07038 or 0x80402010, shifted or one-cell-short shapes, next to genuine ones.  The streaming
    kernel with a palette (build_palette classifies), without one, and the per-tile kernel (tile_half_row classifies).  Poisson
    and the band tests only produce genuine shapes."""
    def plan(i):
        assert i.path == 0 and i.unplanned_tiles == 0 and i.over_cap_tiles == 0
        if kernel == "per_tile":
            assert i.kernel == 1 and i.tile_rows == 64 and i.npal == 0
        else:
            _streaming(i, palette=kernel == "stream_palette")
    pat = _halves_matrix(3000, seed=7, distinct=kernel == "stream_bitmaps")
    _run(B, pat, vdt, xdt, 4, plan, monkeypatch, per_tile=kernel == "per_tile")


# ---------------------------------------------------------------------------------------------------------------- per-tile kernel
def _dense_rows(nbr, nc, per_row, heavy, seed):
    """per_row dense 8x8 blocks per block row near the diagonal (64 cells each), one block row with `heavy` dense blocks spread over
    the columns; nc is no multiple of 32 and the last block column is used"""
    rng = np.random.default_rng(seed)
    nbc = (nc + 7) // 8
    bcs = [np.sort(rng.choice(np.arange(max(0, i * nbc // nbr - 8), min(nbc, i * nbc // nbr + 8)), per_row, replace=False))
           for i in range(nbr)]
    bcs[nbr // 2] = np.sort(rng.choice(nbc, heavy, replace=False))
    bcs[-1] = np.union1d(bcs[-1][1:], [nbc - 1])
    br = np.concatenate([np.full(b.size, i) for i, b in enumerate(bcs)])
    return _from_blocks(nbr * 8 - 1, nc, br, np.concatenate(bcs), np.full(br.size, np.uint64(2 ** 64 - 1)))


@pytest.mark.parametrize("rt", [32, 16])
@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_per_tile_kernel_dense_blocks(B, vdt, xdt, rt):
    """The one-CTA-per-tile kernel at 32- and 16-block-row tiles (dense blocks): staged tiles, one tile over the capacities (read
    from global memory) and the guarded gather of a last x line that reaches past the last column (cols % 32 != 0)."""
    # blocks per block row that give the tile height: an average block row above 320 bytes gives 32-row tiles, above 640 bytes 16
    per_row = {(32, torch.float16): 3, (16, torch.float16): 6, (32, torch.float32): 2, (16, torch.float32): 4}[(rt, vdt)]

    def plan(i):
        assert i.path == 0 and i.kernel == 1 and i.tile_rows == rt
        assert i.unplanned_tiles == 0 and i.over_cap_tiles == 1 and i.tail_line_tiles == 1
    _run(B, _dense_rows(640, 8 * 1500 + 3, per_row, 150, seed=rt), vdt, xdt, 5, plan)


# ---------------------------------------------------------------------------------------------------------------- block-parallel
def _block_parallel_pattern(nbr, seed):
    """one or two cells per block (the block-parallel path): block rows of 0 .. 9 blocks side by side (bundles of four short rows,
    and rows of nine that break their group), two hub rows of 1500 and 700 blocks (sliced, summed by the fix-up), a block-row count
    that is no multiple of four (a ragged last group) and rows % 8 != 0"""
    rng = np.random.default_rng(seed)
    nr, nc = nbr * 8 - 3, 1 << 15
    pattern = [0, 3, 8, 9, 1, 8, 8, 8, 0, 0, 0, 0, 2, 5, 7, 8]
    rows, cols = [], []
    for br in range(nbr):
        k = {nbr // 3: 1500, 2 * nbr // 3: 700}.get(br, pattern[(br + br // 16) % 16])
        for c in np.sort(rng.choice(nc // 8, k, replace=False)):
            cells = rng.choice(64, 1 + int(rng.integers(0, 2)), replace=False)
            rows += (br * 8 + cells // 8).tolist(); cols += (c * 8 + cells % 8).tolist()
    rows, cols = np.array(rows), np.array(cols)
    keep = rows < nr
    return (nr, nc) + _csr(nr, rows[keep], cols[keep])


def _block_parallel_plan(i):
    assert i.path == 1 and i.n_bundles > 0 and i.n_split_rows == 2 and i.n_work > i.n_bundles


@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_block_parallel(B, vdt, xdt):
    """Block-parallel kernel: bundles, a ragged group of four, sliced hub rows and their fix-up, empty block rows, rows % 8 != 0."""
    _run(B, _block_parallel_pattern(1001, seed=9), vdt, xdt, 6, _block_parallel_plan)


# ---------------------------------------------------------------------------------------------------------------- launches
@pytest.mark.parametrize("distinct", [False, True], ids=["palette", "no_palette"])
@pytest.mark.parametrize("vdt", [torch.float16, torch.float32], ids=["v16", "v32"])
def test_dynamic_tile_claims_and_slot_wrap(B, vdt, distinct):
    """Streaming kernel with dynamic tile claims (at least two tiles per CTA, about 1.2 M rows), with and without a palette: 40
    products on one matrix, the first 20 on one stream, the second 20 alternating between two streams.  Each launch takes the next
    of the 16 scheduler slots, so the slots wrap twice and every re-armed counter is used again; at most two launches are in
    flight at a time, so no two share a slot.  Every y is exact.  x is fp32 and fp16 in turn."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pat = _band_plus_random(150000, seed=12) if distinct else _band(1200000 - 5, (-1, 0, 1))
    M, csr = _matrix(B, pat, vdt, 13)
    info = plan_info(M)
    _streaming(info, palette=not distinct)
    assert info.ntiles >= 2 * sms * STREAM_CTAS and info.unplanned_tiles == 0
    x = _x(csr[1], vdt, np.random.default_rng(14))
    ref = _reference(csr, x)
    xdt = lambda k: torch.float32 if k % 3 else torch.float16
    for k in range(20):
        _exact(B, M, csr, x, xdt(k))
    # all buffers first, then 20 launches alternating between two streams, each stream's launches in order
    bufs = [_buffers(csr, x, xdt(k)) for k in range(20, 40)]
    side = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in side:
        s.wait_stream(torch.cuda.current_stream())
    for k, (xs, ybuf) in enumerate(bufs):
        B.bmSparse_SpMV(M, xs, ybuf[PAD:PAD + csr[0]], stream=side[k % 2])
    torch.cuda.synchronize()
    first = _check(ref, bufs[0][1])
    for xs, ybuf in bufs[1:]:
        assert np.array_equal(_check(ref, ybuf), first)


def _band_plus_random(nbr, seed):
    """a tridiagonal band plus random cells within 16 columns of the diagonal: light rows, more than 256 distinct bitmaps"""
    rng = np.random.default_rng(seed)
    n = nbr * 8
    r = np.repeat(np.arange(n), 3)
    c = r + rng.integers(-16, 17, r.size)
    rows = np.concatenate([np.arange(n), r]); cols = np.concatenate([np.arange(n), c])
    keep = (cols >= 0) & (cols < n)
    key = np.unique(rows[keep] * n + cols[keep])
    return (n, n) + _csr(n, key // n, key % n)


@pytest.mark.parametrize("vdt", [torch.float16, torch.float32], ids=["v16", "v32"])
def test_one_plan_serves_both_x_dtypes(B, vdt):
    """one plan, products with fp16 and fp32 x in turn: the plan holds nothing that depends on x's dtype"""
    for pat, path in ((_band(30001, (-1, 0, 1, 300)), 0), (_block_parallel_pattern(64, 3), 1)):
        M, csr = _matrix(B, pat, vdt, 21)
        assert plan_info(M).path == path
        x = _x(csr[1], vdt, np.random.default_rng(22))
        for xdt in (torch.float16, torch.float32, torch.float16, torch.float32):
            _exact(B, M, csr, x, xdt)


@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_non_finite_x(B, monkeypatch, vdt, xdt):
    """x with +Inf, -Inf and NaN in chosen columns: the rows that store those columns are the float64 Inf or NaN, all other rows
    exact -- no kernel multiplies an x element that its row does not store (staged x lines hold neighbours of those columns)."""
    cases = [(_poisson(211, 50), False), (_poisson(211, 50), True), (_block_parallel_pattern(200, 5), False)]
    for k, (pat, per_tile) in enumerate(cases):
        if per_tile:
            monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
        M, csr = _matrix(B, pat, vdt, 30 + k)
        plan_info(M)
        monkeypatch.delenv("BMSP_SPMV_KERNEL", raising=False)
        nc = csr[1]
        x = _x(nc, vdt, np.random.default_rng(40 + k))
        special = np.random.default_rng(50 + k).choice(nc, 30, replace=False)
        x[special[:10]] = np.inf; x[special[10:20]] = -np.inf; x[special[20:]] = np.nan
        y = _exact(B, M, csr, x, xdt, equal_nan=True)
        assert not np.isfinite(y).all()


@pytest.mark.parametrize("vdt,xdt", DTYPES, ids=DT_IDS)
def test_host_buffer_products_exact(B, vdt, xdt):
    """bmSparse_SpMV_host (x and y in pinned host memory) on the scattered and the block-parallel matrices, against the exact
    reference rather than against bmSparse_SpMV: eager, captured as a graph, replayed"""
    for pat in (_scattered(3000, 8 * 20000 + 5, 3, seed=11, distinct=False), _block_parallel_pattern(1001, seed=9)):
        M, csr = _matrix(B, pat, vdt, 60)
        x = _x(csr[1], vdt, np.random.default_rng(61))
        ref = _reference(csr, x)
        xh = torch.from_numpy(x).to(xdt).pin_memory()
        yh = torch.empty(csr[0]).pin_memory()
        for it in range(3):
            yh.fill_(float("nan"))
            B.bmSparse_SpMV_host(M, xh, yh)
            torch.cuda.synchronize()
            assert np.array_equal(yh.numpy().astype(np.float64), ref), it
