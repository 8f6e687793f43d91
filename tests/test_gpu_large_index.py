"""GPU: exact results at the advertised size limits -- value offsets past 2^31 and up to 2^32-1, coordinates at 2^31-1.

The library takes matrices of up to 2^32-1 values (BMSP_ERR_TOO_LARGE), and its kernels narrow the 64-bit offsets to 32 bits in
many places: the per-block-row value offsets (rvb), the tile descriptors and row pairs of SpMV, SpGEMM's pair records, the addition's
operand offsets, the row slices.  A value index held in a signed 32-bit integer anywhere among them goes wrong from 2^31 values on
and nowhere below, so every case here holds more than 2^31 values (or sits at the int32 coordinate limit) and checks its result
exactly.

The matrices are built on the device with from_arrays (from_csr's int32 row_ptr stops at 2^31-1 values).  Value i (its index in
the compact order) is an integer that depends on i: 1 + i mod 251 for fp16 matrices, odd 2049 .. 4089 (not fp16-representable) for
fp32 ones, with a sign that also depends on i.  251 and 1021 are prime, so a value read 2^31 or 2^32 places away is a different
value.  x holds small integers and every row's sum of |a x| stays below 2^24, so fp32 accumulation is exact in any order and y must
equal the float64 reference bit for bit.

The reference is plain torch on the device, independent of the library and of oracle/: each block's bitmap is unpacked into 64
cells, a set cell's value index is offsets[b] + its rank among the block's set cells, and the dense 8x8 blocks are multiplied with x
and summed into y by block row, a few million blocks at a time.  The same unpacking gives the expected contents of output blocks,
spot-checked on a random sample plus every block within 2^16 values of 2^31 or 2^32.

Each case states the device memory it needs (from its array sizes) and skips when less is free.  Every test prints its time and its
peak device memory, the library's (the default memory pool's USED_MEM_HIGH) and torch's, as `LARGE_INDEX <test> ...`, and trims the
pool afterwards so that the memory goes back to the device.  The block-parallel case needs about 90 GB and runs only with
BMSP_LARGE_TESTS=1."""
import ctypes as C
import gc
import os
import time

import numpy as np
import pytest
import torch

from tests.test_gpu_device_memory import USED_MEM_CURRENT, USED_MEM_HIGH, _Pool, pool  # noqa: F401
from tests.test_gpu_spmv_exact import PAD, SENTINEL, plan_info
from tests.test_gpu_spmv_halo import Halo, _halo_push, _spmv_halo

pytestmark = pytest.mark.gpu

F16, F32 = torch.float16, torch.float32
GB = 1 << 30
TWO31, TWO32 = 1 << 31, 1 << 32
INT32_MAX = TWO31 - 1
NEAR = 1 << 16              # blocks within this many values of 2^31 or 2^32 are always spot-checked
CHUNK = 1 << 20             # blocks per reference step
VCHUNK = 1 << 27            # values per generation step
FULL = -1                   # the full bitmap, as torch's int64
SHIFT = None                # 63 - cell, on the device (set on first use)


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


@pytest.fixture(autouse=True)
def _peak_and_trim(request, B):
    """prints the test's time and peak device memory; gives the pool's free memory back to the device afterwards"""
    torch.cuda.init()
    p = _Pool()
    gc.collect(); torch.cuda.synchronize(); torch.cuda.empty_cache()
    base = p.get(USED_MEM_CURRENT)
    p.reset_high(); torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    gc.collect(); torch.cuda.synchronize()
    print(f"\nLARGE_INDEX {request.node.name} {time.time() - t0:.1f} s, library peak {(p.get(USED_MEM_HIGH) - base) / GB:.2f} GiB, "
          f"torch peak {torch.cuda.max_memory_allocated() / GB:.2f} GiB")
    torch.cuda.empty_cache()
    assert p.cu.cuMemPoolTrimTo(p.pool, C.c_size_t(0)) == 0


def _need(nbytes, what):
    """skip unless nbytes of device memory are free"""
    gc.collect(); torch.cuda.synchronize(); torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"{what} needs {nbytes / GB:.1f} GiB of free device memory, {free / GB:.1f} GiB are free")


def _matrix_bytes(nblk, nnz, nbr, vsize):
    """the library's arrays of one matrix: keys, bitmaps, offsets, block columns, masks; values; row pointers and row offsets"""
    return nblk * 29 + nnz * vsize + nbr * 8


# ---------------------------------------------------------------------------------------------------------------- values
def _val16(i):
    """fp16-exact nonzero integers, |v| <= 251"""
    mag = 1 + i % 251
    return torch.where(i % 3 == 1, -mag, mag).to(torch.float64)


def _val16b(i):
    """another set of fp16 values (set_values): |v| <= 241"""
    mag = 1 + (i + 17) % 241
    return torch.where(i % 5 == 2, -mag, mag).to(torch.float64)


def _val32(i):
    """odd integers 2049 .. 4089, which fp16 cannot represent"""
    mag = 2049 + 2 * (i % 1021)
    return torch.where(i % 3 == 1, -mag, mag).to(torch.float64)


class Spec:
    """A matrix described on the device: keys (block row << 32 | block column), bitmaps (MSB first, normal form), offsets
    (nblk + 1 entries, the last one nnz), and value(i) for the value at compact index i."""

    def __init__(self, rows, cols, keys, bmps, offsets, value, dtype):
        self.rows, self.cols, self.keys, self.bmps, self.offsets, self.value, self.dtype = rows, cols, keys, bmps, offsets, value, dtype
        self.nblk = keys.numel()
        self.nnz = int(offsets[-1])
        self.nbr = (rows + 7) // 8

    def values(self, value=None):
        """all values in compact order, in the matrix's dtype"""
        value = value or self.value
        v = torch.empty(self.nnz, dtype=self.dtype, device="cuda")
        for s in range(0, self.nnz, VCHUNK):
            e = min(s + VCHUNK, self.nnz)
            v[s:e] = value(torch.arange(s, e, device="cuda")).to(self.dtype)
        return v

    def lookup(self, br, bc):
        """the block index of each (block row, block column); all must exist"""
        key = (br << 32) | bc
        b = torch.searchsorted(self.keys, key).clamp(max=self.nblk - 1)
        assert torch.equal(self.keys[b], key), "expected block missing from the spec"
        return b

    def cells(self, b):
        """dense float64 [n, 8, 8] blocks b, cell (r, c)"""
        bits, rank = _unpack(self.bmps[b])
        v = torch.where(bits, self.value(self.offsets[b][:, None] + rank), 0.0)
        return v.view(-1, 8, 8)


def _build(B, spec, value=None):
    """the library's matrix of spec (values from value, default spec.value); the input tensors are freed before returning"""
    vals = spec.values(value)
    M = B.bmSpMatrix.from_arrays(spec.rows, spec.cols, spec.nblk, spec.keys, spec.bmps, spec.offsets[:spec.nblk], vals)
    del vals
    assert (M.nnz, M.block_num) == (spec.nnz, spec.nblk)
    return M


def _unpack(bmp):
    """bitmaps [n] -> (set cells [n, 64] bool, rank of each cell among the block's set cells [n, 64] int64), MSB first"""
    global SHIFT
    if SHIFT is None:
        SHIFT = 63 - torch.arange(64, device="cuda")
    bits = (bmp[:, None] >> SHIFT) & 1
    return bits.bool(), bits.cumsum(1) - bits


def _stored_cells(M, idx):
    """(block rows, block columns, dense float64 [n, 8, 8]) of M's stored blocks idx, read from M's arrays in M's form"""
    keys, off = M.keys[idx], M.offsets[idx]
    bits, rank = _unpack(M.bmps[idx])
    vals = M.values
    k = (off[:, None] + rank).clamp(max=M.nnz - 1)
    d = torch.where(bits, vals[k].double(), 0.0).view(-1, 8, 8)
    if M.transposed:                        # cell (r, c) is stored at bit 63 - (8 c + r)
        d = d.transpose(1, 2)
    return keys >> 32, keys & 0xFFFFFFFF, d


def _sample(offsets, nblk, n=4000, seed=0):
    """a random sample of blocks plus every block that crosses or lies within NEAR values of 2^31 or 2^32"""
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    idx = [torch.randint(0, nblk, (n,), device="cuda", generator=g)]
    off = offsets[:nblk]
    for t in (TWO31, TWO32):
        lo = int(torch.searchsorted(off, torch.tensor([t - NEAR], device="cuda")))
        hi = int(torch.searchsorted(off, torch.tensor([t + NEAR], device="cuda"), right=True))
        idx.append(torch.arange(max(lo - 1, 0), min(hi, nblk), device="cuda"))
    return torch.unique(torch.cat(idx))


def _check_blocks(M, idx, expected):
    """M's blocks idx equal expected(block rows, block columns) cell for cell"""
    br, bc, got = _stored_cells(M, idx)
    exp = expected(br, bc)
    bad = (got != exp).flatten(1).any(1)
    assert not bad.any(), f"{int(bad.sum())} of {idx.numel()} blocks differ, first at block {idx[bad][:4].tolist()}"


# ---------------------------------------------------------------------------------------------------------------- reference
def _ref_parts(spec, x, transpose=False, blocks=None, row0=0):
    """float64 contributions of spec's blocks [b0, b1) to A x (A^T x): (output rows, values, |a| |x| sums) per chunk"""
    b0, b1 = blocks or (0, spec.nblk)
    r8 = torch.arange(8, device="cuda")
    for s in range(b0, b1, CHUNK):
        b = torch.arange(s, min(s + CHUNK, b1), device="cuda")
        d = spec.cells(b)
        br, bc = spec.keys[b] >> 32, spec.keys[b] & 0xFFFFFFFF
        src, dst = (br, bc) if transpose else (bc, br)
        xi = src[:, None] * 8 + r8
        xg = torch.where(xi < x.numel(), x[xi.clamp(max=x.numel() - 1)].double(), 0.0)
        eq = "nrc,nr->nc" if transpose else "nrc,nc->nr"
        y = torch.einsum(eq, d, xg)
        ya = torch.einsum(eq, d.abs(), xg.abs())
        yield (dst[:, None] * 8 + r8 - row0).flatten(), y.flatten(), ya.flatten()


def _ref_spmv(spec, x, n_out, transpose=False, blocks=None, row0=0):
    """y = A x (A^T x) in float64 over n_out rows; asserts the exactness bound sum |a x| < 2^24 on every row"""
    y = torch.zeros(n_out, dtype=torch.float64, device="cuda")
    ya = torch.zeros(n_out, dtype=torch.float32, device="cuda")
    for rows, v, va in _ref_parts(spec, x, transpose, blocks, row0):
        keep = (rows >= 0) & (rows < n_out)
        assert not ((v != 0) & ~keep).any(), "a cell outside the matrix"
        y.index_add_(0, rows[keep], v[keep]); ya.index_add_(0, rows[keep], va[keep].float())
    assert float(ya.max()) < 2 ** 24 * 0.99
    del ya
    return y


# ---------------------------------------------------------------------------------------------------------------- products
def _x_buffer(n, dtype, fill):
    """x of n elements inside a NaN-filled buffer; fill(xs) writes its values"""
    xbuf = torch.full((n + 2 * PAD,), float("nan"), dtype=dtype, device="cuda")
    xs = xbuf[PAD:PAD + n]
    fill(xs)
    return xs


def _small_x(n, dtype, hi=7, seed=1):
    """nonzero integers in [-hi, hi]"""
    def fill(xs):
        g = torch.Generator(device="cuda"); g.manual_seed(seed)
        v = torch.randint(1, hi + 1, (n,), device="cuda", generator=g)
        xs.copy_(torch.where(torch.rand(n, device="cuda", generator=g) < 0.5, -v, v).to(dtype))
    return _x_buffer(n, dtype, fill)


def _y_buffer(n):
    ybuf = torch.full((n + 2 * PAD,), SENTINEL, device="cuda")
    ybuf[PAD:PAD + n] = float("nan")
    return ybuf


def _check_y(ybuf, ref, what=""):
    """y inside ybuf equals ref exactly; the sentinels around it are untouched"""
    n = ref.numel()
    got = ybuf[PAD:PAD + n].double()
    bad = got != ref
    nbad = int(bad.sum())
    if nbad:
        first = torch.nonzero(bad)[:6].flatten()
        raise AssertionError(f"{what}: {nbad} rows differ, first {first.tolist()}: {got[first].tolist()} vs {ref[first].tolist()}")
    assert bool((ybuf[:PAD] == SENTINEL).all()) and bool((ybuf[PAD + n:] == SENTINEL).all()), f"{what}: y's neighbours were written"


def _spmv_exact(B, M, x, ref, what=""):
    ybuf = _y_buffer(ref.numel())
    B.bmSparse_SpMV(M, x, ybuf[PAD:PAD + ref.numel()])
    _check_y(ybuf, ref, what)


# ---------------------------------------------------------------------------------------------------------------- matrices
NBLK_PAST = (1 << 25) + (1 << 21)      # full blocks: 2^31 + 2^27 values


def _full_rows(nblk, dtype, value=None, last_bitmap=None, shift=0):
    """one full block per block row, in block column (block row + shift) mod 4 of a 32-column matrix; offsets 64 b (last_bitmap:
    the last block's bitmap instead)"""
    b = torch.arange(nblk, device="cuda")
    keys = (b << 32) | ((b + shift) % 4)
    bmps = torch.full((nblk,), FULL, dtype=torch.int64, device="cuda")
    cnt = torch.full((nblk,), 64, dtype=torch.int64, device="cuda")
    if last_bitmap is not None:
        bmps[-1] = last_bitmap
        cnt[-1] = bin(last_bitmap & (2 ** 64 - 1)).count("1")
    offsets = torch.zeros(nblk + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(cnt, 0, out=offsets[1:])
    del b, cnt
    return Spec(8 * nblk, 32, keys, bmps, offsets, value or (_val16 if dtype == F16 else _val32), dtype)


def _case1(dtype=F16):
    return _full_rows(NBLK_PAST, dtype)


def _expect_same(spec):
    return lambda br, bc: spec.cells(spec.lookup(br, bc))


def _streaming_palette(i, npal=1):
    assert i.path == 0 and i.kernel == 0 and i.tile_rows == 64 and i.npal == npal, (i.path, i.kernel, i.tile_rows, i.npal)
    assert i.unplanned_tiles == 0 and i.over_cap_tiles == 0


# ---------------------------------------------------------------------------------------------------------------- 1: SpMV past 2^31
@pytest.mark.parametrize("run", ["streaming", "per_tile", "host"])
@pytest.mark.parametrize("vdt", [F16, F32], ids=["v16", "v32"])
def test_spmv_full_blocks_past_2_31(B, monkeypatch, vdt, run):
    """2^31 + 2^27 values in full blocks, one per block row over four block columns: the streaming kernel with its one-bitmap
    palette (tile descriptors and row offsets past 2^31), the per-tile kernel (row pairs narrowed to int2), and the host-buffer
    pipeline's row-range launches; fp16 and fp32 x"""
    vs = 2 if vdt == F16 else 4
    nnz = NBLK_PAST * 64
    nbr = NBLK_PAST
    # the matrix, its input copy while it is built, the spec, y, the reference and its bound, a reference step
    _need(_matrix_bytes(NBLK_PAST, nnz, nbr, vs) + nnz * vs + NBLK_PAST * 32 + nbr * 8 * (4 + 8 + 4) + 3 * GB, "2^31 + 2^27 values")
    spec = _case1(vdt)
    if run == "per_tile":
        monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
    M = _build(B, spec)
    info = plan_info(M)
    monkeypatch.delenv("BMSP_SPMV_KERNEL", raising=False)
    if run == "per_tile":
        assert info.path == 0 and info.kernel == 1 and info.tile_rows == 64 and info.npal == 0
    else:
        _streaming_palette(info)
    assert M.nnz > TWO31 and int(M._view().num_block_rows) == nbr
    x16 = _small_x(32, F16)
    ref = _ref_spmv(spec, x16, spec.rows)
    for xdt in (F16, F32):
        x = x16 if xdt == F16 else _x_buffer(32, F32, lambda xs: xs.copy_(x16))
        if run == "host":
            xh = x.cpu().pin_memory()
            yh = torch.empty(spec.rows, dtype=F32).pin_memory()
            for it in range(2):                 # eager, then the captured graph
                yh.fill_(float("nan"))
                B.bmSparse_SpMV_host(M, xh, yh)
                torch.cuda.synchronize()
                got = yh.cuda().double()
                bad = int((got != ref).sum())
                assert bad == 0, f"host pipeline {xdt} call {it}: {bad} rows differ"
                del got
        else:
            _spmv_exact(B, M, x, ref, f"{run} {xdt}")


# ---------------------------------------------------------------------------------------------------------------- 2: no palette
NPAT = 300      # more than PALETTE_MAX (256) distinct bitmaps


def _patterns(seed=5):
    """NPAT bitmaps of 40 .. 56 cells, each in four variants: as is, in the last block column (6 of its 8 columns inside the
    matrix), in the last block row (5 of 8 rows), in both; and their cell counts (int64 device tensors)"""
    rng = np.random.default_rng(seed)
    pats = []
    for _ in range(NPAT):
        cells = rng.choice(64, int(rng.integers(40, 57)), replace=False)
        pats.append(sum(1 << (63 - int(c)) for c in cells))
    colmask = int.from_bytes(bytes([0xFC] * 8), "big")
    rowmask = 0xFFFFFFFFFF000000
    table = [p & m for m in (2 ** 64 - 1, colmask, rowmask, colmask & rowmask) for p in pats]
    cnt = [bin(w).count("1") for w in table]
    words = np.array(table, np.uint64).view(np.int64)
    return torch.from_numpy(words).cuda(), torch.tensor(cnt, dtype=torch.int64, device="cuda")


def _case2(nblk=51_000_000):
    """one block per block row in block column (block row mod 4) of a 30-column matrix whose last block row is partial; the bitmaps
    are drawn from the NPAT patterns"""
    words, cnt = _patterns()
    b = torch.arange(nblk, device="cuda")
    bc = b % 4
    p = (b * 7919 + (b >> 9)) % NPAT + NPAT * ((bc == 3).long() + 2 * (b == nblk - 1).long())
    keys = (b << 32) | bc
    bmps = words[p]
    offsets = torch.zeros(nblk + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(cnt[p], 0, out=offsets[1:])
    del b, bc, p
    return Spec(8 * nblk - 3, 30, keys, bmps, offsets, _val16, F16)


def test_spmv_no_palette_past_2_31(B):
    """about 2^31 + 2^27 values in blocks of 40 .. 56 cells (fewer in the last block column and row) with more than 256 distinct
    bitmaps: the streaming kernel without a palette (per-block x offsets and the (int)-narrowed row pairs), a partial last block
    row, and a last x line that reaches past the 30th column (the hand-loaded line)"""
    nblk = 51_000_000
    nnz = nblk * 46
    _need(_matrix_bytes(nblk, nnz, nblk, 2) + nnz * 2 + nblk * 40 + nblk * 8 * 16 + 3 * GB, "2^31 + 2^27 values without a palette")
    spec = _case2(nblk)
    assert TWO31 + (1 << 26) < spec.nnz < TWO32
    M = _build(B, spec)
    info = plan_info(M)
    assert info.path == 0 and info.kernel == 0 and info.tile_rows == 64 and info.npal == 0
    assert info.unplanned_tiles == 0 and info.tail_line_tiles > 0
    x16 = _small_x(30, F16, seed=2)
    ref = _ref_spmv(spec, x16, spec.rows)
    _spmv_exact(B, M, x16, ref, "fp16 x")
    _spmv_exact(B, M, _x_buffer(30, F32, lambda xs: xs.copy_(x16)), ref, "fp32 x")
    _check_blocks(M, _sample(spec.offsets, nblk), _expect_same(spec))


# ---------------------------------------------------------------------------------------------------------------- 3: 2^32 - 1
def test_spmv_just_under_2_32_and_refusal_at_2_32(B, pool):
    """fp16, 2^32 - 37 values (the last block holds 27 cells): SpMV exact; from_arrays of 2^32 values fails with
    BMSP_ERR_TOO_LARGE and gives back all the memory it took"""
    from bmsparse_spgemm_spmv_b200 import _lib as L
    nblk = 1 << 26
    nnz = TWO32 - 37
    _need(2 * _matrix_bytes(nblk, TWO32, nblk, 2) + 3 * GB, "2^32 - 37 values")
    spec = _full_rows(nblk, F16)
    vals = spec.values()
    assert vals.numel() == TWO32
    gc.collect(); torch.cuda.synchronize()
    base = pool.get(USED_MEM_CURRENT)
    pool.reset_high()
    with pytest.raises(L.BmspError) as e:
        B.bmSpMatrix.from_arrays(spec.rows, spec.cols, nblk, spec.keys, spec.bmps, spec.offsets[:nblk], vals)
    assert e.value.code == 6
    gc.collect(); torch.cuda.synchronize()
    print(f"\nPOOL_PEAK from_arrays_2_32 {pool.get(USED_MEM_HIGH) - base}")
    assert pool.get(USED_MEM_CURRENT) == base, "from_arrays kept memory after refusing 2^32 values"
    last = -(1 << 37)                       # cells 0 .. 26
    assert bin(last & (2 ** 64 - 1)).count("1") == 27 and int(spec.offsets[-2]) + 27 == nnz
    spec.bmps[-1] = last
    spec.offsets[-1] = nnz
    spec.nnz = nnz
    M = B.bmSpMatrix.from_arrays(spec.rows, spec.cols, nblk, spec.keys, spec.bmps, spec.offsets[:nblk], vals[:nnz])
    del vals
    assert M.nnz == nnz
    _streaming_palette(plan_info(M), npal=2)
    x16 = _small_x(32, F16, seed=3)
    ref = _ref_spmv(spec, x16, spec.rows)
    _spmv_exact(B, M, x16, ref, "fp16 x")
    _spmv_exact(B, M, _x_buffer(32, F32, lambda xs: xs.copy_(x16)), ref, "fp32 x")
    _check_blocks(M, _sample(spec.offsets, nblk), _expect_same(spec))


# ---------------------------------------------------------------------------------------------------------------- 4: other operations
def _sparse_x(n, dtype, every=8192, dense=(), seed=4):
    """x of n elements, zero but for every `every`-th element and the ranges `dense`, which hold small nonzero integers"""
    def fill(xs):
        xs.zero_()
        g = torch.Generator(device="cuda"); g.manual_seed(seed)
        idx = torch.cat([torch.arange(0, n, every, device="cuda")] + [torch.arange(a, min(b, n), device="cuda") for a, b in dense])
        v = torch.randint(1, 4, (idx.numel(),), device="cuda", generator=g)
        xs[idx] = torch.where(idx % 2 == 1, -v, v).to(dtype)
    return _x_buffer(n, dtype, fill)


def test_transposes_past_2_31(B):
    """matrix_transpose in both output forms and block_transpose of the case-1 fp16 matrix: A^T x exact against the reference
    A^T x (x nonzero on every 8192nd row and on every row near 2^31 values), and blocks spot-checked"""
    spec = _case1(F16)
    mb = _matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 2)
    _need(3 * mb + spec.nnz * 2 + spec.rows * 4 + 4 * GB, "A and its transposes")
    M = _build(B, spec)
    near = TWO31 // 64 * 8
    x = _sparse_x(spec.rows, F32, dense=[(near - NEAR // 4, near + NEAR // 4)])
    ref = _ref_spmv(spec, x, 32, transpose=True)
    At = M.matrix_transpose()
    assert (At.num_rows, At.num_cols, At.nnz, At.transposed) == (32, spec.rows, spec.nnz, False)
    _spmv_exact(B, At, x, ref, "A^T x")
    _spmv_exact(B, At, _x_buffer(spec.rows, F16, lambda xs: xs.copy_(x)), ref, "A^T x, fp16 x")
    expect_t = lambda br, bc: spec.cells(spec.lookup(bc, br)).transpose(1, 2)
    _check_blocks(At, _sample(At.offsets, At.block_num, seed=1), expect_t)
    del At
    Att = M.matrix_transpose(transpose=True)
    assert Att.transposed and Att.nnz == spec.nnz
    _check_blocks(Att, _sample(Att.offsets, Att.block_num, seed=2), expect_t)
    del Att
    Mb = M.block_transpose()
    assert Mb.transposed and torch.equal(Mb.keys, spec.keys)
    _check_blocks(Mb, _sample(spec.offsets, spec.nblk, seed=3), _expect_same(spec))


def test_add_past_2_31(B):
    """bmSparse_add: A (2^31 + 2^27 values) minus a disjoint B (2^30 - 2^27 values) has 2^31 + 2^30 values; A - A keeps A's
    pattern with all values zero"""
    spec = _case1(F16)
    nb = (1 << 24) - (1 << 21)
    bspec = _full_rows(nb, F16, value=lambda i: _val16(i + 12345), shift=2)
    bspec.rows, bspec.nbr = spec.rows, spec.nbr       # same shape as A: B's blocks occupy the first nb block rows
    ma = _matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 2)
    mb = _matrix_bytes(nb, bspec.nnz, spec.nbr, 2)
    mc = _matrix_bytes(spec.nblk + nb, spec.nnz + bspec.nnz, spec.nbr, 2)
    _need(ma + mb + mc + spec.nnz * 2 + spec.rows * 16 + 4 * GB, "A, B and A - B")
    A = _build(B, spec)
    Bm = _build(B, bspec)
    Cm = B.bmSparse_add(A, Bm, 1.0, -1.0)
    assert Cm.nnz == TWO31 + TWO31 // 2 and Cm.block_num == spec.nblk + nb and Cm.dtype == F16
    x = _small_x(32, F16, seed=5)
    ref = _ref_spmv(spec, x, spec.rows)
    ref -= _ref_spmv(bspec, x, spec.rows)
    _spmv_exact(B, Cm, x, ref, "(A - B) x")
    del ref

    def expected(br, bc):
        in_a = bc == br % 4
        out = torch.empty(br.numel(), 8, 8, dtype=torch.float64, device="cuda")
        if in_a.any():
            out[in_a] = spec.cells(spec.lookup(br[in_a], bc[in_a]))
        if (~in_a).any():
            out[~in_a] = -bspec.cells(bspec.lookup(br[~in_a], bc[~in_a]))
        return out
    # C's own blocks near 2^31 and 2^32 values, and the blocks that take A's values from near 2^31
    a_near = _sample(spec.offsets, spec.nblk, n=0)
    c_from_a = torch.searchsorted(Cm.keys, spec.keys[a_near])
    _check_blocks(Cm, torch.unique(torch.cat([_sample(Cm.offsets, Cm.block_num, seed=6), c_from_a])), expected)
    del Cm, Bm
    Z = B.bmSparse_add(A, A, 1.0, -1.0)
    assert torch.equal(Z.keys, spec.keys) and torch.equal(Z.bmps, spec.bmps) and torch.equal(Z.offsets, spec.offsets[:spec.nblk])
    assert Z.nnz == spec.nnz and not bool((Z.values != 0).any()), "A - A is not all zeros"


def test_set_values_slice_and_to_csr_past_2_31(B):
    """set_values with a CUDA tensor of new values, then SpMV; slice_block_rows(rebase=True) of a range that starts past 2^31
    values against the matching rows of the reference; to_csr refuses (int32 row pointers)"""
    from bmsparse_spgemm_spmv_b200 import _lib as L
    spec = _case1(F16)
    _need(_matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 2) + 2 * spec.nnz * 2 + spec.rows * 16 + 4 * GB, "A and its new values")
    M = _build(B, spec)
    new = spec.values(_val16b)
    M.set_values(new)
    del new
    spec.value = _val16b
    x = _small_x(32, F16, seed=6)
    _spmv_exact(B, M, x, _ref_spmv(spec, x, spec.rows), "after set_values")
    r0 = TWO31 // 64 + 12345
    r1 = r0 + (1 << 20)
    S = M.slice_block_rows(r0, r1, rebase=True)
    assert (S.num_rows, S.nnz, S.block_num) == (8 * (r1 - r0), 64 * (r1 - r0), r1 - r0)
    _spmv_exact(B, S, x, _ref_spmv(spec, x, 8 * (r1 - r0), blocks=(r0, r1), row0=8 * r0), "slice")
    del S
    r0 = TWO31 // 64 - 1000                  # the slice's first values lie below 2^31, its last above
    S = M.slice_block_rows(r0, r0 + 2000, rebase=True)
    _spmv_exact(B, S, x, _ref_spmv(spec, x, 16000, blocks=(r0, r0 + 2000), row0=8 * r0), "slice across 2^31")
    del S
    with pytest.raises(L.BmspError) as e:
        M.to_csr()
    assert e.value.code == 6


# ---------------------------------------------------------------------------------------------------------------- 5: SpGEMM
def _diag(B, d):
    n = d.numel()
    idx = np.arange(n + 1, dtype=np.int32)
    return B.bmSpMatrix.from_csr(n, n, idx, idx[:n], d.cpu().numpy(), transpose=True, dtype=F16)


@pytest.mark.parametrize("path", [0, 1], ids=["scalar", "mma"])
def test_spgemm_c_past_2_31(B, path):
    """C = A D with A the case-1 fp16 matrix and D diagonal (transposed-operand form): every pair is one A block with one D block
    and C's values are a_ij d_j, 2^31 + 2^27 of them.  C's keys, bitmaps and offsets equal A's; C x equals A (D x) exactly; C's
    blocks spot-checked.  Then through a plan: A's values rewritten in place, numeric(), all checks again."""
    spec = _case1(F16)
    _need(_matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 2) + spec.nnz * 2 + _matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 4)
          + spec.nblk * 64 + spec.rows * 16 + 4 * GB, "A and C = A D")
    A = _build(B, spec)
    j = torch.arange(32, device="cuda")
    d = (((j % 3) + 1) * torch.where(j % 4 == 3, -1, 1)).double()
    D = _diag(B, d)
    x = _small_x(32, F32, seed=7)
    xd = x.double() * d

    def check(Cm, what):
        assert (Cm.num_rows, Cm.num_cols, Cm.nnz, Cm.block_num, Cm.dtype) == (spec.rows, 32, spec.nnz, spec.nblk, F32), what
        assert torch.equal(Cm.keys, spec.keys) and torch.equal(Cm.bmps, spec.bmps), what
        assert torch.equal(Cm.offsets[:spec.nblk], spec.offsets[:spec.nblk]), what
        _spmv_exact(B, Cm, x, _ref_spmv(spec, xd, spec.rows), what)
        cols = torch.arange(8, device="cuda")
        _check_blocks(Cm, _sample(spec.offsets, spec.nblk, seed=8),
                      lambda br, bc: spec.cells(spec.lookup(br, bc)) * d[bc[:, None] * 8 + cols][:, None, :])

    Cm, info = B.bmSparse_mult(A, D, numeric_path=path)
    assert info.numeric_path == path
    check(Cm, "bmSparse_mult")
    del Cm
    plan = B.bmSparse_mult_plan(A, D, numeric_path=path)
    assert plan.info.numeric_path == path
    check(plan.C, "plan")
    vals = A.values                            # new values written in place, chunk by chunk
    for s in range(0, spec.nnz, VCHUNK):
        e = min(s + VCHUNK, spec.nnz)
        vals[s:e] = _val16b(torch.arange(s, e, device="cuda")).half()
    del vals
    A.set_values(None)
    spec.value = _val16b
    check(plan.numeric(), "numeric() after set_values")
    plan.close()


def test_spgemm_refuses_c_of_2_32_values(B, pool):
    """A (2^31 + 2^27 values, one full block per block row) times a dense 32 x 16 B: C would hold 2^32 + 2^28 values.  The product
    fails with BMSP_ERR_TOO_LARGE before C's values are allocated: the pool's high-water mark stays below their size, and used
    memory returns to its baseline."""
    from bmsparse_spgemm_spmv_b200 import _lib as L
    spec = _case1(F16)
    _need(_matrix_bytes(spec.nblk, spec.nnz, spec.nbr, 2) + spec.nnz * 2 + 8 * GB, "A and the symbolic product")
    A = _build(B, spec)
    c_values = 2 * spec.nnz * 4
    assert 2 * spec.nnz == TWO32 + (1 << 28)
    gc.collect(); torch.cuda.synchronize()
    base = pool.get(USED_MEM_CURRENT)
    pool.reset_high()
    # B is made and destroyed inside the measurement: the index a product builds for its B operand belongs to B
    Bd = B.bmSpMatrix.from_csr(32, 16, np.arange(0, 33 * 16, 16, dtype=np.int32), np.tile(np.arange(16, dtype=np.int32), 32),
                               np.ones(32 * 16, np.float32), transpose=True, dtype=F16)
    with pytest.raises(L.BmspError) as e:
        B.bmSparse_mult(A, Bd)
    assert e.value.code == 6
    del Bd, e
    gc.collect(); torch.cuda.synchronize()
    peak = pool.get(USED_MEM_HIGH) - base
    print(f"\nPOOL_PEAK spgemm_too_large {peak}")
    assert peak < c_values, f"{peak} bytes at the peak, C's values would take {c_values}"
    assert pool.get(USED_MEM_CURRENT) == base, "the refused product kept memory"


# ---------------------------------------------------------------------------------------------------------------- 6: int32 coordinates
def _few_blocks(rows, cols, br, bc, bmps, value=_val16):
    br = torch.tensor(br, dtype=torch.int64, device="cuda"); bc = torch.tensor(bc, dtype=torch.int64, device="cuda")
    keys = (br << 32) | bc
    o = torch.argsort(keys)
    bm = torch.tensor(np.array([w & (2 ** 64 - 1) for w in bmps], np.uint64).view(np.int64), device="cuda")[o]
    cnt = torch.tensor([bin(int(w) & (2 ** 64 - 1)).count("1") for w in bm.tolist()], dtype=torch.int64, device="cuda")
    offsets = torch.zeros(len(bmps) + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(cnt, 0, out=offsets[1:])
    return Spec(rows, cols, keys[o], bm, offsets, value, F16)


def _sparse_check(B, M, spec, x, n_out, transpose=False, run=None):
    """y = M x over n_out rows (up to 2^31 - 1): the rows the reference touches equal it, every other row is 0.  run(M, x, y) computes
    the product (default bmSparse_SpMV).  Returns the touched rows and their float64 values."""
    rows, vals = [], []
    for r, v, va in _ref_parts(spec, x, transpose):
        keep = (r >= 0) & (r < n_out)
        assert not ((v != 0) & ~keep).any() and float(va.max()) < 2 ** 24
        rows.append(r[keep]); vals.append(v[keep])
    rows, inv = torch.unique(torch.cat(rows), return_inverse=True)
    ref = torch.zeros(rows.numel(), dtype=torch.float64, device="cuda").index_add_(0, inv, torch.cat(vals))
    ybuf = _y_buffer(n_out)
    y = ybuf[PAD:PAD + n_out]
    (run or B.bmSparse_SpMV)(M, x, y)
    got = y[rows].double()
    assert torch.equal(got, ref), f"touched rows differ: {got[got != ref][:4].tolist()} vs {ref[got != ref][:4].tolist()}"
    nz = int(torch.count_nonzero(y))          # NaN counts as nonzero: a row left unwritten shows up here
    assert nz == int(torch.count_nonzero(ref)), f"{nz} nonzero rows, expected {int(torch.count_nonzero(ref))}"
    assert bool((ybuf[:PAD] == SENTINEL).all()) and bool((ybuf[PAD + n_out:] == SENTINEL).all())
    return rows, ref


ROWS7 = 0xFFFFFFFFFFFFFF00          # rows 0 .. 6 of a block
COLS7 = int.from_bytes(bytes([0xFE] * 8), "big")    # columns 0 .. 6


def _x_formula(n, dtype):
    """x[j] = (j mod 13) - 6, in steps of 2^27 elements"""
    def fill(xs):
        for s in range(0, n, VCHUNK):
            e = min(s + VCHUNK, n)
            xs[s:e] = (torch.arange(s, e, device="cuda") % 13 - 6).to(dtype)
    return _x_buffer(n, dtype, fill)


def test_int32_coordinate_limits(B):
    """rows = 2^31 - 1 with blocks in the last, partial block row; cols = 2^31 - 1 with blocks in the last, partial block column
    (fp16 x); both multiplied, transposed in both forms, and their transposes multiplied, every result exact"""
    last = (INT32_MAX + 7) // 8 - 1
    _need(INT32_MAX * 6 + (last + 1) * 32 + 2 * GB, "vectors of 2^31 - 1 elements")
    tall = _few_blocks(INT32_MAX, 16, [0, last, last, last // 2], [1, 0, 1, 0],
                       [FULL, ROWS7, ROWS7 & 0x5A5A5A5A5A5A5A5A, 0x8000000000000001])
    wide = _few_blocks(16, INT32_MAX, [0, 1, 1, 0], [0, last, last // 2, last],
                       [FULL, COLS7, 0x0102040810204080, COLS7 & 0x00FF00FF00FF00FF])
    for spec in (tall, wide):
        M = _build(B, spec)
        plan_info(M)
        nx, ny = spec.cols, spec.rows
        x = _small_x(nx, F32, seed=9) if nx == 16 else _x_formula(nx, F16)
        _sparse_check(B, M, spec, x, ny)
        expect_t = lambda br, bc, spec=spec: spec.cells(spec.lookup(bc, br)).transpose(1, 2)
        every = lambda T: torch.arange(T.block_num, device="cuda")
        Tt = M.matrix_transpose(transpose=True)
        assert (Tt.num_rows, Tt.num_cols) == (spec.cols, spec.rows)
        _check_blocks(Tt, every(Tt), expect_t)
        del Tt
        T = M.matrix_transpose()
        _check_blocks(T, every(T), expect_t)
        del M, x
        xt = _small_x(ny, F32, seed=10) if ny == 16 else _x_formula(ny, F16)
        _sparse_check(B, T, spec, xt, nx, transpose=True)
        del T, xt


# ---------------------------------------------------------------------------------------------------------------- 7: block-parallel
@pytest.mark.skipif(os.environ.get("BMSP_LARGE_TESTS") != "1", reason="about 90 GB of device memory: set BMSP_LARGE_TESTS=1")
def test_block_parallel_past_2_31(B):
    """2^31 + 2^27 values at two cells per block (the block-parallel path): 2^30 + 2^26 blocks, eight per block row"""
    nblk = (1 << 30) + (1 << 26)
    nbr = nblk // 8
    nnz = 2 * nblk
    _need(_matrix_bytes(nblk, nnz, nbr, 2) + nblk * 24 + nnz * 2 + nbr * 8 * 16 + nblk * 16 + 8 * GB, "2^30 + 2^26 blocks")
    pats = torch.tensor([(1 << (63 - a)) | (1 << (63 - b)) for a, b in [(0, 9), (3, 60), (17, 40), (62, 63), (8, 15), (27, 36)]],
                        dtype=torch.int64, device="cuda")
    keys = torch.empty(nblk, dtype=torch.int64, device="cuda")
    bmps = torch.empty(nblk, dtype=torch.int64, device="cuda")
    for s in range(0, nblk, VCHUNK):
        b = torch.arange(s, min(s + VCHUNK, nblk), device="cuda")
        keys[s:s + b.numel()] = ((b // 8) << 32) | (b % 8)
        bmps[s:s + b.numel()] = pats[(b * 7 + (b >> 11)) % pats.numel()]
    offsets = torch.arange(0, 2 * nblk + 1, 2, device="cuda")
    spec = Spec(8 * nbr, 64, keys, bmps, offsets, _val16, F16)
    M = _build(B, spec)
    assert plan_info(M).path == 1
    x = _small_x(64, F16, seed=11)
    _spmv_exact(B, M, x, _ref_spmv(spec, x, spec.rows), "block-parallel")


# ---------------------------------------------------------------------------------------------------------------- 8: halo paths at 2^31 - 1 rows
class _Rows:
    """y over [0, n) given by its nonzero rows: a slice [lo:hi] is the dense float64 rows lo .. hi - 1"""

    def __init__(self, rows, vals):
        self.rows, self.vals = rows.cpu().numpy(), vals.cpu().numpy()

    def __getitem__(self, s):
        out = np.zeros(s.stop - s.start)
        m = (self.rows >= s.start) & (self.rows < s.stop)
        out[self.rows[m] - s.start] = self.vals[m]
        return out


def _tall_ranges(last):
    """rows [0, 8), a range around the middle block row, and the last 1001 rows up to 2^31 - 1"""
    mid = (last // 2) * 8
    return [(0, 8), ((mid - 12) & ~3, mid + 21), ((INT32_MAX - 1001) & ~3, INT32_MAX)]


@pytest.mark.parametrize("kernel", ["streaming", "per_tile", "block_parallel"])
def test_halo_product_at_int32_rows(B, monkeypatch, kernel):
    """bmsp_spmv_halo on a matrix of 2^31 - 1 rows with blocks in block row 0, in the middle block row and in the last, partial
    block row; push ranges [0, 8), one around the middle block row and one ending at 2^31 - 1, each into a guarded sink.  y is
    checked as _sparse_check does; the sinks, their guards, the peer slots and scratch as test_gpu_spmv_halo does.  The streaming
    kernel, the per-tile kernel (BMSP_SPMV_KERNEL=1) and the block-parallel path (one or two cells per block: wait kernel, product,
    push kernel)"""
    last = (INT32_MAX + 7) // 8 - 1
    _need(INT32_MAX * 6 + (last + 1) * 32 + 2 * GB, "vectors of 2^31 - 1 elements")
    if kernel == "block_parallel":
        bmps = [(1 << 63) | (1 << 54), 1 << 43, (1 << 15) | (1 << 8), 1 << 13]
    else:
        bmps = [FULL, 0x8000000000000001, ROWS7, ROWS7 & 0x5A5A5A5A5A5A5A5A]
    spec = _few_blocks(INT32_MAX, 16, [0, last // 2, last, last], [1, 0, 0, 1], bmps)
    M = _build(B, spec)
    if kernel == "per_tile":
        monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
    info = plan_info(M)
    monkeypatch.delenv("BMSP_SPMV_KERNEL", raising=False)
    assert (info.path, info.kernel if info.path == 0 else -1) == {"streaming": (0, 0), "per_tile": (0, 1), "block_parallel": (1, -1)}[kernel]
    x = _small_x(16, F32, seed=12)
    h = Halo(_tall_ranges(last), (0, 16))
    from bmsparse_spgemm_spmv_b200 import _lib as L
    run = lambda M, x, y: L.check(_spmv_halo(M, x.data_ptr(), y.data_ptr(), h.desc, 1, 2))
    rows, ref = _sparse_check(B, M, spec, x, INT32_MAX, run=run)
    torch.cuda.synchronize()
    h.check(_Rows(rows, ref), 2, kernel)


def test_halo_push_at_int32_rows(B):
    """bmsp_halo_push with rows = 2^31 - 1: a range ending at 2^31 - 1 (the push loop's last rows) next to [0, 8), and no range at
    all with peers (the loop must skip its body and still signal)"""
    _need(INT32_MAX * 4 + 2 * GB, "y of 2^31 - 1 elements")
    y = torch.empty(INT32_MAX, device="cuda")            # only the pushed rows are read
    lo = (INT32_MAX - 1001) & ~3
    vals = {0: torch.arange(1, 9, dtype=torch.float64), lo: -torch.arange(1, INT32_MAX - lo + 1, dtype=torch.float64)}
    for a, v in vals.items():
        y[a:a + v.numel()] = v.float().cuda()
    yref = _Rows(torch.cat([torch.arange(a, a + v.numel()) for a, v in vals.items()]), torch.cat(list(vals.values())))
    for ranges, epoch in (([(lo, INT32_MAX), (0, 8)], 3), ([], 4)):
        h = Halo(ranges, (0, 16))
        from bmsparse_spgemm_spmv_b200 import _lib as L
        L.check(_halo_push(y.data_ptr(), INT32_MAX, h.desc, epoch))
        torch.cuda.synchronize()
        h.check(yref, epoch, f"{len(ranges)} ranges")
