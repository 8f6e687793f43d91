"""Times bmsp_spmv on one generator config (CUDA events, inputs larger than L2).  BMSP_LIB_PATH selects the library build.
usage: python tools/spmv_bench.py [p4096|p4096v|p2048|s3d|scat|bc|u1m|rmat20] [reps]
p4096v: P4096's pattern with variable coefficients; s3d: 7-point stencil on a 256^3 grid (variable coefficients); scat: a bitmap
palette (eight patterns) at random block columns, 10.2 M blocks -- structure without repeating rows, so the plan keeps block words."""
import ctypes
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bmsparse_spgemm_spmv_b200 as B  # noqa: E402
from bmsparse_spgemm_spmv_b200 import _lib as L  # noqa: E402

G = B.generators


def p4096v():
    nr, nc, rp, ci, _ = G.poisson5pt(4096, 4096)
    return nr, nc, rp, ci, G.values_fp16(7, ci.size)


def stencil3d(n=256):
    """7-point stencil on an n^3 grid, columns already in row order"""
    N = n ** 3
    i = np.arange(N, dtype=np.int32)
    x, y, z = i % n, (i // n) % n, i // (n * n)
    cols = np.stack([i - n * n, i - n, i - 1, i, i + 1, i + n, i + n * n], axis=1)
    valid = np.stack([z > 0, y > 0, x > 0, np.ones(N, bool), x < n - 1, y < n - 1, z < n - 1], axis=1)
    rp = np.zeros(N + 1, np.int64)
    np.cumsum(valid.sum(1), out=rp[1:])
    ci = cols[valid]
    return N, N, rp.astype(np.int32), ci, G.values_fp16(11, ci.size)


def scattered(nbr=3_400_000, seed=5):
    """three blocks per block row at random block columns, each one of eight bitmaps with one cell per row (cell (r, (p + 3 r) % 8)
    of pattern p): a palette of 8 entries, 8 values per block, and rows whose shapes do not repeat"""
    rng = np.random.default_rng(seed)
    nbc = nbr
    bc = np.sort(rng.integers(0, nbc - 2, (nbr, 3)), axis=1) + np.arange(3)
    pat = rng.integers(0, 8, (nbr, 3))
    r = np.arange(8)
    cols = bc[:, None, :] * 8 + (pat[:, None, :] + 3 * r[None, :, None]) % 8          # [block row, row, block]
    N = nbr * 8
    ci = cols.reshape(N * 3).astype(np.int32)
    rp = (np.arange(N + 1, dtype=np.int64) * 3).astype(np.int32)
    return N, nbc * 8, rp, ci, G.values_fp16(13, ci.size)



which = sys.argv[1] if len(sys.argv) > 1 else "p4096"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
gen = {"p4096": lambda: G.poisson5pt(4096, 4096), "p4096v": p4096v, "s3d": stencil3d, "scat": scattered, "p2048": lambda: G.poisson5pt(2048, 2048), "bc": lambda: G.block_clustered(1 << 19),
       "u1m": lambda: G.uniform_random(1_000_000, 16), "rmat20": lambda: G.rmat(20), "rmat22": lambda: G.rmat(22)}[which]
nr, nc, rp, ci, v = gen()
d = lambda a: torch.from_numpy(a).cuda()
A = B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v))
x = d(G.x_vector(nc))
y = torch.empty(nr, dtype=torch.float32, device="cuda")
t0 = time.perf_counter()
B.bmSparse_SpMV(A, x, y)
torch.cuda.synchronize()
plan_ms = (time.perf_counter() - t0) * 1e3
for _ in range(10):
    B.bmSparse_SpMV(A, x, y)
e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    B.bmSparse_SpMV(A, x, y)
e1.record(); e1.synchronize()
us = e0.elapsed_time(e1) / reps * 1e3
nbytes = A.spmv_bytes()


def row_shapes():
    """the plan streams row shapes (bmsp_debug_spmv_shapes; a build without row shapes has no such entry point)"""
    if not hasattr(L.lib(), "bmsp_debug_spmv_shapes"):
        return False
    from bmsparse_spgemm_spmv_b200.matrix import _stream_ptr
    n, w = ctypes.c_int32(), ctypes.c_int32()
    L.check(L.lib().bmsp_debug_spmv_shapes(A._h, ctypes.byref(n), ctypes.byref(w), _stream_ptr()))
    return n.value >= 0


def stream_bytes():
    """bytes the streaming kernel reads and writes per product, counted from the plan's rules (spmv.cu plan_spmv / plan_tiles);
    None when another kernel runs.  Per block: nothing with row shapes, a 4-byte word with a bitmap palette (<= 256 distinct
    bitmaps), else 8 B bitmap + 2 B x offset; per block row 4 B (palette) or 8 B; fp16 values; x and y once; a 64-byte descriptor per
    tile of 64 block rows."""
    nbr, nblk, nnz = (nr + 7) // 8, A.block_num, A.nnz
    if nnz < 2.5 * nblk or (nblk * 26 + nnz * 2) / nbr + 8 > 320:
        return None
    npal = np.unique(A.download()[1]).size
    meta = nblk * 4 + nbr * 4 if npal <= 256 else nblk * 10 + nbr * 8
    if npal <= 256 and row_shapes():
        meta = nbr * 4
    return meta + nnz * 2 + nc * 4 + nr * 4 + (nbr + 63) // 64 * 64


sb = stream_bytes()
sb_txt = f"stream_MB={sb / 1e6:.1f} stream_GBps={sb / us / 1e3:.1f}" if sb else "stream_MB=n/a"
print(f"SPMV {which} shapes={int(bool(sb) and row_shapes())} rows={nr} nnz={A.nnz} blocks={A.block_num} "
      f"us={us:.2f} GBps={nbytes / us / 1e3:.1f} {sb_txt} frac6468={nbytes / us / 1e3 / 6468.3:.3f} first_call_ms={plan_ms:.1f} "
      f"ysum={float(y.double().sum()):.6e}")
