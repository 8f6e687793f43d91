"""Times bmsp_spmv on one generator config (CUDA events, inputs larger than L2).  BMSP_LIB_PATH selects the library build.
usage: python tools/spmv_bench.py [p4096|p2048|bc|u1m|rmat20] [reps]"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bmsparse_spgemm_spmv_b200 as B  # noqa: E402

G = B.generators
which = sys.argv[1] if len(sys.argv) > 1 else "p4096"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
gen = {"p4096": lambda: G.poisson5pt(4096, 4096), "p2048": lambda: G.poisson5pt(2048, 2048), "bc": lambda: G.block_clustered(1 << 19),
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


def stream_bytes():
    """bytes the streaming kernel reads and writes per product, counted from the plan's rules (spmv.cu plan_spmv / plan_tiles);
    None when another kernel runs.  Per block: a 4-byte word with a bitmap palette (<= 256 distinct bitmaps), else 8 B bitmap + 2 B x
    offset; per block row 4 B (palette) or 8 B; fp16 values; x and y once; a 64-byte descriptor per tile of 64 block rows."""
    nbr, nblk, nnz = (nr + 7) // 8, A.block_num, A.nnz
    if nnz < 2.5 * nblk or (nblk * 26 + nnz * 2) / nbr + 8 > 320:
        return None
    npal = np.unique(A.download()[1]).size
    meta = nblk * 4 + nbr * 4 if npal <= 256 else nblk * 10 + nbr * 8
    return meta + nnz * 2 + nc * 4 + nr * 4 + (nbr + 63) // 64 * 64


sb = stream_bytes()
sb_txt = f"stream_MB={sb / 1e6:.1f} stream_GBps={sb / us / 1e3:.1f}" if sb else "stream_MB=n/a"
print(f"SPMV {which} rows={nr} nnz={A.nnz} blocks={A.block_num} "
      f"us={us:.2f} GBps={nbytes / us / 1e3:.1f} {sb_txt} frac6468={nbytes / us / 1e3 / 6468.3:.3f} first_call_ms={plan_ms:.1f} "
      f"ysum={float(y.double().sum()):.6e}")
