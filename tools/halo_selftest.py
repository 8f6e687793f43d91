"""One-GPU timing of the fused multi-GPU SpMV code path (bmsp_spmv_halo) with the rank as its own peer: the flags it waits for are
already past the epoch, its pushes land in a scratch buffer.  Isolates what the halo variant of the kernel costs from what the
exchange protocol costs (the difference to a real 2-GPU step).  usage: python tools/halo_selftest.py [steps]"""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bmsparse_spgemm_spmv_b200 as B  # noqa: E402
from bmsparse_spgemm_spmv_b200 import _lib as L  # noqa: E402

G = B.generators
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
GRID = 4096
nr, nc, rp, ci, v = G.poisson5pt(GRID, GRID)
d = lambda a: torch.from_numpy(a).cuda()
A = B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v))
x = d(G.x_vector(nc)); y = torch.empty(nr, device="cuda")
flags = torch.full((64,), 1 << 30, dtype=torch.int32, device="cuda")      # "peer" slots: already far past every epoch we wait for
out_flags = torch.zeros(64, dtype=torch.int32, device="cuda")
scratch = torch.zeros(4, dtype=torch.int32, device="cuda")
sink = torch.zeros(2 * GRID + 64, device="cuda")
desc = L.HaloDesc()
desc.n_push = 2
desc.push_lo[0] = 0; desc.push_hi[0] = GRID; desc.push_dst[0] = sink.data_ptr()
desc.push_lo[1] = nr - GRID; desc.push_hi[1] = nr; desc.push_dst[1] = sink.data_ptr() + GRID * 4
desc.n_peer = 2
for i in range(2):
    desc.peer_flag[i] = out_flags.data_ptr() + 4 * i; desc.my_flag[i] = flags.data_ptr() + 4 * i
desc.scratch = scratch.data_ptr()
desc.own_col_lo = GRID; desc.own_col_hi = nc - GRID          # the first / last grid row of columns count as a neighbour's
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)


def timeit(fn):
    for _ in range(10):
        fn()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / steps * 1e3


ep = [1]


def halo_step():
    L.check(L.lib().bmsp_spmv_halo(A._h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), C.byref(desc), ep[0], ep[0] + 1, st))
    ep[0] += 1


plain = timeit(lambda: B.bmSparse_SpMV(A, x, y)) if os.environ.get("HALO_ONLY", "0") != "1" else float("nan")
B.bmSparse_SpMV(A, x, y)
y_ref = y.clone()
halo = timeit(halo_step)
torch.cuda.synchronize()
ok = torch.equal(y, y_ref) and torch.equal(sink[:GRID], y_ref[:GRID]) and torch.equal(sink[GRID:2 * GRID], y_ref[nr - GRID:])
print(f"HALO_SELFTEST plain_us={plain:.2f} halo_variant_us={halo:.2f} "
      f"results_match={ok} signalled_epoch={int(out_flags[0])}")
