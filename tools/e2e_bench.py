"""End-to-end SpMV through bmsp_spmv_host (x and y in pinned host memory) on P4096: wall time per step of the chunked
pipeline, next to the unpipelined copy / launch / copy sequence.
usage: python tools/e2e_bench.py [grid] [reps]"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bmsparse_spgemm_spmv_b200 as B  # noqa: E402

G = B.generators
m = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
nr, nc, rp, ci, v = G.poisson5pt(m, m)
d = lambda a: torch.from_numpy(a).cuda()
A = B.bmSpMatrix.from_csr(nr, nc, d(rp), d(ci), d(v))
xp = torch.from_numpy(G.x_vector(nc)).pin_memory()
yp = torch.empty(nr).pin_memory()
xd = torch.empty(nc, device="cuda"); yd = torch.empty(nr, device="cuda")


def piped():
    B.bmSparse_SpMV_host(A, xp, yp)
    torch.cuda.current_stream().synchronize()


def plain():
    xd.copy_(xp, non_blocking=True)
    B.bmSparse_SpMV(A, xd, yd)
    yp.copy_(yd, non_blocking=True)
    torch.cuda.current_stream().synchronize()


for name, fn in (("pipelined", piped), ("plain", plain)):
    for _ in range(3):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    ms = (time.perf_counter() - t0) / reps * 1e3
    print(f"E2E {name} grid={m} ms={ms:.3f} GBps={A.spmv_bytes() / ms / 1e6:.1f} "
          f"link_GBps_each_way={nr * 4 / ms / 1e6:.1f}")
