#!/usr/bin/env python
"""SpGEMM A*A reuse: what a plan (bmSparse_mult_plan) saves when the same product is formed again with new values.

Per config: the one-shot bmSparse_mult (wall, symbolic, numeric), plan creation (wall) and the device memory the plan keeps,
set_values_csr on A and on B (CUDA events, with its algorithmic bytes and the rate they imply against the HBM data-sheet peak),
plan.numeric() (CUDA events, every rep timed on its own), and the largest difference between the reused C and a fresh product of
the updated operands, relative to sum |a||b| of the entry.

set_values_csr bytes, defined here: CSR in (row_ptr, col_idx, fp32 values) + fp16 values out + the block metadata read once (block-row
pointers, block columns, bitmaps, offsets).  The call also checks the pattern in a first pass (it reads the metadata and col_idx
twice in all), reads one flag back, and rewrites B's packed records, so its rate is a floor on the scatter's."""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bmsparse_spgemm_spmv_b200 as B

G = B.generators
HBM_PEAK = 7.7e12          # B/s, HGX B200 data sheet, one GPU

CONFIGS = {"P4096": lambda: G.poisson5pt(4096, 4096), "U1M": lambda: G.uniform_random(1_000_000, 16, seed=2),
           "BC4M": lambda: G.block_clustered(524288), "R-MAT-18": lambda: G.rmat(18)}


def events_ms(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return np.array(out)


def set_values_bytes(M, rows, nnz):
    v = M._view()
    return (rows + 1) * 4 + nnz * 4 + nnz * 4 + nnz * 2 + (v.num_block_rows + 1) * 4 + v.block_num * (4 + 8 + 8)


def run(name, reps, numeric_reps):
    nr, nc, rp, ci, v = CONFIGS[name]()
    d = lambda a: torch.from_numpy(a).cuda()
    rp_d, ci_d = d(rp), d(ci)
    A = B.bmSpMatrix.from_csr(nr, nc, rp_d, ci_d, d(v)); Bt = B.bmSpMatrix.from_csr(nr, nc, rp_d, ci_d, d(v), transpose=True)
    print(f"{name}: rows {nr} nnz {ci.size} blocks {A.block_num}", flush=True)
    shots = []
    for _ in range(reps + 1):
        torch.cuda.synchronize(); t = time.perf_counter()
        C, info = B.bmSparse_mult(A, Bt, None, 0, True, 5)
        torch.cuda.synchronize(); shots.append(((time.perf_counter() - t) * 1e3, info.symbolic_ms, info.numeric_ms))
        del C
    s = np.array(shots[1:])
    print(f"  one-shot bmSparse_mult  wall {s[:, 0].min():.2f} ms  symbolic {s[:, 1].min():.2f}  numeric {s[:, 2].min():.2f}   (min of {reps})"
          f"  path {info.numeric_path} surviving {info.surviving_pairs} C blocks {info.c_blocks} C nnz {info.c_nnz}")
    torch.cuda.synchronize(); t = time.perf_counter()
    plan = B.bmSparse_mult_plan(A, Bt)
    torch.cuda.synchronize(); t_plan = (time.perf_counter() - t) * 1e3
    print(f"  plan_create             wall {t_plan:.2f} ms  plan.nbytes {plan.nbytes / 1e6:.1f} MB", flush=True)
    v2 = G.values_fp16(99, ci.size).astype(np.float32)
    v2_d = d(v2)
    for label, M in (("A", A), ("B", Bt)):
        ms = events_ms(lambda: M.set_values_csr(rp_d, ci_d, v2_d), reps + 1)[1:]
        nb = set_values_bytes(M, nr, ci.size)
        print(f"  set_values_csr({label})     {ms.min():.3f} ms (min of {reps}, median {np.median(ms):.3f})  {nb / 1e6:.1f} MB"
              f" -> {nb / (ms.min() * 1e-3) / 1e9:.0f} GB/s = {100 * nb / (ms.min() * 1e-3) / HBM_PEAK:.1f} % of {HBM_PEAK / 1e12:.1f} TB/s")
    for _ in range(3):
        plan.numeric()
    ms = events_ms(plan.numeric, numeric_reps)
    print(f"  plan.numeric()          median {np.median(ms):.3f} ms  min {ms.min():.3f}  max {ms.max():.3f}  ({numeric_reps} reps after 3 warm-up)")
    fresh, _ = B.bmSparse_mult(A, Bt)
    diff = (plan.C.values - fresh.values).abs().double()
    del fresh
    a2 = d(np.abs(v2))
    A.set_values_csr(rp_d, ci_d, a2); Bt.set_values_csr(rp_d, ci_d, a2)
    mag, _ = B.bmSparse_mult(A, Bt)
    rel = float((diff / (mag.values.double() + 1e-30)).max()) if diff.numel() else 0.0
    print(f"  reused vs fresh product: max |diff| / sum|a||b| = {rel:.3e}", flush=True)
    plan.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=list(CONFIGS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--numeric-reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    for n in a.configs:
        run(n, a.reps, a.numeric_reps)
