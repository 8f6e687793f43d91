#!/usr/bin/env python
"""bmSparse_add (C = alpha*A + beta*B, fp16 plain) on the bench.py workloads, against the route it replaces.

Workloads: A + A^T on P4096, BC4M, U1M and RM22 (A^T from matrix_transpose, fp16, plain), and A - 0.5*I on P4096.
Per workload, one JSON line:
  add_ms            median of --reps calls (CUDA events around the call, which ends in its own stream synchronisation; one
                    untimed call first: pool growth, module load)
  bytes             algorithmic bytes: both operands' keys, bitmaps, offsets and values read, C's written, plus C's derived arrays
                    (block columns, k-masks, block-row pointers, block-row value offsets) written.  The merge's second pass, the
                    source-block arrays and the tile counts are not counted.
  copy_ms           a device-to-device cudaMemcpyAsync (torch copy_) of bytes / 2, so that it reads and writes the same bytes in all;
                    bytes / copy_ms is the copy rate of this card in this run
  route_ms          median of --route-reps of to_csr() on both operands -> torch.add of the two CUDA sparse-CSR tensors (its alpha
                    scales the second operand) -> from_csr
  equal_to_route    C equals from_csr of the route's sum in all four arrays, bit for bit
and the GPU's name and power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bmsparse_spgemm_spmv_b200 as B

G = B.generators
SPGEMM_N, SPGEMM_K = 1_000_000, 16          # bench.py's U1M sizes

WORKLOADS = {
    "P4096": ("poisson5pt 4096x4096", lambda: _dev(G.poisson5pt(4096, 4096))),
    "BC4M": ("block_clustered(524288)", lambda: G.block_clustered_torch(524288)),
    "U1M": (f"uniform_random({SPGEMM_N}, {SPGEMM_K}, seed=2)", lambda: _dev(G.uniform_random(SPGEMM_N, SPGEMM_K, seed=2))),
    "RM22": ("rmat(22)", lambda: G.rmat_torch(22)),
    "P4096-shift": ("poisson5pt 4096x4096", lambda: _dev(G.poisson5pt(4096, 4096))),
}


def _dev(w):
    nr, nc, rp, ci, v = w
    return nr, nc, torch.from_numpy(rp).cuda(), torch.from_numpy(ci).cuda(), torch.from_numpy(v).cuda()


def events_ms(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); r = fn(); e1.record(); e1.synchronize()
        del r
        out.append(e0.elapsed_time(e1))
    return np.array(out)


def identity(n):
    ar = torch.arange(n + 1, dtype=torch.int32, device="cuda")
    return B.bmSpMatrix.from_csr(n, n, ar, ar[:n], torch.ones(n, dtype=torch.float32, device="cuda"))


def operands(name):
    """(A, second operand, beta, description of the sum)"""
    desc, make = WORKLOADS[name]
    nr, nc, rp, ci, v = make()
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    del rp, ci, v
    if name == "P4096-shift":
        return A, identity(nr), -0.5, desc, "A - 0.5*I, fp16 plain"
    return A, A.matrix_transpose(), 1.0, desc, "A + A^T, fp16 plain"


def algorithmic_bytes(X, Y, Cm):
    def arrays(M):
        v = M._view()
        return 3 * 8 * v.block_num + (2 if v.dtype == B._lib.F16 else 4) * v.nnz
    v = Cm._view()
    derived = v.block_num * (4 + 1) + (v.num_block_rows + 1) * (4 + 4)    # block columns, k-masks; block-row pointers, value offsets
    return arrays(X) + arrays(Y) + arrays(Cm) + derived


def route(X, Y, beta):
    sx = torch.sparse_csr_tensor(*X.to_csr(), size=(X.num_rows, X.num_cols))
    sy = torch.sparse_csr_tensor(*Y.to_csr(), size=(Y.num_rows, Y.num_cols))
    S = torch.add(sx, sy, alpha=beta)
    return B.bmSpMatrix.from_csr(X.num_rows, X.num_cols, S.crow_indices(), S.col_indices(), S.values())


def same(X, Y):
    for name in ("keys", "bmps", "offsets"):
        a, b = getattr(X, name), getattr(Y, name)
        if a.shape != b.shape or not torch.equal(a, b):
            return False
    return X.values.shape == Y.values.shape and torch.equal(X.values.view(torch.int16), Y.values.view(torch.int16))


def gpu_provenance():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = (s.strip() for s in r.stdout.strip().splitlines()[0].split(","))
    except Exception as e:          # the name from torch at least
        name, power = torch.cuda.get_device_name(), f"unknown ({e.__class__.__name__})"
    return name, power


def run(name, reps, route_reps, gpu, power):
    t = time.perf_counter()
    X, Y, beta, desc, form = operands(name)
    torch.cuda.synchronize()
    print(f"{name}: {desc}: {X.num_rows} x {X.num_cols}, nnz {X.nnz} + {Y.nnz}, blocks {X.block_num} + {Y.block_num} "
          f"(built in {time.perf_counter() - t:.1f} s)", flush=True)
    add = lambda: B.bmSparse_add(X, Y, 1.0, beta)
    Cm = add()                                              # untimed first call
    nbytes = algorithmic_bytes(X, Y, Cm)
    nblk, nnz = Cm.block_num, Cm.nnz
    del Cm
    ms = events_ms(add, reps)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device="cuda"); dst = torch.empty_like(src)
    dst.copy_(src)
    copy = events_ms(lambda: dst.copy_(src), reps)
    del src, dst
    R = route(X, Y, beta)                                   # warm the route (torch's sparse kernels, pool)
    del R
    torch.cuda.synchronize()
    route_ms = events_ms(lambda: route(X, Y, beta), route_reps)
    Cm = add()
    R = route(X, Y, beta)
    torch.cuda.synchronize()
    equal = same(Cm, R)
    med, cmed, rmed = float(np.median(ms)), float(np.median(copy)), float(np.median(route_ms))
    rec = {"workload": name, "desc": desc, "sum": form, "rows": X.num_rows, "cols": X.num_cols, "nnz_a": X.nnz, "nnz_b": Y.nnz,
           "blocks_a": X.block_num, "blocks_b": Y.block_num, "blocks_c": nblk, "nnz_c": nnz, "route_nnz_c": R.nnz,
           "add_ms": round(med, 4), "add_ms_min": round(float(ms.min()), 4), "add_ms_max": round(float(ms.max()), 4), "reps": reps,
           "bytes": nbytes, "bytes_note": "algorithmic (both operands' arrays read, C's arrays and derived arrays written)",
           "add_GBps": round(nbytes / (med * 1e-3) / 1e9, 1), "copy_ms": round(cmed, 4), "copy_GBps": round(nbytes / (cmed * 1e-3) / 1e9, 1),
           "frac_of_copy": round(cmed / med, 3), "route_ms": round(rmed, 3), "route_reps": route_reps,
           "speedup_vs_route": round(rmed / med, 1), "route": "to_csr x2 -> torch.add(csr, csr, alpha) -> from_csr",
           "equal_to_route": bool(equal), "gpu": gpu, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def kernels(name, reps=5):
    """Per-kernel device time of bmSparse_add (torch.profiler, a run of its own: tracing slows the host), mean of reps calls"""
    from torch.profiler import ProfilerActivity, profile
    X, Y, beta, _, form = operands(name)
    B.bmSparse_add(X, Y, 1.0, beta)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            B.bmSparse_add(X, Y, 1.0, beta)
        torch.cuda.synchronize()
    rows = [(e.key, e.device_time_total / reps / 1e3, e.count // reps) for e in prof.key_averages() if e.device_time_total > 0]
    rows.sort(key=lambda r: -r[1])
    print(f"{name} ({form}): per call, ms (launches)")
    for k, ms, n in rows:
        print(f"  {ms:8.4f}  ({n:2d})  {k[:110]}")
    print(f"  {sum(r[1] for r in rows):8.4f}  total", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--route-reps", type=int, default=5)
    ap.add_argument("--kernels", action="store_true", help="print the per-kernel breakdown instead of timing")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r3_add.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if a.kernels:
        for n in a.workloads:
            kernels(n)
        raise SystemExit(0)
    gpu, power = gpu_provenance()
    recs = [run(n, a.reps, a.route_reps, gpu, power) for n in a.workloads]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("".join(json.dumps(r) + "\n" for r in recs))
    if not all(r["equal_to_route"] for r in recs):
        raise SystemExit("C differs from the route's sum")
