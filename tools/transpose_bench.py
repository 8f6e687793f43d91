#!/usr/bin/env python
"""bmSpMatrix.matrix_transpose (A^T, plain -> plain, fp16) on the bench.py workloads, against the route it replaces.

Per workload, one JSON line:
  transpose_ms      median of --reps calls (CUDA events around the call; one untimed call first: pool growth, module load)
  bytes             algorithmic bytes: A's keys, bitmaps, offsets and values read, A^T's written, plus the derived arrays
                    (block columns, k-masks, block-row pointers, block-row value offsets) written.  The radix sort's traffic
                    (digit histograms, scans, (column, index) pairs moved once per pass) is not counted.
  copy_ms           a device-to-device cudaMemcpyAsync (torch copy_) of bytes / 2, so that it reads and writes the same bytes in all;
                    bytes / copy_ms is the copy rate of this card in this run
  route_ms          median of --route-reps of to_csr() -> torch CSR transpose on the device (.t().to_sparse_csr()) -> from_csr
  bit_exact         A^T equals from_csr of that transposed CSR in all four arrays, bit for bit
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


def algorithmic_bytes(A):
    v = A._view()
    nblk, nnz = v.block_num, v.nnz
    vb = 2 if v.dtype == B._lib.F16 else 4
    nbr_t = (v.num_cols + 7) // 8
    arrays = 2 * (3 * 8 * nblk + vb * nnz)                      # keys, bitmaps, offsets, values: read from A, written to A^T
    derived = nblk * (4 + 1) + (nbr_t + 1) * (4 + 4)            # block columns, k-masks; block-row pointers, block-row value offsets
    return arrays + derived


def route(A):
    rp, ci, vals = A.to_csr()
    S = torch.sparse_csr_tensor(rp, ci, vals, size=(A.num_rows, A.num_cols))
    T = S.t().to_sparse_csr()
    return B.bmSpMatrix.from_csr(A.num_cols, A.num_rows, T.crow_indices(), T.col_indices(), T.values())


def same(X, Y):
    for name in ("keys", "bmps", "offsets"):
        a, b = getattr(X, name), getattr(Y, name)
        if a.shape != b.shape or not torch.equal(a, b):
            return False
    return torch.equal(X.values.view(torch.int16), Y.values.view(torch.int16))


def gpu_provenance():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = (s.strip() for s in r.stdout.strip().splitlines()[0].split(","))
    except Exception as e:          # the name from torch at least
        name, power = torch.cuda.get_device_name(), f"unknown ({e.__class__.__name__})"
    return name, power


def run(name, reps, route_reps, gpu, power):
    desc, make = WORKLOADS[name]
    t = time.perf_counter()
    nr, nc, rp, ci, v = make()
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    del rp, ci, v
    torch.cuda.synchronize()
    print(f"{name}: {desc}: {nr} x {nc}, nnz {A.nnz}, blocks {A.block_num} (built in {time.perf_counter() - t:.1f} s)", flush=True)
    At = A.matrix_transpose()                               # untimed first call
    torch.cuda.synchronize()
    del At
    ms = events_ms(A.matrix_transpose, reps)
    nbytes = algorithmic_bytes(A)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device="cuda"); dst = torch.empty_like(src)
    dst.copy_(src)
    copy = events_ms(lambda: dst.copy_(src), reps)
    del src, dst
    R = route(A)                                            # warm the route (torch's sparse kernels, pool)
    del R
    torch.cuda.synchronize()
    route_ms = events_ms(lambda: route(A), route_reps)
    At = A.matrix_transpose()
    R = route(A)
    torch.cuda.synchronize()
    exact = same(At, R)
    med, cmed = float(np.median(ms)), float(np.median(copy))
    rec = {"workload": name, "desc": desc, "rows": nr, "cols": nc, "nnz": A.nnz, "blocks": A.block_num, "form": "plain -> plain, fp16",
           "transpose_ms": round(med, 4), "transpose_ms_min": round(float(ms.min()), 4), "transpose_ms_max": round(float(ms.max()), 4),
           "reps": reps, "bytes": nbytes, "bytes_note": "algorithmic (arrays read + written, derived arrays written); radix-sort traffic not counted",
           "transpose_GBps": round(nbytes / (med * 1e-3) / 1e9, 1), "copy_ms": round(cmed, 4),
           "copy_GBps": round(nbytes / (cmed * 1e-3) / 1e9, 1), "frac_of_copy": round(cmed / med, 3),
           "route_ms": round(float(np.median(route_ms)), 3), "route_reps": route_reps, "speedup_vs_route": round(float(np.median(route_ms)) / med, 1),
           "route": "to_csr -> torch sparse_csr .t().to_sparse_csr() -> from_csr", "bit_exact": bool(exact),
           "gpu": gpu, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def kernels(name, reps=5):
    """Per-kernel device time of matrix_transpose (torch.profiler, a run of its own: tracing slows the host), mean of reps calls"""
    from torch.profiler import ProfilerActivity, profile
    nr, nc, rp, ci, v = WORKLOADS[name][1]()
    A = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    del rp, ci, v
    A.matrix_transpose()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            A.matrix_transpose()
        torch.cuda.synchronize()
    rows = [(e.key, e.device_time_total / reps / 1e3, e.count // reps) for e in prof.key_averages() if e.device_time_total > 0]
    rows.sort(key=lambda r: -r[1])
    print(f"{name}: per call, ms (launches)")
    for k, ms, n in rows:
        print(f"  {ms:8.4f}  ({n:2d})  {k[:110]}")
    print(f"  {sum(r[1] for r in rows):8.4f}  total", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--route-reps", type=int, default=5)
    ap.add_argument("--kernels", action="store_true", help="print the per-kernel breakdown instead of timing")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r3_transpose.json"))
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
    if not all(r["bit_exact"] for r in recs):
        raise SystemExit("A^T differs from the transposed CSR's conversion")
