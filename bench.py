#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark of the bmSparse hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--budget-s S] [--dump-outputs DIR]

Headline (BASELINE.json configs[1]): bmSparse SpMV, fp16 values / fp32 x, y / fp32 accumulate, synthetic
2-D Poisson 4096x4096 grid (16.7M rows, 83.9M nnz) -- metric "SpMV HBM GB/s" = algorithmic bytes of the
compact surface (SURVEY.md 8d: nblk*12 + nbr*8 + nnz*2 + ncols*4 + nrows*4 = 444 452 864 B) / device time.
A step = one SpMV.  N > 1 (torchrun, one rank per GPU): weak scaling, every rank owns one 4096x4096-grid
slab of a 4096 x (4096 N) grid; the SpMV kernel itself pushes its boundary rows of y into the neighbours' next x over
NVLink peer memory (bmsp_spmv_halo; NCCL send/recv when peer mapping is unavailable or BMSP_BENCH_HALO=nccl).
After the timed region the product is VERIFIED at every N: three exchanged products of an integer-valued x against an
independent numpy evaluation of the 5-point stencil on this rank's rows (bit-exact); a mismatch exits non-zero.

The same JSON line carries, measured after the headline and bounded by --budget-s (sections that would not fit are
skipped and say so):
  "spgemm"    N = 1: A*A on the BASELINE configs (U1M headline, BC4M, P4096, P256) -- GFLOP/s including the symbolic phase,
              HBM roofline fraction from the algorithmic bytes of SURVEY.md 8d, and on the same box in the same run the
              reference's own bmSparse CUDA operator (rebuilt for sm_100, oracle/_ref/ref_spgemm) and cuSPARSE SpGEMM;
  "convert"   N = 1: CSR -> bmSparse conversion of P4096 as an HBM roofline fraction (bytes in + bytes out / device time);
  "strong"    every N: strong scaling of R-MAT-22 SpMV, R-MAT-22 A*A (chunked, C reduced to checksums) and P4096 SpMV split
              N ways; the N = 1 run of the same lease is the denominator of the speed-ups.

--impl reference times the reference's own CPU path (cusp host CSR kernels compiled from the reference tree
into oracle/_ref; the oracle port if that library is missing) on the same workload, on every host core.

--dump-outputs DIR writes what the timed path computed in its last step (y of the last SpMV) as DIR/spmv_y.npy, float32
(DIR/spmv_y_rank<r>.npy at N > 1), at most 64 MB in all: an output larger than that is written as a sample at fixed, seeded
positions.  The inputs are the same in every run with the same arguments, so the files of two builds compare element for element.
The JSON line counts the non-finite elements of each file.  At N = 1 every step is y = A x with the same x.  At N > 1 a step is
x <- A x: the 5-point operator's largest eigenvalue is close to 8, so y overflows to inf / NaN after about 40 products, and the
dumps only say something while warmup + steps stays below that.  .gitignore ignores *.npy outside tests/golden/.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = 4096
_OUT = sys.stdout
SPGEMM_N, SPGEMM_K = 1_000_000, 16
T_START = time.perf_counter()
DUMP_BYTES = 64 * 10**6      # --dump-outputs writes at most this much in all (shared by the ranks)
DUMP_SAMPLE = 1 << 22        # elements kept of an output too large to write whole


def dump_outputs(d, outputs, rank, world):
    """Write each output (a tensor or array) as d/<name>.npy in float32 / float64.  One that does not fit its share of DUMP_BYTES
    is written as DUMP_SAMPLE elements at positions drawn with a fixed seed: the same positions in every run.  Returns what was
    written, for the JSON line."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // (world * len(outputs))
    written = {}
    for name, t in outputs.items():
        a = (t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)).ravel()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        total = a.size
        if a.nbytes > share:
            n = min(DUMP_SAMPLE, share // a.itemsize)
            a = a[np.sort(np.random.default_rng(0).choice(total, n, replace=False))]
        fname = f"{name}_rank{rank}.npy" if world > 1 else f"{name}.npy"
        np.save(os.path.join(d, fname), a)
        written[fname] = {"elements": int(a.size), "of": int(total), "sampled": a.size < total, "dtype": str(a.dtype),
                          "nonfinite": int(a.size - np.count_nonzero(np.isfinite(a)))}
    return written


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic(key):
    """DRAM bytes per launch / per call from the committed ncu captures (profiles/traffic.json), or None."""
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tf)).get(key)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """polls NVML (clocks + event reasons) while the timed region runs"""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples = []   # (t, sm_mhz, reasons)
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, r))
            except Exception:
                pass
            time.sleep(0.002)          # ~7 samples in a 14 ms timed region; a tighter poll competes with the launching thread

    def summary(self, t0, t1):
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        where = "timed region"
        if not inside:
            inside = [s for s in self.samples if s[0] <= t1][-5:]
            where = "last samples before the timed region ended (region shorter than the NVML poll)"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0, "where": "nvml unavailable"}
        mask = 0
        for s in inside:
            mask |= s[2]
        reasons = [n for b, n in self.REASONS.items() if mask & b and n != "gpu_idle"]
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(inside), "where": where}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned host buffers of the e2e leg are allocated
    (first touch places their pages on that node): at N > 1 every rank pushes 134 MB per step through host memory, and buffers on
    the far socket were part of why the round-1 e2e step grew 4.6x from N = 1 to N = 8.  Best effort; returns what it did."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"node": node, "bound": False}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": str(e)[:80]}


# ------------------------------------------------------------------------------------------------ CPU baseline / reference arm
def cpu_spmv_baseline(O, nr, nc, rp, ci, v, x, nbytes, reps, slabs=1):
    """reference cusp host CSR SpMV (sequential = thrust::cpp dispatch, and the OMP back-end) on this box's host cores.
    slabs > 1: a step is `slabs` products (the N-GPU workload of the weak-scaling arm: N slabs)."""
    have_ref = O.ref_lib() is not None
    threads = O.use_all_cores()          # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: undo it
    best = None
    for omp in (False, True):
        ts = []
        for i in range(reps + 1):
            t = time.perf_counter()
            for _ in range(slabs):
                if have_ref:
                    O.ref_csr_spmv(nr, nc, rp, ci, v, x, omp=omp)
                else:
                    O.csr_spmv(rp, ci, v, x, threads=threads if omp else 1)
            if i:
                ts.append(time.perf_counter() - t)
        t = float(np.median(ts))
        if best is None or t < best[0]:
            best = (t, threads if omp else 1)
    return {"value": slabs * nbytes / best[0] / 1e9, "unit": "GB/s", "cores": best[1], "kind": "reference" if have_ref else "port",
            "seconds_per_step": best[0], "host_threads_available": threads,
            "sample": f"full workload: {reps} steps of {slabs} CSR SpMV(s) of the {nr}-row slab, fp32, cusp sequential and OMP back-ends, best kept; "
                      f"numerator = the metric's {nbytes} algorithmic bytes per slab"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    from oracle import oracle as O
    from bmsparse_spgemm_spmv_b200 import generators as G
    nr, nc, rp, ci, v = G.poisson5pt(GRID, GRID)
    x = G.x_vector(nc)
    nblk_bytes = 444452864
    steps = args.steps
    O.use_all_cores()
    for _ in range(max(args.warmup, 1)):
        O.ref_csr_spmv(nr, nc, rp, ci, v, x, omp=True) if O.ref_lib() is not None else O.csr_spmv(rp, ci, v, x, threads=O.max_threads())
    base = cpu_spmv_baseline(O, nr, nc, rp, ci, v, x, nblk_bytes, steps, slabs=world)
    line = {"impl": "reference", "metric": "SpMV HBM GB/s", "value": base["value"], "unit": "GB/s", "n_gpus": world,
            "steps": steps, "warmup": max(args.warmup, 1), "ms_per_step": base["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"poisson5pt {GRID}x{GRID} CSR SpMV on host memory (cusp::multiply host path); a step = {world} slab product(s), "
                                   f"the N-GPU arm's workload, on every host core of the box"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_OUT, flush=True)


# ------------------------------------------------------------------------------------------------ verification (every N)
def stencil_expected(rank, world, steps):
    """x_g(i) = small integers; returns (x0 slice of this rank, expected A^steps x_g on this rank's rows) evaluated with numpy in
    float64 on the rank's grid rows extended by `steps` rows on either side (exact: integers far below 2^24)."""
    gy0, gy1 = rank * GRID, (rank + 1) * GRID
    lo, hi = max(0, gy0 - steps), min(GRID * world, gy1 + steps)
    i = np.arange(lo * GRID, hi * GRID, dtype=np.uint64)
    xg = (((i * np.uint64(2654435761)) >> np.uint64(7)) & np.uint64(7)).astype(np.float64).reshape(hi - lo, GRID)
    x0 = xg[gy0 - lo:gy1 - lo].astype(np.float32).ravel().copy()
    for _ in range(steps):
        y = 4.0 * xg
        y[1:, :] -= xg[:-1, :]; y[:-1, :] -= xg[1:, :]; y[:, 1:] -= xg[:, :-1]; y[:, :-1] -= xg[:, 1:]
        xg = y          # rows next to a cut that is not the global boundary are wrong from here on; they never reach the own rows
    return x0, xg[gy0 - lo:gy1 - lo].astype(np.float32).ravel()


def verify(torch, B, rank, world, dev, A, sharded, steps=3):
    x0, exp = stencil_expected(rank, world, steps)
    if world == 1:
        x = torch.from_numpy(x0).to(dev)
        for _ in range(steps):
            x = B.bmSparse_SpMV(A, x)
        got = x
    else:
        sharded.set_x(torch.from_numpy(x0).to(dev))
        for _ in range(steps):
            sharded.step()
        torch.cuda.synchronize()
        sharded.check()
        got = sharded.y_own()
    return bool(torch.equal(got.cpu(), torch.from_numpy(exp)))


# ------------------------------------------------------------------------------------------------ SpGEMM section (N = 1)
def spgemm_algorithmic_bytes(A, Bt, c_blocks, c_nnz, surviving):
    """SURVEY.md 8d: bytes(A) + bytes(B^t) + bytes(C) on the compact surface, plus for every surviving pair and operand one 12-byte
    block metadata read and the block's values (2 * nnz/block on average)."""
    def compact(nblk, nbr, nnz, vsize):
        return nblk * 12 + nbr * 8 + nnz * vsize
    a = compact(A.block_num, A.num_block_rows, A.nnz, 2); b = compact(Bt.block_num, Bt.num_block_rows, Bt.nnz, 2)
    c = compact(c_blocks, A.num_block_rows, c_nnz, 4)
    per_pair = (12 + 2.0 * A.nnz / max(A.block_num, 1)) + (12 + 2.0 * Bt.nnz / max(Bt.block_num, 1))
    return int(a + b + c + surviving * per_pair)


def write_csr(path, nr, nc, rp, ci, v):
    with open(path, "wb") as f:
        np.array([nr, nc, ci.size], np.int64).tofile(f); rp.astype(np.int32).tofile(f); ci.astype(np.int32).tofile(f); v.astype(np.float32).tofile(f)


def run_cusparse(kind, csr, reps):
    exe = os.path.join(ROOT, "tools", "_build", "cusparse_baseline")
    if not os.path.exists(exe):
        return {"unavailable": "tools/_build/cusparse_baseline not built"}
    try:
        out = subprocess.run([exe, kind, csr, str(reps)], capture_output=True, text=True, timeout=600)
    except subprocess.TimeoutExpired:
        return {"error": "timeout"}
    for l in out.stdout.splitlines():
        if l.startswith("CUSPARSE_"):
            t = l.split()
            r = {"ms": float(t[1])}
            if "alg" in t:
                r["alg"] = t[t.index("alg") + 1]
            return r
    return {"error": (out.stdout + out.stderr)[-300:]}


def spgemm_config(name, label, gen, B, torch, O, peak, tmp, with_cpu, reps=3):
    """one BASELINE config: ours (CUDA events around bmSparse_mult), reference bmSparse CUDA, cuSPARSE -- same box, same inputs"""
    nr, nc, rp, ci, v = gen()
    d = lambda a: torch.from_numpy(a).cuda()
    rp_d, ci_d, v_d = d(rp), d(ci), d(v)
    A = B.bmSpMatrix.from_csr(nr, nc, rp_d, ci_d, v_d)
    Bt = B.bmSpMatrix.from_csr(nr, nc, rp_d, ci_d, v_d, transpose=True)
    del rp_d, ci_d, v_d
    rowlen = np.diff(rp).astype(np.int64)
    flops = 2 * int(rowlen[ci].sum())
    times, info, cb, cn = [], None, 0, 0
    for i in range(reps + 1):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        C, info = B.bmSparse_mult(A, Bt, None, 0, True, 5)
        e1.record(); e1.synchronize()
        if i:
            times.append(e0.elapsed_time(e1))
        cb, cn = C.block_num, C.nnz
        del C
    ms = float(np.median(times))
    nbytes = spgemm_algorithmic_bytes(A, Bt, cb, cn, info.surviving_pairs)
    out = {"workload": label, "metric": "SpGEMM GFLOP/s incl. symbolic", "gflops": flops / ms / 1e6, "ms": ms,
           "symbolic_ms": info.symbolic_ms, "numeric_ms": info.numeric_ms, "numeric_path": "mma.sync" if info.numeric_path == 1 else "scalar",
           "flops": flops, "candidate_pairs": info.candidate_pairs, "surviving_pairs": info.surviving_pairs, "c_blocks": cb, "c_nnz": cn,
           "roofline": {"bound": "hbm", "achieved": nbytes / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": nbytes / ms / 1e6 / peak,
                        "algorithmic_bytes": nbytes, "traffic": traffic(f"spgemm_{name}_dram_bytes"),
                        "scope": "whole bmsp_spgemm call (count + fill + numeric passes); algorithmic bytes per SURVEY.md 8d"}}
    # the reference's own bmSparse CUDA operator (comparison leg, like cpu_baseline: runs after our measurement, never on our path)
    if O is not None and O.ref_cuda_bin("ref_spgemm"):
        try:
            k, b, o, vals = A.download(); oa = O.OracleMatrix(nr, nc, k, b, o, vals, False)
            k, b, o, vals = Bt.download(); ob = O.OracleMatrix(nr, nc, k, b, o, vals, True)
            r = O.run_ref_spgemm_digest(oa, ob, tmp, tc_version=5, mode=0, reps=2)
            out["reference_cuda_ms"] = r["us"] / 1e3
            out["reference_cuda"] = {"ms": r["us"] / 1e3, "c_blocks": r["c_blocks"], "c_nnz": r["c_nnz"], "structure_counts_match": r["c_blocks"] == cb and r["c_nnz"] == cn,
                                     "what": "bmSparse_mult<half,float> (default kernel multiplyV15) rebuilt for sm_100, whole call as its main times it (SPGEMM.cu:1274-1280), best of 2"}
            del oa, ob
        except Exception as e:  # noqa: BLE001
            out["reference_cuda"] = {"error": str(e)[-200:]}
    else:
        out["reference_cuda"] = {"unavailable": "oracle/_ref/ref_spgemm not built"}
    csr = os.path.join(tmp, name + ".csr")
    write_csr(csr, nr, nc, rp, ci, v)
    cs = run_cusparse("spgemm", csr, 2)
    os.remove(csr)
    out["cusparse"] = cs
    if "ms" in cs:
        out["cusparse_ms"] = cs["ms"]
    ref_ms = [t for t in (out.get("reference_cuda_ms"), out.get("cusparse_ms")) if t]
    out["faster_than_both"] = bool(ref_ms) and len(ref_ms) == 2 and ms < min(ref_ms)
    if with_cpu and O is not None:
        rows = nr // 16
        srp = rp[:rows + 1]; sci = ci[:srp[-1]]; sv = v[:srp[-1]]
        t = time.perf_counter()
        if O.ref_lib() is not None:
            O.ref_csr_spgemm(rows, nc, srp, sci, sv, nr, nc, rp, ci, v, omp=False, copy=False); kind = "reference"
        else:
            O.csr_spgemm(rows, nc, srp, sci, sv, rp, ci, v); kind = "port"
        dt = time.perf_counter() - t
        sflops = 2 * int(rowlen[sci].sum())
        out["cpu_baseline"] = {"value": sflops / dt / 1e9, "unit": "GFLOP/s", "cores": 1, "kind": kind,
                               "sample": f"first {rows} rows of A times the full B through cusp sequential csr_spgemm ({dt:.2f} s)"}
    del A, Bt
    torch.cuda.empty_cache()
    return out


def convert_section(B, torch, nr, nc, rp, ci, v, peak):
    """CSR -> bmSparse conversion of P4096 with the CSR arrays resident in HBM: the second call (memory pool warm) is timed with CUDA
    events; algorithmic bytes = CSR in (row_ptr, col_idx, fp32 values) + bmSparse out (keys, bmps, offsets, fp16 values, brp, bcol, rvb, kmask)."""
    rp_d, ci_d, v_d = (torch.from_numpy(a).cuda() for a in (rp, ci, v))
    ms = []
    for i in range(3):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        A = B.bmSpMatrix.from_csr(nr, nc, rp_d, ci_d, v_d)
        e1.record(); e1.synchronize()
        if i:
            ms.append(e0.elapsed_time(e1))
        nblk, nbr, nnz = A.block_num, A.num_block_rows, A.nnz
        del A
    t = float(np.min(ms))
    nbytes = (nr + 1) * 4 + nnz * 8 + nblk * 24 + nnz * 2 + (nbr + 1) * 8 + nblk * 5
    return {"workload": "CSR -> bmSparse (fp32 -> fp16), P4096, CSR arrays resident in HBM", "ms": t, "first_call_note": "pool growth and module load are in the first, untimed call",
            "roofline": {"bound": "hbm", "achieved": nbytes / t / 1e6, "peak": peak, "unit": "GB/s", "frac": nbytes / t / 1e6 / peak, "algorithmic_bytes": nbytes,
                         "traffic": traffic("convert_p4096_dram_bytes")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps; --impl reference runs each of them once per CPU back-end (sequential, then OpenMP) and per slab, "
                         "and --budget-s does not bound it")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-spgemm", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--budget-s", type=float, default=float(os.environ.get("BMSP_BENCH_BUDGET_S", "300")),
                    help="wall-clock budget of the whole run; optional sections (spgemm comparisons, strong scaling) that would start after it are skipped")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write y of the last timed SpMV to DIR/spmv_y.npy (float32; a fixed, seeded sample when larger than 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path; --impl reference computes y on the host and does not dump it")
    args.warmup = max(args.warmup, 3)
    # native libraries (NCCL's version banner) print to fd 1: keep the real stdout for the one JSON line only
    global _OUT
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    import bmsparse_spgemm_spmv_b200 as B
    from bmsparse_spgemm_spmv_b200 import generators as G

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup
    peak, peak_src = peaks()
    left = lambda: args.budget_s - (time.perf_counter() - T_START)

    sampler = ClockSampler(local)
    sampler.start()

    # ---- build the workload: one 4096 x 4096-grid slab per rank
    nr, nc, rp, ci, v = G.poisson5pt(GRID, GRID)      # slab template (interior coupling added below for N > 1)
    x_host = G.x_vector(nc, seed=1 + rank)
    sharded = None
    if world == 1:
        A = B.bmSpMatrix.from_csr(nr, nc, torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev), torch.from_numpy(v).to(dev))
        torch.cuda.synchronize()
        x = torch.from_numpy(x_host).to(dev)
        y = torch.empty(nr, dtype=torch.float32, device=dev)
        step = lambda: B.bmSparse_SpMV(A, x, y)
        nbytes = A.spmv_bytes()
        launches_per_step = 1
    else:
        from bmsparse_spgemm_spmv_b200.dist import ShardedSpMV
        # global grid 4096 x (4096*world): this rank's rows, with the +-4096 couplings into the neighbour slabs
        n_glob = nr * world
        base = rank * nr
        i = np.arange(nr, dtype=np.int64) + base
        xg = i % GRID; yg = i // GRID
        cols = np.stack([i - GRID, i - 1, i, i + 1, i + GRID], axis=1)
        valid = np.stack([yg > 0, xg > 0, np.ones(nr, bool), xg < GRID - 1, yg < GRID * world - 1], axis=1)
        vals = np.broadcast_to(np.array([-1, -1, 4, -1, -1], np.float32), (nr, 5))
        lrp = np.zeros(nr + 1, np.int64); np.cumsum(valid.sum(1), out=lrp[1:])
        bounds = np.arange(world + 1, dtype=np.int64) * nr
        sharded = ShardedSpMV(bounds, (lrp.astype(np.int32), cols[valid], vals[valid].copy()), n_glob, device=dev,
                              halo=os.environ.get("BMSP_BENCH_HALO", "auto"))
        sharded.set_x(torch.from_numpy(x_host).to(dev))
        A = sharded.local
        step = sharded.step
        nbytes = A.spmv_bytes()
        launches_per_step = 1
        del i, xg, yg, cols, valid, vals, lrp

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        step()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    t_start = time.perf_counter()
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    barrier()
    t_end = time.perf_counter()
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / K
    clocks = sampler.summary(t_start, t_end)
    # ---- the last timed step's product, before anything below reuses its buffers
    dumped = dump_outputs(args.dump_outputs, {"spmv_y": y if world == 1 else sharded.y_own()}, rank, world) if args.dump_outputs else None

    # ---- kernel-only duration of the dominant kernel (same stream, CUDA events, x resident): N = 1 uses the step itself
    kern_ms = ms_step
    if world > 1:
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        xb, yb = sharded.x[sharded.cur], sharded.own_slice(sharded.x[(sharded.cur + 1) % len(sharded.x)])
        for _ in range(3):
            B.bmSparse_SpMV(A, xb, yb)
        ev0.record()
        for _ in range(K):
            B.bmSparse_SpMV(A, xb, yb)
        ev1.record(); ev1.synchronize()
        kern_ms = ev0.elapsed_time(ev1) / K

    # ---- the result is checked at every N: three exchanged products against an independent stencil evaluation (bit-exact)
    ok_local = verify(torch, B, rank, world, dev, A, sharded)
    if world > 1:
        t = torch.tensor([1 if ok_local else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        verified = bool(int(t.item()))
    else:
        verified = ok_local

    # ---- end to end through the public API with HOST buffers: H2D x, SpMV, D2H y inside the timed region
    ncols_local = nc if world == 1 else A.num_cols
    numa = bind_to_gpu_numa(local) if world > 1 else {"bound": False, "why": "single rank: left to the scheduler"}
    xp = torch.zeros(ncols_local, dtype=torch.float32).pin_memory()
    xoff = 0 if world == 1 else sharded.own_lo - sharded.ext_lo
    xp[xoff:xoff + nr].copy_(torch.from_numpy(x_host))
    yp = torch.empty(nr, dtype=torch.float32).pin_memory()
    Ke = max(3, min(K, 50))

    def e2e_step():
        B.bmSparse_SpMV_host(A, xp, yp)               # H2D of x, the product, D2H of y: pipelined inside the library
        torch.cuda.current_stream().synchronize()     # the caller needs y on the host before the next step

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / Ke
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    sampler.stop_flag = True

    total_bytes = nbytes * world
    value = total_bytes / (ms_step * 1e-3) / 1e9
    kname = "spmv_stream_kernel<__half,float,64,...>" if os.environ.get("BMSP_SPMV_KERNEL", "0") != "1" else "spmv_tile_kernel<__half,float,64,2,12>"
    line = {
        "metric": "SpMV HBM GB/s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 values, f32 x/y/accumulate",
        "data": "synthetic", "verified": verified,
        "config": {"workload": f"bmSparse SpMV, 2-D Poisson 5-point {GRID}x{GRID} grid per GPU ({nr} rows, {A.nnz} nnz, {A.block_num} 8x8 blocks)"
                               + ("" if world == 1 else f"; global grid {GRID}x{GRID * world}, x halo ({sharded.halo_bytes} B in per rank and step) "
                                                             + ("pushed over NVLink peer memory by the SpMV kernel itself (bmsp_spmv_halo)" if sharded.p2p is not None
                                                                else "exchanged with NCCL send/recv before each product")),
                   "algorithmic_bytes_per_step_per_gpu": nbytes,
                   "l2": "inputs larger than L2 (444 MB streamed per step vs 126 MB L2); no flush between steps",
                   "timing": "CUDA events on the launching stream around K steps, max over ranks",
                   "verification": "after the timed region: 3 exchanged products of an integer-valued x == numpy 5-point stencil on this rank's rows, bit for bit, all ranks"},
        "roofline": {"bound": "hbm", "achieved": nbytes / (kern_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": nbytes / (kern_ms * 1e-3) / 1e9 / peak, "traffic": traffic("spmv_stream_p4096_dram_bytes"), "peak_source": peak_src,
                     "frac_of_nominal_8TBs": nbytes / (kern_ms * 1e-3) / 1e9 / 8000.0,
                     "kernel": kname, "kernel_ms": kern_ms},
        "e2e": {"value": total_bytes / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": ncols_local * 4, "d2h_bytes_per_step": nr * 4,
                "ms_per_step": e2e_s * 1e3, "numa": numa, "note": "bmsp_spmv_host: matrix resident in HBM (as in the reference's timed region); every step x comes from pinned host memory in chunks on a copy stream while the row-range launches of the same kernel store y straight into the pinned host buffer (PCIe-bound both ways)"},
        "gpu_launches": K * launches_per_step,
        "clocks": clocks,
    }
    if not verified:
        line["verification_failed_on_rank"] = rank if not ok_local else "another rank"
    if dumped is not None:
        line["dump_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "files": dumped}

    skipped = {}
    O = None
    if rank == 0 and world == 1:
        if not args.no_cpu:
            from oracle import oracle as O
            line["cpu_baseline"] = cpu_spmv_baseline(O, nr, nc, rp, ci, v, x_host, nbytes, 5)
        del A
        torch.cuda.empty_cache()
        line["convert"] = convert_section(B, torch, nr, nc, rp, ci, v, peak)
        if not args.no_spgemm:
            tmp = tempfile.mkdtemp(prefix="bmsp_bench_")
            configs = [("u1m", f"uniform-random {SPGEMM_N}x{SPGEMM_N}, {SPGEMM_K} nnz/row, A*A, fp16 in / fp32 out", lambda: G.uniform_random(SPGEMM_N, SPGEMM_K, seed=2), 25),
                       ("p4096", f"poisson5pt {GRID}x{GRID}, A*A", lambda: (nr, nc, rp, ci, v), 25),
                       ("p256", "poisson5pt 256x256, A*A (BASELINE configs[0] shape)", lambda: G.poisson5pt(256, 256), 6),
                       ("bc4m", "block-clustered 4M x 4M (30 % block occupancy in a 32-block band, 50 % fill), A*A", lambda: G.block_clustered(524288), 90)]
            sp = {}
            for name, label, gen, need_s in configs:
                if left() < need_s:
                    skipped[f"spgemm.{name}"] = f"time budget ({args.budget_s:.0f} s) -- needs about {need_s} s"
                    continue
                try:
                    sp[name] = spgemm_config(name, label, gen, B, torch, O, peak, tmp, with_cpu=(name == "u1m" and not args.no_cpu))
                except Exception as e:  # noqa: BLE001 -- a comparison leg must not take the headline down
                    sp[name] = {"error": str(e)[-300:]}
            line["spgemm"] = dict(sp.get("u1m", {}), configs=sp)      # the U1M result stays at the top level of "spgemm" (round-1 layout)
    if not args.no_strong:
        if sharded is not None:
            sharded.close(); sharded = None
        A = None
        torch.cuda.empty_cache()
        from tools import strong_scaling as S
        try:
            line_strong = S.run(B, G, torch, dist if world > 1 else None, rank, world, dev, left, skipped)
        except Exception as e:  # noqa: BLE001
            line_strong = {"error": str(e)[-300:]}
        if rank == 0:
            line["strong"] = line_strong
    if skipped:
        line["skipped"] = skipped
    if rank == 0:
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        if sharded is not None:
            sharded.check()
            sharded.close()
        dist.barrier()
        dist.destroy_process_group()
    if not verified:
        sys.exit(3)


if __name__ == "__main__":
    main()
