"""GPU: one process driving two devices, first in turn and then from two threads at once.

Kernel attributes, device properties and the memory pool's setting belong to one device, so the library keeps them per device.  The
sequence below runs every entry point family on one device: the conversion, SpMV on each of its kernels (the streaming kernel with a
palette, with a stage above the 48 KB of dynamic shared memory a kernel gets without asking, the per-tile kernel and the
block-parallel kernel), the host-buffer pipeline with its graph replay, SpGEMM with the heavy-row split on a side stream, a SpGEMM
plan's numeric(), the transpose and the addition.  Every result on device 1, and every result of the two-thread runs, must equal
device 0's bit for bit.  The SpGEMM inputs have small dyadic values, so that C's sums are exact whatever order its atomics take.
The two-device cases are skipped with fewer than two devices; two threads on one device need one."""
import threading

import numpy as np
import pytest
import torch

from tests.test_gpu_spgemm_paths import _plan

pytestmark = pytest.mark.gpu
two_devices = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _up8(v):
    return (v + 7) & ~7


def _up16(v):
    return (v + 15) & ~15


def _stream_stage_smem(nr, rp, ci, smem_per_sm):
    """the streaming kernel's dynamic shared memory for an fp16 matrix and fp32 x (spmv.cu plan_tiles, stage_layout and
    launch_stream_kernel), for a matrix whose tile maxima fit plan_tiles' 40 KB budget and that has no bitmap palette"""
    rows = np.repeat(np.arange(nr), np.diff(rp))
    blk = np.unique((rows // 8).astype(np.int64) << 32 | (ci // 8))
    tile = (blk >> 32) // 64
    nb = np.bincount(tile)
    nv = np.bincount(rows // 8 // 64)
    nl = np.bincount(np.unique(tile << 32 | (blk & 0xFFFFFFFF) >> 2) >> 32)
    nbr = (nr + 7) // 8
    assert ci.size / blk.size >= 2.5 and (blk.size * 26 + ci.size * 2) / nbr + 8 <= 320, "row-tiled path, 64-block-row tiles"
    cb, cv, cl = _up8(int(nb.max())), _up8(int(nv.max())), int(nl.max())
    tile_total = _up16((cb + 2) * 8 + (cb + 16) * 2 + (cv + 16) * 2 + 66 * 8 + cl * 33 * 4) + 16
    assert tile_total <= 40 * 1024, "capacities are the tile maxima"
    xo = _up16(16 + (cb + 2) * 8); val = _up16(xo + (cb + 16) * 2); row = _up16(val + (cv + 16) * 2); xs = _up16(row + 66 * 8)
    per_stage = ((xs + cl * 32 * 4 + 16 + 127) & ~127) + 16
    fixed = 8 * 64 + 64
    for c in range(7, 0, -1):
        per_cta = min(smem_per_sm // c - 1280, 227 * 1024)
        fit = (per_cta - fixed) // per_stage if per_cta > fixed else 0
        if fit >= 2 or (c == 1 and fit >= 1):
            return min(fit, 8) * per_stage + fixed
    raise AssertionError("no stage fits")


def _large_stage_csr(nbr=4096, ncols=1 << 20, blocks=3, cells=4, seed=11):
    """light block rows of `blocks` blocks with `cells` values each, at scattered block columns: every tile stages ~192 x lines"""
    rng = np.random.default_rng(seed)
    nbc = ncols // 8
    rows, cols = [], []
    for br in range(nbr):
        for bc in rng.choice(nbc, blocks, replace=False):
            cell = rng.choice(64, cells, replace=False)
            rows.append(br * 8 + cell // 8); cols.append(bc * 8 + cell % 8)
    r = np.concatenate(rows); c = np.concatenate(cols)
    o = np.lexsort((c, r)); r, c = r[o], c[o]
    n = nbr * 8
    rp = np.zeros(n + 1, np.int64); np.cumsum(np.bincount(r, minlength=n), out=rp[1:])
    v = rng.uniform(-1, 1, r.size).astype(np.float16).astype(np.float32)
    v[v == 0] = 0.5
    return n, ncols, rp.astype(np.int32), c.astype(np.int32), v


def _dyadic(n, seed):
    return np.random.default_rng(seed).choice(np.array([-2, -1.5, -1, -0.5, 0.5, 1, 1.5, 2], np.float32), n)


@pytest.fixture(scope="module")
def inputs(B, oracle):
    G = B.generators
    nr, nc, rp, ci, _ = G.poisson5pt(64, 64)
    stencil = (nr, nc, rp, ci, _dyadic(ci.size, 1))
    p = _plan((nr, nc), (rp, ci), (nr, nc), (rp, ci))
    heavy = p["max_cand"] // 4
    assert heavy > 0 and int((p["cand"] >= heavy).sum()) > 0          # BMSP_SPGEMM_HEAVY=heavy runs the split
    large = _large_stage_csr()
    assert np.unique(oracle.csr_to_bmsp(*large).bmps).size > 256       # no palette
    for d in range(min(2, torch.cuda.device_count())):
        smem = _stream_stage_smem(large[0], large[2], large[3], torch.cuda.get_device_properties(d).shared_memory_per_multiprocessor)
        assert smem > 48 * 1024, smem
    return dict(stencil=stencil, stencil_v2=_dyadic(ci.size, 2), heavy=heavy, clustered=G.block_clustered(300),
                uniform=G.uniform_random(4096, 16), large=large)


def _products(B, inp):
    """the sequence on the current device and stream; every result as numpy arrays"""
    st = torch.cuda.current_stream()
    out = {}
    A = B.bmSpMatrix.from_csr(*inp["stencil"])
    out["from_csr"] = A.download()
    for name in ("stencil", "clustered", "uniform", "large"):
        M = A if name == "stencil" else B.bmSpMatrix.from_csr(*inp[name])
        x = torch.tensor(B.generators.x_vector(M.num_cols), device="cuda")
        out["spmv_" + name] = B.bmSparse_SpMV(M, x).cpu().numpy()
    xh = torch.tensor(B.generators.x_vector(A.num_cols)).pin_memory()
    yh = torch.empty(A.num_rows, dtype=torch.float32).pin_memory()
    for k in range(2):                                   # eager, then captured and replayed
        B.bmSparse_SpMV_host(A, xh, yh)
        st.synchronize()
        out[f"spmv_host_{k}"] = yh.numpy().copy()
    Bt = B.bmSpMatrix.from_csr(*inp["stencil"], transpose=True)
    C, _ = B.bmSparse_mult(A, Bt)
    out["spgemm"] = C.download()
    plan = B.bmSparse_mult_plan(A, Bt)
    nr, nc, rp, ci, _ = inp["stencil"]
    A.set_values_csr(rp, ci, inp["stencil_v2"]); Bt.set_values_csr(rp, ci, inp["stencil_v2"])
    plan.numeric()
    out["plan_numeric"] = plan.C.download()
    At = A.matrix_transpose()
    out["transpose"] = At.download()
    out["add"] = B.bmSparse_add(A, At, 1.0, -0.5).download()
    st.synchronize()
    return out


def _sequence(B, inp, dev, stream=False):
    """_products on device dev: on its current stream, or on a new stream of its own"""
    with torch.cuda.device(dev):
        s = torch.cuda.Stream() if stream else torch.cuda.current_stream()
        with torch.cuda.stream(s):
            return _products(B, inp)


def _assert_same(got, ref, what):
    assert got.keys() == ref.keys()
    for k in ref:
        g, r = (got[k], ref[k]) if isinstance(ref[k], tuple) else ((got[k],), (ref[k],))
        for i, (a, b) in enumerate(zip(g, r)):
            assert a.dtype == b.dtype and np.array_equal(a, b), f"{what}: {k}[{i}] differs"


@two_devices
def test_devices_in_turn(B, inputs, monkeypatch):
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", str(inputs["heavy"]))
    ref = _sequence(B, inputs, 0)
    _assert_same(_sequence(B, inputs, 1), ref, "device 1")
    _assert_same(_sequence(B, inputs, 0), ref, "device 0 again")


@pytest.mark.parametrize("devs", [pytest.param((0, 1), marks=two_devices), (0, 0)], ids=["two-devices", "one-device"])
def test_two_threads(B, inputs, monkeypatch, devs):
    """two threads, each on its device and a stream of its own, running the sequence three times; ctypes releases the GIL during
    the library's calls, so they overlap"""
    monkeypatch.setenv("BMSP_SPGEMM_HEAVY", str(inputs["heavy"]))
    ref = _sequence(B, inputs, 0)
    results, errors = [[], []], []

    def work(i):
        try:
            for _ in range(3):
                results[i].append(_sequence(B, inputs, devs[i], stream=True))
        except BaseException as e:       # re-raised in the main thread
            errors.append(e)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    for i, runs in enumerate(results):
        assert len(runs) == 3
        for k, got in enumerate(runs):
            _assert_same(got, ref, f"thread {i} on device {devs[i]}, run {k}")
