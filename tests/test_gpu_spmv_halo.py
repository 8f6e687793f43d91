"""The multi-GPU SpMV entry points (bmsp_spmv_halo, bmsp_halo_push) on one GPU, with the rank as its own peer, in exact arithmetic.

Integer values and integer x with sum_j |a_ij x_j| < 2^24 on every row (test_gpu_spmv_exact.py): y must equal scipy's float64 product
bit for bit, and it is also compared with bmSparse_SpMV.  y sits inside a sentinel buffer.  Every push range gets a slice of its own
in a sink buffer, 16-byte aligned, with at least 16 sentinel floats before and after it: the slice must equal its rows of the exact
y and the guards must be untouched, so a store past either end of a range shows up.

The "peers'" slots of the inbox hold 1 << 30 before each call, so every wait is satisfied at once and no call can spin (except in
the wait test at the end, which a copy engine releases).  After every call: scratch == [0, 0] (the count of signalling tiles was
exact and no wait timed out), every peer slot holds the signalled epoch, the unused slots and the rank's own inbox are unchanged.

Every path runs every range shape: the streaming kernel with and without a palette, the per-tile kernel at the 32- and 16-row tiles
the planner picks for heavy rows, and the block-parallel path (wait kernel, product, push kernel), each with fp16 and fp32 values.
Each input asserts the plan it is written for (bmsp_debug_spmv_plan), and every matrix has rows % 4 != 0."""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from tests.test_gpu_spmv_exact import (PAD, SENTINEL, _block_parallel_pattern, _block_parallel_plan, _buffers, _check, _dense_rows,
                                       _matrix, _reference, _scattered, _streaming, _x, plan_info)

pytestmark = pytest.mark.gpu

HALO_MAX = 8
N_PEER = 2
OWN_MARGIN = 256         # columns at either end of x that count as a peer's
GUARD = 16               # sentinel floats before and after every sink slice (a multiple of 4: slices stay 16-byte aligned)
FAR = 1 << 30            # the peers' epoch in the inbox: every wait is satisfied
INVALID, UNSUPPORTED = 1, 7
VDT = {"v16": torch.float16, "v32": torch.float32}


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _L():
    from bmsparse_spgemm_spmv_b200 import _lib as L
    return L


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------------------------- inputs
def _per_row(rt, vdt):
    """dense blocks per block row that give the per-tile kernel tile height rt (test_per_tile_kernel_dense_blocks)"""
    return {(32, torch.float16): 3, (16, torch.float16): 6, (32, torch.float32): 2, (16, torch.float32): 4}[(rt, vdt)]


def _tile_plan(rt):
    def plan(i):
        assert i.path == 0 and i.kernel == 1 and i.tile_rows == rt
    return plan


# kernel -> (pattern(vdt), plan check)
KERNELS = {
    "stream_palette": (lambda vdt: _scattered(3000, 8 * 20000 + 5, 3, seed=11, distinct=False), lambda i: _streaming(i, palette=True)),
    "stream_bitmaps": (lambda vdt: _scattered(3000, 8 * 20000 + 5, 3, seed=11, distinct=True), lambda i: _streaming(i, palette=False)),
    "tile32": (lambda vdt: _dense_rows(640, 8 * 1500 + 3, _per_row(32, vdt), 150, seed=32), _tile_plan(32)),
    "tile16": (lambda vdt: _dense_rows(640, 8 * 1500 + 3, _per_row(16, vdt), 150, seed=16), _tile_plan(16)),
    "block_parallel": (lambda vdt: _block_parallel_pattern(1001, seed=9), _block_parallel_plan),
}
_CACHE = {}


def _case(B, kernel, vd):
    """(matrix, csr, x on the device, exact y as float64, rows per tile) of one kernel and value dtype, built once per module"""
    key = (kernel, vd)
    if key not in _CACHE:
        vdt = VDT[vd]
        pat_fn, plan = KERNELS[kernel]
        M, csr = _matrix(B, pat_fn(vdt), vdt, seed=len(kernel))
        info = plan_info(M)
        plan(info)
        assert csr[0] % 4 != 0
        x = _x(csr[1], vdt, np.random.default_rng(7))
        xs, _ = _buffers(csr, x, torch.float32)
        rpt = info.tile_rows * 8 if info.path == 0 else 512
        _CACHE[key] = (M, csr, xs, _reference(csr, x), rpt)
    return _CACHE[key]


def _shapes(nr, T):
    """push ranges by name, for a matrix of nr rows and T rows per tile (lo always a multiple of 4)"""
    q = lambda r: r & ~3
    mid = q(nr // 2)
    return {
        "eight_disjoint": [(q(k * nr // 8), q(k * nr // 8) + 4 * k + 3 + (k % 3) * T // 2) for k in range(HALO_MAX)],
        "all_gather_7": [(0, nr)] * 7,
        "nested_overlapping": [(0, 3 * T + 10), (T, 2 * T), (T + 4, T + 8), (2 * T - 100, 4 * T + 7)],
        "tile_edges": [(T + 16, T + 40), (T + 40, T + 101), (2 * T, 2 * T + 50), (3 * T + 4, 3 * T + 9)],
        "mid_quad": [(mid - 8, mid + 30)],
        "empty_among": [(0, 13), (2 * T, 2 * T), (q(nr - 40), nr - 5)],
        "tail": [(q(nr - 777), nr)],
        "none": [],
    }


SHAPES = list(_shapes(10000, 512))


# ---------------------------------------------------------------------------------------------------------------- harness
class Halo:
    """a descriptor for `ranges` with its guarded sink, the inbox (my_flag), the peers' slots (peer_flag) and scratch"""

    def __init__(self, ranges, own_cols, n_peer=N_PEER):
        L = _L()
        self.ranges = list(ranges)
        self.slots, cur = [], 0
        for lo, hi in self.ranges:
            self.slots.append(cur + GUARD)
            cur += GUARD + (hi - lo + 3) // 4 * 4 + GUARD
        self.sink = torch.empty(max(cur, GUARD), device="cuda")
        self.my_flag = torch.zeros(HALO_MAX, dtype=torch.int32, device="cuda")
        self.peer_flag = torch.zeros(HALO_MAX, dtype=torch.int32, device="cuda")
        self.scratch = torch.zeros(4, dtype=torch.int32, device="cuda")
        d = L.HaloDesc()
        d.n_push = len(self.ranges)
        for i, (lo, hi) in enumerate(self.ranges):
            d.push_lo[i] = lo; d.push_hi[i] = hi; d.push_dst[i] = self.sink.data_ptr() + 4 * self.slots[i]
        d.n_peer = n_peer
        for i in range(n_peer):
            d.peer_flag[i] = self.peer_flag.data_ptr() + 4 * i
            d.my_flag[i] = self.my_flag.data_ptr() + 4 * i
        d.scratch = self.scratch.data_ptr()
        d.own_col_lo, d.own_col_hi = own_cols
        self.desc = d
        self.reset()

    def reset(self, inbox=FAR):
        self.sink.fill_(SENTINEL)
        self.my_flag.fill_(0); self.my_flag[:self.desc.n_peer] = inbox
        self.inbox = self.my_flag.clone()

    def check(self, yref, epoch, what=""):
        """sink slices == their rows of yref (float64, exact), guards untouched; the protocol state after signalling `epoch`"""
        exp = np.full(self.sink.numel(), SENTINEL, np.float64)
        for (lo, hi), s in zip(self.ranges, self.slots):
            exp[s:s + hi - lo] = yref[lo:hi]
        got = self.sink.cpu().numpy().astype(np.float64)
        bad = got != exp
        assert not bad.any(), f"{what}: sink differs at {np.flatnonzero(bad)[:8].tolist()}: {got[bad][:4]} vs {exp[bad][:4]}"
        assert self.scratch.tolist() == [0, 0, 0, 0], f"{what}: scratch {self.scratch.tolist()} (signal count or timeout)"
        n = self.desc.n_peer
        assert self.peer_flag.tolist() == [epoch] * n + [0] * (HALO_MAX - n), f"{what}: peer slots {self.peer_flag.tolist()}"
        assert torch.equal(self.my_flag, self.inbox), f"{what}: the rank's own inbox changed"


def _spmv_halo(M, x_ptr, y_ptr, desc, wait, signal):
    L = _L()
    return L.lib().bmsp_spmv_halo(M._h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), C.byref(desc), C.c_uint32(wait), C.c_uint32(signal), _stream())


def _halo_push(y_ptr, rows, desc, signal):
    L = _L()
    return L.lib().bmsp_halo_push(C.c_void_p(y_ptr), C.c_int32(rows), C.byref(desc), C.c_uint32(signal), _stream())


def _check_halo(B, case, ranges):
    """two consecutive epochs of bmsp_spmv_halo over `ranges`, every result and the protocol state checked"""
    M, csr, xs, ref, _ = case
    nr, nc = csr[0], csr[1]
    h = Halo(ranges, (OWN_MARGIN, nc - OWN_MARGIN))
    plain = B.bmSparse_SpMV(M, xs)
    _, ybuf = _buffers(csr, np.zeros(nc, np.float32), torch.float32)
    for epoch in (1, 2):
        ybuf.fill_(SENTINEL); ybuf[PAD:PAD + nr] = float("nan"); h.reset()
        _L().check(_spmv_halo(M, xs.data_ptr(), ybuf[PAD:].data_ptr(), h.desc, epoch, epoch + 1))
        torch.cuda.synchronize()
        _check(ref, ybuf)
        assert torch.equal(ybuf[PAD:PAD + nr], plain), epoch
        h.check(ref, epoch + 1, f"epoch {epoch}")


# ---------------------------------------------------------------------------------------------------------------- fused product
def _exact_case(B, kernel, vd, shape):
    case = _case(B, kernel, vd)
    _check_halo(B, case, _shapes(case[1][0], case[4])[shape])


def _every_case(B, kernels, shapes):
    """_exact_case for every kernel, value dtype and shape; reports every case that fails, by name, not only the first"""
    failed = []
    for kernel in kernels:
        for vd in VDT:
            for shape in shapes:
                try:
                    _exact_case(B, kernel, vd, shape)
                except AssertionError as e:
                    failed.append(f"{kernel}-{vd}-{shape}: {(str(e) or repr(e)).splitlines()[0]}")
    assert not failed, f"{len(failed)} cases fail:\n" + "\n".join(failed)


PUSHING = [s for s in SHAPES if s != "none"]


def test_streaming_kernel_palette(B):
    """the streaming kernel with a palette, fp16 and fp32 values, every push-range shape"""
    _every_case(B, ["stream_palette"], PUSHING)


def test_streaming_kernel_no_palette(B):
    """the streaming kernel without a palette (more than 256 distinct bitmaps), fp16 and fp32 values, every push-range shape"""
    _every_case(B, ["stream_bitmaps"], PUSHING)


@pytest.mark.parametrize("shape", PUSHING)
@pytest.mark.parametrize("vd", list(VDT))
@pytest.mark.parametrize("rt", [32, 16])
def test_per_tile_kernel(B, rt, vd, shape):
    _exact_case(B, f"tile{rt}", vd, shape)


def test_block_parallel(B):
    """the block-parallel path (wait kernel, product, push kernel), fp16 and fp32 values, every push-range shape"""
    _every_case(B, ["block_parallel"], PUSHING)


def test_nothing_pushed_still_signals(B):
    """no push range, on every kernel and value dtype: the row-tiled kernels' tile 0 signals on behalf of a rank that pushes
    nothing, the push kernel of the block-parallel path signals with an empty loop"""
    _every_case(B, list(KERNELS), ["none"])


@pytest.mark.parametrize("shape", SHAPES)
def test_halo_push_alone(B, shape):
    """bmsp_halo_push on its own (the first exchange after x is set): y holds distinct integers, rows % 4 == 1, every range shape
    including no range at all with peers (a rank that only receives still publishes its epoch)"""
    nr = 23997
    y = torch.full((nr + 2 * PAD,), SENTINEL, device="cuda")
    yref = np.arange(1, nr + 1, dtype=np.float64) * np.where(np.arange(nr) % 3 == 1, -1, 1)
    y[PAD:PAD + nr] = torch.from_numpy(yref).float().cuda()
    h = Halo(_shapes(nr, 512)[shape], (0, nr))
    for epoch in (7, 8):
        h.reset()
        _L().check(_halo_push(y[PAD:].data_ptr(), nr, h.desc, epoch))
        torch.cuda.synchronize()
        h.check(yref, epoch, f"epoch {epoch}")


def test_rank_without_rows_still_signals(B):
    """a rank that owns no rows (an empty shard) reads and writes no vector -- its x and y may be null -- but still publishes its
    epoch to the peers that wait for it"""
    M = B.bmSpMatrix.from_csr(0, 16, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    h = Halo([(0, 0)], (0, 16))
    _L().check(_spmv_halo(M, 0, 0, h.desc, 3, 4))
    torch.cuda.synchronize()
    h.check(np.zeros(0), 4)


# ---------------------------------------------------------------------------------------------------------------- rejection
def test_descriptor_rejection(B):
    """malformed descriptors return BMSP_ERR_INVALID from both entry points and touch neither y, the sinks nor the flags;
    misaligned x or y is BMSP_ERR_INVALID, a transposed matrix BMSP_ERR_UNSUPPORTED"""
    L = _L()
    M, csr, xs, ref, T = _case(B, "stream_palette", "v16")
    nr, nc = csr[0], csr[1]
    h = Halo([(0, 100), (T, 2 * T)], (OWN_MARGIN, nc - OWN_MARGIN))
    _, ybuf = _buffers(csr, np.zeros(nc, np.float32), torch.float32)
    y_ptr = ybuf[PAD:].data_ptr()

    def bad(**kw):
        d = L.HaloDesc.from_buffer_copy(h.desc)
        for k, v in kw.items():
            if k in ("push_lo", "push_hi", "push_dst"):
                getattr(d, k)[0] = v
            else:
                setattr(d, k, v)
        return d
    cases = {
        "lo % 4 != 0": bad(push_lo=2),
        "misaligned push_dst": bad(push_dst=h.desc.push_dst[0] + 4),
        "hi > rows": bad(push_lo=nr & ~3, push_hi=nr + 1),
        "lo > hi": bad(push_lo=8, push_hi=4),
        "n_push > 8": bad(n_push=HALO_MAX + 1),
        "n_peer > 8": bad(n_peer=HALO_MAX + 1),
        "peers without scratch": bad(scratch=None),
        "pushes without peers": bad(n_peer=0),
    }
    snap = lambda: (ybuf.clone(), h.sink.clone(), h.peer_flag.clone(), h.my_flag.clone(), h.scratch.clone())
    before = snap()
    for what, d in cases.items():
        assert _spmv_halo(M, xs.data_ptr(), y_ptr, d, 1, 2) == INVALID, what
        assert _halo_push(y_ptr, nr, d, 2) == INVALID, what
    assert _spmv_halo(M, xs.data_ptr() + 4, y_ptr, h.desc, 1, 2) == INVALID, "misaligned x"
    assert _spmv_halo(M, xs.data_ptr(), y_ptr + 4, h.desc, 1, 2) == INVALID, "misaligned y"
    nr_, nc_, rp, ci, v = csr
    Mt = B.bmSpMatrix.from_csr(nr_, nc_, rp, ci, v, transpose=True)
    assert _spmv_halo(Mt, xs.data_ptr(), y_ptr, h.desc, 1, 2) == UNSUPPORTED, "transposed"
    torch.cuda.synchronize()
    for a, b, what in zip(before, snap(), ("y", "sink", "peer slots", "inbox", "scratch")):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"a rejected call changed {what}"


# ---------------------------------------------------------------------------------------------------------------- the wait orders x
H_COLS = 100             # halo columns at the high end of x
WAIT_EPOCH = 5


def _halo_reader(nr, kernel, seed=3):
    """nr rows over nr + H_COLS columns: a band on the own columns, and the last rows also read one halo column each.  Block-parallel:
    three random own columns per row instead of the band (one or two cells per block)."""
    rng = np.random.default_rng(seed)
    i = np.arange(nr)
    if kernel == "block_parallel":
        rows = np.repeat(i, 3); cols = np.concatenate([np.sort(rng.choice(nr, 3, replace=False)) for _ in range(nr)])
    else:
        rows = np.repeat(i, 4); cols = (rows + np.tile([0, 1, 2, 9], nr)).clip(max=nr - 1)
        keep = np.ones(rows.size, bool); keep[1:] = (rows[1:] != rows[:-1]) | (cols[1:] != cols[:-1])
        rows, cols = rows[keep], cols[keep]
    tail = i[-3 * H_COLS:]
    rows = np.concatenate([rows, tail]); cols = np.concatenate([cols, nr + tail % H_COLS])
    from tests.test_gpu_spmv_exact import _csr
    return (nr, nr + H_COLS) + _csr(nr, rows, cols)


@pytest.mark.parametrize("kernel", ["stream_palette", "per_tile", "block_parallel"])
def test_wait_orders_x(B, monkeypatch, kernel):
    """The tiles that read halo columns wait for the peer's epoch before they touch x.  One peer's slot holds wait_epoch - 1 and
    the halo columns of x hold NaN; the product is launched and must still be running 50 ms later (tiles are waiting).  Then a
    copy engine, on a second stream, writes the halo values from pinned host memory and after them the epoch.  y must be exact and
    no wait may have timed out.  The halo columns are at the high end of x only, and the tiles that read them push nothing (the
    one push range is rows [0, 8)): a pushing tile waits anyway, and so does the signalling tile of a rank that pushes nothing.
    Per-tile kernel: own_col_hi is no multiple of 32, so a 32-column x line straddles the boundary (the L1 fence path); the
    streaming kernel takes the acquire-load path, block-parallel the wait kernel.  Nothing synchronises between the launch and
    the copies; if they could not run the kernel would give up after its 4 s timeout and the test fail on scratch[1]."""
    nr = 40000 + 3
    pat = _halo_reader(nr, kernel)
    if kernel == "per_tile":
        monkeypatch.setenv("BMSP_SPMV_KERNEL", "1")
    M, csr = _matrix(B, pat, torch.float16, seed=5)
    info = plan_info(M)
    monkeypatch.delenv("BMSP_SPMV_KERNEL", raising=False)
    if kernel == "stream_palette":
        _streaming(info, palette=True)
    elif kernel == "per_tile":
        assert info.path == 0 and info.kernel == 1
    else:
        assert info.path == 1
    nc = csr[1]
    own_hi = nr
    assert kernel != "per_tile" or own_hi % 32 != 0
    x = _x(nc, torch.float16, np.random.default_rng(9))
    ref = _reference(csr, x)
    xs, ybuf = _buffers(csr, x, torch.float32)
    halo_host = torch.from_numpy(x[own_hi:]).pin_memory()
    epoch_host = torch.tensor([WAIT_EPOCH], dtype=torch.int32).pin_memory()
    h = Halo([(0, 8)], (0, own_hi))
    h.my_flag[0] = WAIT_EPOCH - 1; h.my_flag[1] = WAIT_EPOCH
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    # one product on s1 with the epoch already there: whatever the library builds on first use of a stream exists before the timed
    # launch, so nothing in that launch synchronises with the device
    h.my_flag[0] = WAIT_EPOCH
    with torch.cuda.stream(s1):
        _L().check(_spmv_halo(M, xs.data_ptr(), ybuf[PAD:].data_ptr(), h.desc, WAIT_EPOCH, WAIT_EPOCH + 1))
    torch.cuda.synchronize()
    h.my_flag[0] = WAIT_EPOCH - 1; h.peer_flag.zero_()
    xs[own_hi:] = float("nan"); ybuf[PAD:PAD + nr] = float("nan")
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        _L().check(_spmv_halo(M, xs.data_ptr(), ybuf[PAD:].data_ptr(), h.desc, WAIT_EPOCH, WAIT_EPOCH + 1))
    time.sleep(0.05)
    running = not s1.query()
    with torch.cuda.stream(s2):
        xs[own_hi:].copy_(halo_host, non_blocking=True)
        h.my_flag[:1].copy_(epoch_host, non_blocking=True)
    torch.cuda.synchronize()
    assert running, "the product finished while a peer's epoch was missing"
    assert int(h.scratch[1]) == 0, "a wait timed out: the epoch or the halo never arrived"
    _check(ref, ybuf)
    h.inbox = h.my_flag.clone()
    h.check(ref, WAIT_EPOCH + 1)
