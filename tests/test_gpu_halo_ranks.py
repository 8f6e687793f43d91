"""N ranks of the peer-memory SpMV emulated in one process on one GPU: the real range plan and descriptor arithmetic of dist.py
(halo_ranges, halo_peers, csr_row_slice, halo_descriptor) and the real kernels, with data flowing between the ranks.

Every fake rank has one device allocation laid out like PeerHalo's region -- an inbox of epoch slots, then three x buffers -- with
sentinel gaps between them (behind the inbox and behind every buffer); the x buffers start out NaN.  Its local matrix has columns
rebased to its extended range.  The protocol is PeerHalo's, on one stream: bmsp_halo_push of every rank's own slice of x[cur] with
epoch e, then K steps, each running every rank in turn: bmsp_spmv_halo(local, x[cur], own(x[nxt]), desc[nxt], e, e + 1).  Because
the ranks run in order on one stream, every wait is satisfied when its kernel starts: nothing spins.

The matrices hold integers and x starts as integers, and the test asserts sum_j |a_ij x_j| < 2^24 for every row at every step, so
the fp32 products are exact.  After the first push and after every step each rank's whole region is compared bit for bit with a model
of what the protocol writes: its own slice equals the float64 product of the global matrix with the previous global x, every slice it
received equals those rows of the new global x (checked before the next step consumes it), the inbox slots of its peers hold the
epoch, and everything else is still NaN or sentinel.  scratch must stay [0, 0]."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from tests.test_gpu_spmv_exact import plan_info

pytestmark = pytest.mark.gpu

NBUF = 3
INBOX = 1024                 # bytes of epoch slots
XOFF = INBOX + 256           # x buffer 0 starts behind a sentinel gap
GAP = 64                     # sentinel floats at least behind every x buffer
SENTINEL = -12345.5


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _L():
    from bmsparse_spgemm_spmv_b200 import _lib as L
    return L


# ---------------------------------------------------------------------------------------------------------------- matrices
def _integers(csr, mag, seed):
    """the pattern of csr with nonzero integer values in [-mag, mag]"""
    n, nc, rp, ci, _ = csr
    rng = np.random.default_rng(seed)
    v = (np.where(rng.random(ci.size) < 0.5, -1.0, 1.0) * rng.integers(1, mag + 1, ci.size)).astype(np.float32)
    return n, nc, np.asarray(rp, np.int32), np.asarray(ci, np.int32), v


def _weight_bounds(n, rp, world):
    """the split dist_worker uses: block rows balanced by stored values, bounds multiples of 8"""
    from bmsparse_spgemm_spmv_b200.dist import split_by_weight
    w = np.add.reduceat(np.diff(rp).astype(np.float64), np.arange(0, n, 8)) + 1.0
    b = split_by_weight(w, world) * 8
    b[-1] = n
    return b


def _bidiagonal(n):
    """the lower-bidiagonal matrix of dist_worker.one_directional: row i reads columns i - 1 and i"""
    i = np.arange(n, dtype=np.int64)
    cols = np.stack([i - 1, i], axis=1); valid = np.stack([i > 0, np.ones(n, bool)], axis=1)
    rp = np.zeros(n + 1, np.int64); np.cumsum(valid.sum(1), out=rp[1:])
    ci = cols[valid]
    return n, n, rp.astype(np.int32), ci.astype(np.int32), np.ones(ci.size, np.float32)


# ---------------------------------------------------------------------------------------------------------------- fake ranks
class Rank:
    def __init__(self, B, r, bounds, csr, vdt):
        from bmsparse_spgemm_spmv_b200.dist import csr_row_slice
        n, _, rp, ci, v = csr
        self.r = r
        self.own_lo, self.own_hi = int(bounds[r]), int(bounds[r + 1])
        lrp, lci, lv = csr_row_slice(rp, ci, v, self.own_lo, self.own_hi)
        # the extended range, as ShardedSpMV computes it
        lo = min(self.own_lo, int(lci.min()) if len(lci) else self.own_lo)
        hi = max(self.own_hi, int(lci.max()) + 1 if len(lci) else self.own_hi)
        self.ext_lo, self.ext_hi = (lo // 8) * 8, min(((hi + 7) // 8) * 8, n)
        self.n_ext = self.ext_hi - self.ext_lo
        self.rows = self.own_hi - self.own_lo
        self.stride = ((self.n_ext + GAP) * 4 + 255) // 256 * 256          # bytes, a multiple of 256 as in PeerHalo
        nf = (XOFF + NBUF * self.stride) // 4
        self.model = np.full(nf, SENTINEL, np.float32)
        self.model.view(np.uint32)[:INBOX // 4] = 0
        for b in range(NBUF):
            self.model[self._x0(b):self._x0(b) + self.n_ext] = np.nan
        self.region = torch.from_numpy(self.model.copy()).cuda()
        self.base = self.region.data_ptr()
        self.scratch = torch.zeros(4, dtype=torch.int32, device="cuda")
        self.M = B.bmSpMatrix.from_csr(self.rows, self.n_ext, lrp, (lci.astype(np.int64) - self.ext_lo).astype(np.int32), lv, dtype=vdt)

    def _x0(self, b):
        return (XOFF + b * self.stride) // 4

    def own_ptr(self, b):
        """the own slice of x buffer b; a rank without rows has empty x buffers, whose tensors have no address"""
        return self.base + 4 * (self._x0(b) + self.own_lo - self.ext_lo) if self.rows else 0

    def x_ptr(self, b):
        return self.base + 4 * self._x0(b) if self.rows else 0

    def plan(self, ranks, bounds):
        from bmsparse_spgemm_spmv_b200.dist import halo_descriptor, halo_peers, halo_ranges
        self.recv, self.send = halo_ranges(self.r, bounds, [(q.ext_lo, q.ext_hi) for q in ranks])
        self.peers = halo_peers(self.recv, self.send, len(ranks))
        self.desc = [halo_descriptor(b, self.r, self.send, self.peers, self.own_lo, self.own_hi, self.ext_lo, self.base,
                                     {p: ranks[p].base for p in self.peers}, {p: (ranks[p].stride, ranks[p].ext_lo) for p in self.peers},
                                     self.scratch.data_ptr(), XOFF) for b in range(NBUF)]

    def model_x(self, b, a, e, values):
        """the model: global rows [a, e) of x buffer b hold values"""
        s = self._x0(b) + a - self.ext_lo
        self.model[s:s + e - a] = values


def _publish(ranks, b, xg, epoch):
    """the model after every rank pushed rows of xg into buffer b and signalled epoch; its own slice holds its rows too"""
    for q in ranks:
        q.model_x(b, q.own_lo, q.own_hi, xg[q.own_lo:q.own_hi])
        for p, a, e in q.send:
            ranks[p].model_x(b, a, e, xg[a:e])
        for p in q.peers:
            ranks[p].model.view(np.uint32)[q.r] = epoch % (1 << 32)


def _check(ranks, what):
    torch.cuda.synchronize()
    for q in ranks:
        got = q.region.cpu().numpy().view(np.uint32)
        exp = q.model.view(np.uint32)
        bad = np.flatnonzero(got != exp)
        assert bad.size == 0, (f"{what}: rank {q.r}: {bad.size} words differ, first at float {bad[:6].tolist()} "
                               f"(x buffers at {[q._x0(b) for b in range(NBUF)]}): {got[bad[:4]].view(np.float32)} vs "
                               f"{exp[bad[:4]].view(np.float32)}")
        assert q.scratch.tolist() == [0, 0, 0, 0], f"{what}: rank {q.r}: scratch {q.scratch.tolist()}"


def _run(B, csr, bounds, vdt, steps, epoch0=1, x_mag=3, plans=None):
    L = _L()
    n = csr[0]
    S = sp.csr_matrix((csr[4].astype(np.float64), csr[3], csr[2]), shape=(n, csr[1]))
    world = len(bounds) - 1
    ranks = [Rank(B, r, bounds, csr, vdt) for r in range(world)]
    for q in ranks:
        q.plan(ranks, bounds)
        if plans and q.rows:
            plans(plan_info(q.M))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(world)
    xg = (np.where(rng.random(n) < 0.5, -1.0, 1.0) * rng.integers(1, x_mag + 1, n)).astype(np.float32)
    # the inbox slots hold epoch0 - 1 before the first push (a fresh region holds 0 and the first push signals 1)
    for q in ranks:
        for p in q.peers:
            q.model.view(np.uint32)[p] = (epoch0 - 1) % (1 << 32)
            q.region.view(torch.int32)[p] = int(np.uint32((epoch0 - 1) % (1 << 32)).view(np.int32))
    cur, e = 0, epoch0
    for q in ranks:                                                                       # set_x + first_push
        if q.rows:
            q.region[q._x0(cur) + q.own_lo - q.ext_lo:q._x0(cur) + q.own_hi - q.ext_lo] = torch.from_numpy(xg[q.own_lo:q.own_hi]).cuda()
        L.check(L.lib().bmsp_halo_push(C.c_void_p(q.own_ptr(cur)), q.rows, C.byref(q.desc[cur]), C.c_uint32(e % (1 << 32)), st))
    _publish(ranks, cur, xg, e)
    _check(ranks, "first push")
    for k in range(steps):
        nxt = (cur + 1) % NBUF
        for q in ranks:
            L.check(L.lib().bmsp_spmv_halo(q.M._h, C.c_void_p(q.x_ptr(cur)), C.c_void_p(q.own_ptr(nxt)), C.byref(q.desc[nxt]),
                                           C.c_uint32(e % (1 << 32)), C.c_uint32((e + 1) % (1 << 32)), st))
        bound = float((abs(S) @ np.abs(xg.astype(np.float64))).max())
        assert bound < 2 ** 24, f"step {k}: the exactness bound fails ({bound})"
        xg = (S @ xg.astype(np.float64)).astype(np.float32)
        e += 1
        _publish(ranks, nxt, xg, e)
        _check(ranks, f"step {k}")
        cur = nxt
    return ranks


def _streaming(i):
    assert i.path == 0 and i.kernel == 0


def _per_tile(i):
    assert i.path == 0 and i.kernel == 1


def _block_parallel(i):
    assert i.path == 1


def _row_tiled(i):
    assert i.path == 0


# ---------------------------------------------------------------------------------------------------------------- cases
@pytest.mark.parametrize("world", [2, 3, 5])
def test_poisson_slabs(B, world):
    """5-point Poisson slabs: neighbours only, streaming kernel; the bounds are no multiples of the 512-row tile"""
    csr = _integers(B.generators.poisson5pt(200, 30 * world), 1, seed=world)
    bounds = _weight_bounds(csr[0], csr[2], world)
    assert any(b % 512 for b in bounds[1:-1])
    ranks = _run(B, csr, bounds, torch.float16, 3, plans=_streaming)
    assert all(len(q.peers) == (1 if q.r in (0, world - 1) else 2) for q in ranks)


def test_poisson_slabs_fp32(B):
    csr = _integers(B.generators.poisson5pt(200, 90), 2, seed=4)
    _run(B, csr, _weight_bounds(csr[0], csr[2], 3), torch.float32, 3, plans=_streaming)


@pytest.mark.parametrize("vdt", [torch.float16, torch.float32], ids=["v16", "v32"])
def test_block_clustered(B, vdt):
    """a block-banded matrix of heavy rows: the per-tile kernel"""
    csr = _integers(B.generators.block_clustered(3000), 1, seed=5)
    _run(B, csr, _weight_bounds(csr[0], csr[2], 3), vdt, 3, plans=_per_tile)


@pytest.mark.parametrize("world", [4, 9])
def test_scattered_all_gather(B, world):
    """uniformly scattered columns: every rank needs all of x (block-parallel path).  At 9 ranks: eight peers and eight push
    ranges of the same rows, the descriptor's maximum"""
    csr = _integers(B.generators.uniform_random(20000, 16), 1, seed=6)
    ranks = _run(B, csr, _weight_bounds(csr[0], csr[2], world), torch.float16, 3, x_mag=2, plans=_block_parallel)
    for q in ranks:
        assert len(q.peers) == world - 1 and len(q.send) == world - 1
        assert all((a, e) == (q.own_lo, q.own_hi) for _, a, e in q.send)


def test_scattered_fp32(B):
    csr = _integers(B.generators.uniform_random(20000, 16), 1, seed=7)
    _run(B, csr, _weight_bounds(csr[0], csr[2], 4), torch.float32, 3, x_mag=2, plans=_block_parallel)


def test_ten_ranks_refused(B):
    """ten ranks of a scattered matrix need nine peers each: more than one descriptor holds, refused as PeerHalo.create refuses it"""
    from bmsparse_spgemm_spmv_b200.dist import halo_peers, halo_ranges
    n, _, rp, ci, _ = B.generators.uniform_random(20000, 16)
    bounds = _weight_bounds(n, rp, 10)
    ranges = [(0, n)] * 10
    for r in range(10):
        recv, send = halo_ranges(r, bounds, ranges)
        with pytest.raises(RuntimeError, match="too many peers"):
            halo_peers(recv, send, 10)


def test_one_directional(B):
    """lower bidiagonal: rank r pushes its last row to rank r + 1 and reads nothing remote (its pushing tile still waits); the
    last rank pushes nothing (n_push == 0) and still signals the rank it reads from"""
    csr = _integers(_bidiagonal(4 * 4096), 1, seed=8)
    bounds = np.arange(5, dtype=np.int64) * 4096
    ranks = _run(B, csr, bounds, torch.float16, 4, plans=_row_tiled)
    assert ranks[-1].desc[0].n_push == 0 and ranks[-1].desc[0].n_peer == 1
    # the reader's extended range starts at a multiple of 8: the last 8 rows of every other rank go to the next one
    assert all(q.send == [(q.r + 1, q.own_hi - 8, q.own_hi)] for q in ranks[:-1])


def test_empty_shard(B):
    """a split with a rank of no rows: its extended range is empty (no peers, null x and y), the others exchange around it"""
    csr = _integers(B.generators.poisson5pt(200, 60), 1, seed=9)
    b = (csr[0] // 2) // 8 * 8
    ranks = _run(B, csr, np.array([0, b, b, csr[0]], np.int64), torch.float16, 3)
    assert ranks[1].rows == 0 and ranks[1].n_ext == 0 and ranks[1].peers == []
    assert ranks[0].peers == [2] and ranks[2].peers == [0]


def test_epochs_cross_2_32(B):
    """the epoch counter wraps: the first push signals 2^32 - 4, eight steps later the slots hold 4"""
    csr = _integers(B.generators.poisson5pt(200, 60), 1, seed=10)
    _run(B, csr, _weight_bounds(csr[0], csr[2], 2), torch.float16, 8, epoch0=(1 << 32) - 4, x_mag=1)
