"""Block-row sharding over one process per GPU (torch.distributed: NCCL on GPUs, gloo in the CPU tests).

The reference is single-GPU (SURVEY.md section 2: no collectives anywhere); this is the multi-GPU layer the
north star adds.  Both operators shard by block rows and need no reduction:

  SpMV    rank r owns a contiguous range of block rows and the matching slice of x / y.  Before each
          product it fetches only the slices of x its block columns touch ("range halo": for a banded
          matrix two neighbours, for a scattered one everybody -- then it degenerates to an all-gather).
          y is written straight into the owner's slice of the next x, so repeated products rotate
          through two (NCCL) or three (peer memory) buffers with no copy.
  SpGEMM  rank r multiplies its block rows of A by a replicated B^t (bmSparse_mult(..., brow_range)); the
          concatenation of the per-rank C arrays is bit-identical to the single-GPU product.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def split_by_weight(weights: np.ndarray, nparts: int, align: int = 1) -> np.ndarray:
    """Contiguous split of len(weights) items into nparts ranges of near-equal total weight.
    Returns int64 bounds[nparts+1]; interior bounds are multiples of `align`."""
    n = len(weights)
    prefix = np.concatenate([[0], np.cumsum(np.asarray(weights, np.float64))])
    bounds = np.zeros(nparts + 1, np.int64)
    bounds[nparts] = n
    for p in range(1, nparts):
        b = int(np.searchsorted(prefix, prefix[-1] * p / nparts, side="left"))
        b = (b // align) * align
        bounds[p] = min(max(b, bounds[p - 1]), n)
    return bounds


def deal_chunks(nchunks: int, world: int, rank: int) -> list:
    """Which of `nchunks` work chunks (ordered from the heaviest rows to the lightest) rank `rank` of `world` takes: rounds of
    `world` chunks, every other round in reverse rank order, so that no rank is handed the heavier chunk of every round (a plain
    cyclic deal does that to rank 0).  Every chunk goes to exactly one rank; counts differ by at most one."""
    mine = []
    for rnd in range((nchunks + world - 1) // world):
        c = rnd * world + (rank if rnd % 2 == 0 else world - 1 - rank)
        if c < nchunks:
            mine.append(c)
    return mine


def csr_row_slice(rp, ci, v, r0, r1):
    """rows [r0, r1) of a CSR triple, row_ptr rebased to 0 (columns untouched)."""
    s, e = int(rp[r0]), int(rp[r1])
    return (np.asarray(rp[r0:r1 + 1]) - s).astype(np.int32), ci[s:e], v[s:e]


def halo_ranges(rank, bounds, ranges):
    """The range halo of one rank: (recv, send), lists of (peer, a, b) global rows [a, b).  What I receive from peer p: the
    overlap of my extended range with p's owned rows; what I send to p: the overlap of p's extended range with my owned rows.
    bounds: the global row split (len world + 1); ranges[p] = (ext_lo, ext_hi) of every rank, mine included."""
    own_lo, own_hi = int(bounds[rank]), int(bounds[rank + 1])
    ext_lo, ext_hi = ranges[rank]
    recv, send = [], []
    for p in range(len(ranges)):
        if p == rank:
            continue
        plo, phi = int(bounds[p]), int(bounds[p + 1])
        a, b = max(ext_lo, plo), min(ext_hi, phi)
        if a < b:
            recv.append((p, a, b))
        a, b = max(ranges[p][0], own_lo), min(ranges[p][1], own_hi)
        if a < b:
            send.append((p, a, b))
    return recv, send


class ShardedSpMV:
    """y = A x with A sharded by rows and x sharded the same way (square matrices).

    Parameters
    ----------
    row_bounds : global row split (len world+1), interior bounds multiples of 8
    local_csr  : (row_ptr, col_idx, vals) of this rank's rows, GLOBAL column indices, ascending per row
    spmv_fn    : callable(x_ext, y_out) computing the local product; default builds a bmSpMatrix on the
                 current CUDA device and calls bmSparse_SpMV (the CPU tests inject the oracle here)
    """

    def __init__(self, row_bounds, local_csr, n_cols, group=None, device=None, spmv_fn=None, build_fn=None, halo="auto"):
        self.group = group
        self.p2p = None                      # PeerHalo when the exchange runs over peer memory inside the SpMV kernel
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.bounds = np.asarray(row_bounds, np.int64)
        self.device = device if device is not None else torch.device("cpu")
        rp, ci, v = local_csr
        self.own_lo, self.own_hi = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        lo = min(self.own_lo, int(ci.min()) if len(ci) else self.own_lo)
        hi = max(self.own_hi, int(ci.max()) + 1 if len(ci) else self.own_hi)
        self.ext_lo, self.ext_hi = (lo // 8) * 8, min(((hi + 7) // 8) * 8, n_cols)
        # everybody learns everybody's extended range
        mine = torch.tensor([self.ext_lo, self.ext_hi], dtype=torch.int64, device=self.device)
        allr = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(allr, mine, group=group)
        ranges = [tuple(int(t) for t in a.cpu()) for a in allr]
        self.recv, self.send = halo_ranges(self.rank, self.bounds, ranges)
        n_ext = self.ext_hi - self.ext_lo
        self.cur = 0
        self.x = None
        if halo != "nccl" and spmv_fn is None and self.device.type == "cuda" and self.world > 1:
            self.p2p = PeerHalo.create(self, ranges, n_ext)          # collective; None when any rank cannot map its peers
            if self.p2p is None and halo == "p2p":
                raise RuntimeError("peer-memory halo exchange requested but not available")
        if self.p2p is not None:
            self.x = self.p2p.x
        else:
            self.x = [torch.zeros(n_ext, dtype=torch.float32, device=self.device) for _ in range(2)]
        self.halo_bytes = sum(b - a for _, a, b in self.recv) * 4
        local_ci = (np.asarray(ci, np.int64) - self.ext_lo).astype(np.int32)
        n_rows = self.own_hi - self.own_lo
        if spmv_fn is not None:
            self._spmv = spmv_fn
            self.local = build_fn(n_rows, n_ext, rp, local_ci, v) if build_fn else None
        else:
            from .matrix import bmSpMatrix
            from .ops import bmSparse_SpMV
            self.local = bmSpMatrix.from_csr(n_rows, n_ext, rp, local_ci, v)
            self._spmv = lambda x_ext, y_out: bmSparse_SpMV(self.local, x_ext, y_out)

    def own_slice(self, buf):
        return buf[self.own_lo - self.ext_lo: self.own_hi - self.ext_lo]

    def set_x(self, x_own: torch.Tensor):
        """collective: every rank sets its slice of x (then, in peer-memory mode, pushes it to the peers that need it)"""
        self.own_slice(self.x[self.cur]).copy_(x_own)
        if self.p2p is not None:
            self.p2p.first_push(self)

    def exchange(self):
        """fetch the halo slices of the current x from their owners (NCCL send/recv over NVLink)."""
        buf = self.x[self.cur]
        ops = []
        for p, a, b in self.send:
            ops.append(dist.P2POp(dist.isend, buf[a - self.ext_lo: b - self.ext_lo], p, group=self.group))
        for p, a, b in self.recv:
            ops.append(dist.P2POp(dist.irecv, buf[a - self.ext_lo: b - self.ext_lo], p, group=self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    def step(self):
        """one product: halo exchange of x, then y = A_local x_ext written into the next x's own slice.
        Peer-memory mode: one kernel does all of it (wait for the peers' epoch, product, P2P stores of the boundary rows
        into the peers' next x, publish the next epoch)."""
        nxt = (self.cur + 1) % len(self.x)
        if self.p2p is not None:
            self.p2p.step(self, nxt)
        else:
            self.exchange()
            self._spmv(self.x[self.cur], self.own_slice(self.x[nxt]))
        self.cur = nxt

    def check(self):
        """raises if a peer-memory wait timed out (a peer died); no-op in NCCL mode"""
        if self.p2p is not None:
            self.p2p.check()

    def close(self):
        if self.p2p is not None:
            self.p2p.close(self)
            self.p2p = None

    def y_own(self):
        return self.own_slice(self.x[self.cur])


def balanced_block_row_bounds(A, group=None, iters: int = 5, reps: int = 20, push_gbps: float = 750.0, tol: float = 1.015):
    """Block-row split of a scattered matrix (block-parallel SpMV path: every rank needs all of x) by MEASURED cost.

    The model split (bmsp_partition_block_rows: blocks + block rows + the bytes a rank pushes to its peers) is only a start: on a
    power-law matrix the cost of a block depends on where its row and column sit (hub rows gather x from everywhere, tail rows from
    the few hub columns that stay in L1), +-15 % between shards with the same counts.  Every rank holds the whole matrix here, so it
    slices ITS shard, times the local product, adds the time its pushes take (rows x 4 bytes x (N - 1) peers at the egress rate), the
    ranks exchange the totals, every block row's weight in a shard is scaled by that shard's total / mean, and the split is redone.
    Collective; returns int64 bounds[N + 1] in block rows, identical on every rank.  Setup cost: `iters` x (slice + plan + reps products).
    """
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = torch.device("cuda", torch.cuda.current_device())
    nb = np.diff(A.block_row_ptr.cpu().numpy().astype(np.int64))
    nbr = len(nb)
    w = (14.0 * nb + 330.0 + 76.0 * (world - 1))                     # the C partitioner's model for this path (dist.cu)
    x = torch.ones(A.num_cols, dtype=torch.float32, device=dev)
    bounds = split_by_weight(w, world)
    best, best_max = bounds, float("inf")
    for it in range(iters):
        b0, b1 = int(bounds[rank]), int(bounds[rank + 1])
        t_local = 0.0
        if b1 > b0:
            S = A.slice_block_rows(b0, b1, rebase=True)
            y = torch.empty(S.num_rows, dtype=torch.float32, device=dev)
            from .ops import bmSparse_SpMV
            for _ in range(3):
                bmSparse_SpMV(S, x, y)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                bmSparse_SpMV(S, x, y)
            e1.record(); e1.synchronize()
            t_local = e0.elapsed_time(e1) / reps * 1e3                 # us
            del S, y
        push = (b1 - b0) * 32.0 * (world - 1) / (push_gbps * 1e3)       # us: 32 bytes per block row and peer
        mine = torch.tensor([t_local + push], dtype=torch.float64, device=dev)
        allt = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allt, mine, group=group)
        tot = np.array([float(t.item()) for t in allt])
        mean = float(tot.mean())
        if float(tot.max()) < best_max:
            best, best_max = bounds, float(tot.max())                  # the split returned is always one that was measured
        if mean <= 0 or float(tot.max()) <= tol * mean or it == iters - 1:
            break
        for p in range(world):
            w[int(bounds[p]):int(bounds[p + 1])] *= max(0.5, min(2.0, tot[p] / mean))
        bounds = split_by_weight(w, world)
    return best


def halo_descriptor(buf, rank, send, peers, own_lo, own_hi, ext_lo, my_base, peer_base, peer_layout, scratch_ptr, inbox=1024):
    """bmsp_halo_desc of x buffer `buf` for one rank (pure address arithmetic: the CPU tests check it without a GPU).
    send: [(peer, a, e)] global row ranges of mine a peer needs; peers: everybody I exchange epochs with (both directions);
    peer_base[p]: where p's region is mapped here; peer_layout[p] = (buffer stride in bytes, p's ext_lo)."""
    from . import _lib as L
    d = L.HaloDesc()
    d.n_push = len(send)
    for i, (p, a, e) in enumerate(send):
        stride, p_ext_lo = peer_layout[p]
        d.push_lo[i] = a - own_lo; d.push_hi[i] = e - own_lo
        d.push_dst[i] = peer_base[p] + inbox + buf * stride + (a - p_ext_lo) * 4
    d.n_peer = len(peers)
    for i, p in enumerate(peers):
        d.peer_flag[i] = peer_base[p] + 4 * rank           # my slot in p's inbox
        d.my_flag[i] = my_base + 4 * p                     # p's slot in mine
    d.scratch = scratch_ptr
    d.own_col_lo = own_lo - ext_lo; d.own_col_hi = own_hi - ext_lo
    return d


def halo_peers(recv, send, world, inbox=1024):
    """the ranks one rank exchanges epochs with (both directions, sorted); RuntimeError when one halo descriptor cannot hold them"""
    from . import _lib as L
    peers = sorted({p for p, _, _ in send} | {p for p, _, _ in recv})
    if len(peers) > L.HALO_MAX or len(send) > L.HALO_MAX or world > inbox // 4:
        raise RuntimeError("too many peers for one halo descriptor")
    return peers


class PeerHalo:
    """Three rotating peer-mapped x buffers + epoch inbox of one rank, and the bmsp_halo_desc of each buffer.

    Region layout (one cudaMalloc per rank, exported as a CUDA IPC handle and opened by the ranks that talk to it):
        [0, 1024)            inbox: uint32 epoch slot per source rank
        [1024, 1024+S)       x buffer 0 (n_ext fp32, S = n_ext*4 rounded up to 256)
        [1024+S, 1024+2S)    x buffer 1
        [1024+2S, 1024+3S)   x buffer 2
    Three buffers, not two: the kernel publishes its epoch as soon as its boundary tiles are done (mid-kernel, see the tile
    rotation in spmv.cu), so a peer may start writing the next-but-one x while this rank's kernel still reads the current
    one; with three buffers the buffer being overwritten is always one whose last reader finished a whole launch earlier.
    """
    INBOX = 1024
    NBUF = 3

    @classmethod
    def create(cls, sh, ranges, n_ext):
        import ctypes as C
        from . import _lib as L
        from .matrix import _alias
        self = cls()
        self.epoch = 0
        self._args = {}
        self.opened = {}
        self.base = None
        ok = True
        try:
            peers = halo_peers(sh.recv, sh.send, sh.world, cls.INBOX)
            stride = (n_ext * 4 + 255) // 256 * 256
            base = C.c_void_p(); handle = (C.c_ubyte * 64)()
            L.check(L.lib().bmsp_peer_alloc(C.c_int64(cls.INBOX + cls.NBUF * stride), C.byref(base), handle))
            self.base, self.stride = base.value, stride
        except Exception as e:  # noqa: BLE001 -- every rank must reach the all_gather below
            ok, handle, stride, peers = False, None, 0, []
            self.err = e
        info = [None] * sh.world
        dist.all_gather_object(info, {"ok": ok, "handle": bytes(handle) if ok else b"", "stride": stride, "ext_lo": sh.ext_lo}, group=sh.group)
        if ok and all(i["ok"] for i in info):
            try:
                for p in peers:
                    ptr = C.c_void_p()
                    L.check(L.lib().bmsp_peer_open((C.c_ubyte * 64).from_buffer_copy(info[p]["handle"]), C.byref(ptr)))
                    self.opened[p] = ptr.value
            except Exception as e:  # noqa: BLE001
                ok = False
                self.err = e
        flag = torch.tensor([1 if ok and all(i["ok"] for i in info) else 0], device=sh.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=sh.group)
        if int(flag.item()) == 0:
            self._release()
            return None
        self.x = [_alias(self.base + cls.INBOX + b * stride, n_ext, "<f4", torch.float32, self) for b in range(cls.NBUF)]
        self.scratch = torch.zeros(4, dtype=torch.int32, device=sh.device)
        self.desc = [halo_descriptor(b, sh.rank, sh.send, peers, sh.own_lo, sh.own_hi, sh.ext_lo, self.base, self.opened,
                                     {p: (info[p]["stride"], info[p]["ext_lo"]) for p in peers}, self.scratch.data_ptr(), cls.INBOX)
                     for b in range(cls.NBUF)]
        return self

    def first_push(self, sh):
        import ctypes as C
        from . import _lib as L
        from .matrix import _stream_ptr
        torch.cuda.synchronize(); dist.barrier(group=sh.group)        # nobody still reads the buffer we are about to fill
        self.epoch += 1
        own = sh.own_slice(self.x[sh.cur])
        L.check(L.lib().bmsp_halo_push(C.c_void_p(own.data_ptr()), own.numel(), C.byref(self.desc[sh.cur]), C.c_uint32(self.epoch), _stream_ptr()))

    def step(self, sh, nxt):
        """one fused product.  The call's arguments only depend on which of the three buffers is current: they are built once per
        buffer (a 68 us kernel leaves no room for ~40 us of per-step Python: tensor slicing, data_ptr(), byref)."""
        args = self._args.get(sh.cur)
        if args is None:
            import ctypes as C
            from . import _lib as L
            from .matrix import _stream_ptr
            args = (L.lib().bmsp_spmv_halo, sh.local._h, C.c_void_p(self.x[sh.cur].data_ptr()), C.c_void_p(sh.own_slice(self.x[nxt]).data_ptr()),
                    C.byref(self.desc[nxt]), _stream_ptr(), L.check)
            self._args[sh.cur] = args
        fn, h, xp, yp, dref, st, check = args
        check(fn(h, xp, yp, dref, self.epoch, self.epoch + 1, st))
        self.epoch += 1

    def check(self):
        import ctypes as C
        from . import _lib as L
        from .matrix import _stream_ptr
        t = C.c_int32()
        L.check(L.lib().bmsp_halo_status(C.byref(self.desc[0]), _stream_ptr(), C.byref(t)))
        if t.value:
            raise RuntimeError("peer-memory halo exchange: a wait timed out (peer lost)")

    def _release(self):
        from . import _lib as L
        import ctypes as C
        for ptr in self.opened.values():
            L.lib().bmsp_peer_close(C.c_void_p(ptr))
        self.opened = {}
        if self.base:
            L.lib().bmsp_peer_free(C.c_void_p(self.base))
            self.base = None

    def close(self, sh):
        torch.cuda.synchronize(); dist.barrier(group=sh.group)        # no peer still writes into my region
        self.x = None
        self._release()


def broadcast_matrix(M, src: int = 0, group=None):
    """Replicate a bmSpMatrix (e.g. B^t for SpGEMM) from rank `src` to every rank: four array broadcasts."""
    from .matrix import bmSpMatrix
    rank = dist.get_rank(group)
    dev = torch.device("cuda", torch.cuda.current_device())
    if rank == src:
        v = M._view()
        hdr = torch.tensor([v.num_rows, v.num_cols, v.block_num, v.nnz, v.offsets_len, v.dtype, v.transposed], dtype=torch.int64, device=dev)
    else:
        hdr = torch.zeros(7, dtype=torch.int64, device=dev)
    dist.broadcast(hdr, src, group=group)
    nr, nc, nblk, nnz, noff, dt, tr = (int(t) for t in hdr.cpu())
    vt = torch.float16 if dt == 0 else torch.float32
    if rank == src:
        arrs = [M.keys.clone(), M.bmps.clone(), M.offsets.clone(), M.values.clone()]
    else:
        arrs = [torch.empty(nblk, dtype=torch.int64, device=dev), torch.empty(nblk, dtype=torch.int64, device=dev),
                torch.empty(noff, dtype=torch.int64, device=dev), torch.empty(nnz, dtype=vt, device=dev)]
    for a in arrs:
        dist.broadcast(a, src, group=group)
    if rank == src:
        return M
    return bmSpMatrix.from_arrays(nr, nc, nblk, arrs[0], arrs[1], arrs[2], arrs[3], transpose=bool(tr))
