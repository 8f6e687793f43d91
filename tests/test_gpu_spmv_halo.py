"""The multi-GPU SpMV entry point (bmsp_spmv_halo) on one GPU, with the rank as its own peer.

The "peers'" slots of the inbox hold 1 << 30 before the first call, so every wait is satisfied at once and no call can spin; the rows
a peer would receive land in a scratch sink.  The own column range leaves out the first and last 256 columns, so the first and last
tiles depend on "peers".  Each input states in numpy which path and kernel the plan picks (spmv.cu plan_spmv / plan_tiles).  For two
consecutive epochs every case checks: y == bmSparse_SpMV bit for bit, every pushed slice == its rows of y, every peer slot holds the
signalled epoch, and no wait timed out."""
import ctypes as C

import pytest
import torch

from tests.test_gpu_spmv_palette import _assert_light_rows, _distinct_bitmaps, _patterned_blocks_csr

pytestmark = pytest.mark.gpu

N_PEER = 2
OWN_MARGIN = 256         # columns at either end of x that count as a peer's
SINK_SLICE = 1024        # floats of the sink per push range (16-byte aligned slices)


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _assert_heavy_rows(oracle, nr, nc, rp, ci, v):
    """>= 2.5 values per block is the row-tiled path; an average block row over 320 bytes (bitmaps, x offsets, ~x lines, fp16
    values; fp32 values only add to it) gives 16- or 32-block-row tiles, which run the per-tile kernel"""
    m = oracle.csr_to_bmsp(nr, nc, rp, ci, v)
    nblk, nnz, nbr = m.bmps.size, int(rp[-1]), (nr + 7) // 8
    assert nnz / nblk >= 2.5
    assert (nblk * 26 + nnz * 2) / nbr + 8 > 320


def _assert_block_parallel(oracle, nr, nc, rp, ci, v):
    """fewer than 2.5 values per block: the block-parallel path (wait kernel, product, push kernel)"""
    m = oracle.csr_to_bmsp(nr, nc, rp, ci, v)
    assert int(rp[-1]) / m.bmps.size < 2.5


def _check_halo(B, nr, nc, rp, ci, v, dtype=torch.float16, push=True):
    from bmsparse_spgemm_spmv_b200 import _lib as L
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=dtype)
    x = torch.from_numpy(B.generators.x_vector(nc)).cuda()
    ref = B.bmSparse_SpMV(M, x)
    my_flag = torch.full((N_PEER,), 1 << 30, dtype=torch.int32, device="cuda")
    peer_flag = torch.zeros(N_PEER, dtype=torch.int32, device="cuda")
    scratch = torch.zeros(4, dtype=torch.int32, device="cuda")
    sink = torch.empty(2 * SINK_SLICE, device="cuda")
    # the first rows (a range that ends inside a group of four) and the last rows
    ranges = [(0, 1001), ((nr - 777) & ~3, nr)] if push else []
    desc = L.HaloDesc()
    desc.n_push = len(ranges)
    for i, (lo, hi) in enumerate(ranges):
        desc.push_lo[i] = lo; desc.push_hi[i] = hi; desc.push_dst[i] = sink.data_ptr() + 4 * i * SINK_SLICE
    desc.n_peer = N_PEER
    for i in range(N_PEER):
        desc.peer_flag[i] = peer_flag.data_ptr() + 4 * i
        desc.my_flag[i] = my_flag.data_ptr() + 4 * i
    desc.scratch = scratch.data_ptr()
    desc.own_col_lo = OWN_MARGIN; desc.own_col_hi = nc - OWN_MARGIN
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    y = torch.empty(nr, device="cuda")
    for epoch in (1, 2):
        y.fill_(float("nan")); sink.fill_(float("nan"))
        L.check(L.lib().bmsp_spmv_halo(M._h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), C.byref(desc),
                                       C.c_uint32(epoch), C.c_uint32(epoch + 1), st))
        torch.cuda.synchronize()
        assert torch.equal(y, ref), epoch
        for i, (lo, hi) in enumerate(ranges):
            assert torch.equal(sink[i * SINK_SLICE:i * SINK_SLICE + hi - lo], ref[lo:hi]), (epoch, i)
        assert peer_flag.tolist() == [epoch + 1] * N_PEER, epoch
        assert int(scratch[1]) == 0, "a wait timed out"
        assert my_flag.tolist() == [1 << 30] * N_PEER


def test_streaming_kernel_palette(B, oracle):
    """Poisson, no multiple of a tile: the halo variant of the streaming kernel with a palette, over enough tiles that the last
    part of every CTA's share is claimed at run time"""
    nr, nc, rp, ci, v = B.generators.poisson5pt(1100, 1003)
    assert nr % (64 * 8) != 0
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) <= 256
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    _check_halo(B, nr, nc, rp, ci, v)


def test_streaming_kernel_no_palette(B, oracle):
    nr, nc, rp, ci, v = _patterned_blocks_csr(3000, 257, seed=11)
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) > 256
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    _check_halo(B, nr, nc, rp, ci, v)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_per_tile_kernel(B, oracle, dtype):
    nr, nc, rp, ci, v = B.generators.block_clustered(3001)
    _assert_heavy_rows(oracle, nr, nc, rp, ci, v)
    _check_halo(B, nr, nc, rp, ci, v, dtype=dtype)


def test_block_parallel(B, oracle):
    nr, nc, rp, ci, v = B.generators.uniform_random(20000, 16)
    _assert_block_parallel(oracle, nr, nc, rp, ci, v)
    _check_halo(B, nr, nc, rp, ci, v)


def test_nothing_pushed_still_signals(B, oracle):
    """no push range: the streaming kernel's tile 0 signals on behalf of a rank that pushes nothing"""
    nr, nc, rp, ci, v = B.generators.poisson5pt(300, 221)
    assert _distinct_bitmaps(oracle, nr, nc, rp, ci, v) <= 256
    _assert_light_rows(oracle, nr, nc, rp, ci, v)
    _check_halo(B, nr, nc, rp, ci, v, push=False)
