"""GPU parity: bmSparse_SpMV through the C ABI vs the oracle.

Tolerance: fp16 values x fp32 x, fp32 accumulate in a different order than the oracle's double sum:
|y - y_ref| <= 1e-5 * sum_j |a_ij x_j| + tiny   (per row; the bound scales with the row's magnitude)."""
import numpy as np
import pytest
import torch

from tests.util import load_golden, random_csr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bmsparse_spgemm_spmv_b200 as B
    return B


def _spmv_check(B, O, nr, nc, rp, ci, v, x, dtype=torch.float16, x_half=False):
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=dtype)
    exp_m = O.csr_to_bmsp(nr, nc, rp, ci, v, f16=(dtype == torch.float16))
    xt = torch.tensor(x, device="cuda")
    if x_half:
        xt = xt.half(); x = xt.float().cpu().numpy()
    y = torch.full((nr,), 123.0, device="cuda")
    B.bmSparse_SpMV(M, xt, y, False)
    torch.cuda.synchronize()
    ref = O.spmv(exp_m, x)
    absref = O.spmv(O.OracleMatrix(nr, nc, exp_m.keys, exp_m.bmps, exp_m.offsets, np.abs(exp_m.values)), np.abs(x))
    err = np.abs(y.cpu().numpy().astype(np.float64) - ref)
    assert np.all(err <= 1e-5 * absref + 1e-30), f"max err {err.max()} path={M}"
    return M


def test_fixture_exact(B):
    g = load_golden("ragusa16.json")
    M = B.bmSpMatrix.from_coo(24, 24, g["A"]["rows"], g["A"]["cols"], g["A"]["vals"])
    y = B.bmSparse_SpMV(M, torch.ones(24, device="cuda"))
    assert y.cpu().tolist() == g["survey_spmv_ones"]


@pytest.mark.parametrize("shape,density", [((24, 24), 0.3), ((61, 29), 0.2), ((1000, 1000), 0.05), ((513, 2049), 0.4),
                                           ((4000, 3000), 0.002), ((2000, 2000), 0.0008)])
def test_random(B, oracle, shape, density):
    nr, nc = shape
    rp, ci, v = random_csr(nr, nc, density, seed=nr + nc, empty_block_rows=(0, 2) if nr > 24 else ())
    x = np.random.default_rng(1).uniform(-1, 1, nc).astype(np.float32)
    _spmv_check(B, oracle, nr, nc, rp, ci, v, x)
    _spmv_check(B, oracle, nr, nc, rp, ci, v, x, x_half=True)
    _spmv_check(B, oracle, nr, nc, rp, ci, v, x, dtype=torch.float32)


def test_poisson_and_generators(B, oracle):
    G = B.generators
    for gen in (lambda: G.poisson5pt(96, 80), lambda: G.block_clustered(300), lambda: G.uniform_random(3000, 16),
                lambda: G.rmat(12)):
        nr, nc, rp, ci, v = gen()
        _spmv_check(B, oracle, nr, nc, rp, ci, v, G.x_vector(nc))


def test_long_block_row_is_sliced(B, oracle):
    """one block row with far more than 512 blocks (sliced work items + fix-up) next to empty block rows"""
    rng = np.random.default_rng(4)
    nc = 80000
    rows = []
    for r in range(24):
        k = 9000 if r in (9, 10) else (0 if r >= 16 else 3)
        rows.append(np.sort(rng.choice(nc, k, replace=False)))
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int32)
    ci = np.concatenate(rows).astype(np.int32)
    v = rng.uniform(-1, 1, ci.size).astype(np.float16).astype(np.float32)
    _spmv_check(B, oracle, 24, nc, rp, ci, v, rng.uniform(-1, 1, nc).astype(np.float32))


@pytest.mark.parametrize("nbr", [4, 7, 64, 1001, 4099])
def test_block_parallel_bundles_of_short_block_rows(B, oracle, nbr):
    """scattered single entries (fewer than 2.5 per block: the block-parallel path).  Block rows with 0 .. 9 blocks next to each
    other exercise the bundles -- four consecutive block rows of at most 8 blocks share one warp item -- and their boundaries: a
    block row of 9 blocks breaks its group of four, a block-row count that is no multiple of four leaves a ragged tail, and a long
    row in the middle is still sliced."""
    rng = np.random.default_rng(100 + nbr)
    nr, nc = nbr * 8 - 3, 1 << 15
    pattern = [0, 3, 8, 9, 1, 8, 8, 8, 0, 0, 0, 0, 2, 5, 7, 8]
    rows, cols = [], []
    for br in range(nbr):
        k = 700 if (nbr > 64 and br == nbr // 2) else pattern[(br + br // 16) % 16]
        bc = np.sort(rng.choice(nc // 8, k, replace=False))
        for c in bc:                                   # one or two entries per 8x8 block
            for _ in range(1 + int(rng.integers(0, 2))):
                r = br * 8 + int(rng.integers(0, 8))
                if r < nr:
                    rows.append(r); cols.append(int(c) * 8 + int(rng.integers(0, 8)))
    rc = np.unique(np.stack([rows, cols], 1), axis=0) if rows else np.zeros((0, 2), np.int64)
    r, c = rc[:, 0], rc[:, 1]
    v = rng.uniform(-1, 1, r.size).astype(np.float16).astype(np.float32)
    rp = np.zeros(nr + 1, np.int64); np.cumsum(np.bincount(r, minlength=nr), out=rp[1:])
    M = _spmv_check(B, oracle, nr, nc, rp.astype(np.int32), c.astype(np.int32), v, rng.uniform(-1, 1, nc).astype(np.float32))
    assert M.nnz / max(M.block_num, 1) < 2.5


@pytest.mark.parametrize("nparts", [3, 64])
def test_partition_of_a_matrix_without_blocks(B, nparts):
    """an all-zero matrix has no blocks, runs on the block-parallel path, and is partitioned by that path's cost of a block row
    (330 byte units + 76 per peer, dist.cu).  All block rows weigh the same: the bounds are the scan-and-search over equal weights."""
    nr = 1000
    M = B.bmSpMatrix.from_csr(nr, nr, np.zeros(nr + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    assert M.block_num == 0
    assert torch.equal(B.bmSparse_SpMV(M, torch.ones(nr, device="cuda")), torch.zeros(nr, device="cuda"))
    nbr = (nr + 7) // 8
    h = np.arange(nbr + 1, dtype=np.int64) * (330 + 76 * (nparts - 1))
    exp = [0]
    for p in range(1, nparts):
        exp.append(min(max(int(np.searchsorted(h, h[-1] * p // nparts, side="left")), exp[-1]), nbr))
    exp.append(nbr)
    assert M.partition_block_rows(nparts).tolist() == exp


def test_tile_overflow_falls_back_to_global(B, oracle):
    """dense-ish blocks but one tile far above the average: the row-tiled kernel must read it from global"""
    rng = np.random.default_rng(5)
    nr, nc = 1024, 4096
    mask = rng.random((nr, nc)) < 0.004
    mask[100:108, :] = rng.random((8, nc)) < 0.9
    mask[:, :8] |= rng.random((nr, 8)) < 0.9
    r, c = np.nonzero(mask)
    v = rng.uniform(-1, 1, r.size).astype(np.float16).astype(np.float32)
    rp = np.zeros(nr + 1, np.int64); np.cumsum(np.bincount(r, minlength=nr), out=rp[1:])
    _spmv_check(B, oracle, nr, nc, rp.astype(np.int32), c.astype(np.int32), v, rng.uniform(-1, 1, nc).astype(np.float32))


def test_full_size_poisson_properties(B):
    """BASELINE config 2 size (poisson 4096^2): size-independent checks.
    A*1: interior rows sum to 0, edges 1, corners 2 (exact in fp32); linearity A(2x) = 2 A x exactly."""
    G = B.generators
    m = 4096
    nr, nc, rp, ci, v = G.poisson5pt(m, m)
    M = B.bmSpMatrix.from_csr(nr, nc, torch.from_numpy(rp).cuda(), torch.from_numpy(ci).cuda(), torch.from_numpy(v).cuda())
    assert M.nnz == 83869696 and M.block_num == 10476544
    y = B.bmSparse_SpMV(M, torch.ones(nc, device="cuda")).view(m, m)
    exp = torch.zeros(m, m, device="cuda")
    exp[0, :] += 1; exp[-1, :] += 1; exp[:, 0] += 1; exp[:, -1] += 1
    assert torch.equal(y, exp)
    x = torch.from_numpy(G.x_vector(nc)).cuda()
    y1 = B.bmSparse_SpMV(M, x)
    y2 = B.bmSparse_SpMV(M, 2 * x)
    assert torch.equal(2 * y1, y2)
    # against an independent fp64 stencil evaluation
    xg = x.double().view(m, m)
    ref = 4 * xg
    ref[1:, :] -= xg[:-1, :]; ref[:-1, :] -= xg[1:, :]; ref[:, 1:] -= xg[:, :-1]; ref[:, :-1] -= xg[:, 1:]
    assert (y1.double().view(m, m) - ref).abs().max().item() < 1e-5
    assert M.spmv_bytes() == 444452864


def test_host_buffer_pipeline(B):
    """bmsp_spmv_host (x and y in pinned host memory, chunked H2D / launch / D2H pipeline) == bmsp_spmv bit for bit,
    on a banded matrix large enough to be chunked, a scattered one (first chunk needs all of x) and a path-1 matrix."""
    G = B.generators
    # poisson5pt(64, 64): a row-tiled matrix too small to be chunked (ADVICE r1: the one-chunk plan launched no tile at all)
    cases = [G.poisson5pt(640, 512), G.block_clustered(40000), G.uniform_random(300000, 8), G.poisson5pt(64, 64), G.block_clustered(96)]
    rng = np.random.default_rng(9)
    nr, nc = 400000, 400000           # scattered but dense-ish blocks: 8x8 blocks at random block positions
    br = np.repeat(np.arange(nr // 8), 3); bc = rng.integers(0, nc // 8, br.size)
    key = np.unique(br.astype(np.int64) * (nc // 8) + bc)
    br, bc = key // (nc // 8), key % (nc // 8)
    rows = (br[:, None, None] * 8 + np.arange(8)[None, :, None] + np.zeros((1, 1, 4), np.int64)).ravel()
    cols = (bc[:, None, None] * 8 + np.zeros((1, 8, 1), np.int64) + np.array([0, 2, 5, 7])[None, None, :]).ravel()
    o = np.lexsort((cols, rows)); rows, cols = rows[o], cols[o]
    rp = np.zeros(nr + 1, np.int64); np.cumsum(np.bincount(rows, minlength=nr), out=rp[1:])
    cases.append((nr, nc, rp.astype(np.int32), cols.astype(np.int32), rng.uniform(-1, 1, rows.size).astype(np.float16).astype(np.float32)))
    # fp32 matrices too, on both paths (chunked row-tiled, block-parallel)
    runs = [(c, torch.float16) for c in cases] + [(cases[0], torch.float32), (cases[2], torch.float32)]
    for (nr, nc, rp, ci, v), dtype in runs:
        M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v, dtype=dtype)
        for xdt in (torch.float32, torch.float16):
            xh = torch.from_numpy(G.x_vector(nc)).to(xdt).pin_memory()
            yh = torch.full((nr,), 7.0).pin_memory()
            ref = B.bmSparse_SpMV(M, xh.cuda())
            for it in range(4):       # 1st call eager, 2nd captures the pipeline as a CUDA graph, 3rd/4th replay it
                yh.fill_(7.0)
                B.bmSparse_SpMV_host(M, xh, yh)
                torch.cuda.synchronize()
                assert torch.equal(yh, ref.cpu()), (nr, dtype, xdt, it)
            # other buffers after a capture: eager again, then re-captured
            xh2 = (xh.float() * 0.5).to(xdt).pin_memory(); yh2 = torch.empty(nr).pin_memory()
            ref2 = B.bmSparse_SpMV(M, xh2.cuda()).cpu()
            for it in range(3):
                B.bmSparse_SpMV_host(M, xh2, yh2)
                torch.cuda.synchronize()
                assert torch.equal(yh2, ref2), (nr, dtype, xdt, it)
    # pageable host memory works too (slower)
    nr, nc, rp, ci, v = cases[0]
    M = B.bmSpMatrix.from_csr(nr, nc, rp, ci, v)
    xh = torch.from_numpy(G.x_vector(nc)); yh = torch.empty(nr)
    B.bmSparse_SpMV_host(M, xh, yh); torch.cuda.synchronize()
    assert torch.equal(yh, B.bmSparse_SpMV(M, xh.cuda()).cpu())


def test_destroy_is_ordered_behind_side_stream_work(B):
    """ADVICE r1: frees used to go to stream 0, which does not order after non-blocking streams.  A matrix built, multiplied and
    dropped on a side stream while the kernels may still run, with the pool handing the memory to the next allocation straight
    away, must still give the right answers."""
    G = B.generators
    nr, nc, rp, ci, v = G.poisson5pt(512, 512)
    d = lambda a, s: torch.from_numpy(a).cuda()
    side = torch.cuda.Stream()
    x = torch.from_numpy(G.x_vector(nc)).cuda()
    ref = B.bmSparse_SpMV(B.bmSpMatrix.from_csr(nr, nc, rp, ci, v), x).clone()
    torch.cuda.synchronize()
    outs = []
    with torch.cuda.stream(side):
        for it in range(12):
            M = B.bmSpMatrix.from_csr(nr, nc, torch.from_numpy(rp).cuda(), torch.from_numpy(ci).cuda(), torch.from_numpy(v).cuda(), stream=side)
            y = torch.empty(nr, device="cuda")
            B.bmSparse_SpMV(M, x, y, stream=side)
            outs.append(y)
            del M                                    # frees are stream-ordered behind the product above
    side.synchronize()
    for y in outs:
        assert torch.equal(y, ref)
