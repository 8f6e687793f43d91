// dist.cu -- block-row sharding helpers for multi-GPU runs (SURVEY.md section 8e).
// The reference is single-GPU; these are the only additions to its surface.  SpMV shards by block
// rows (x replicated / all-gathered by the caller over NCCL), SpGEMM shards A's block rows with B
// replicated; the concatenation of the per-shard C arrays (offsets rebased) is bit-identical to the
// single-GPU product.
#include "common.cuh"
#include <vector>
#include <algorithm>

namespace bmsp {

// SpMV cost of a block row in byte units: its blocks and values, plus a per-row term.  The row-tiled kernel pays little per row
// (row pointers, y); the block-parallel kernel spends a whole warp on every block row, worth about 20 blocks of streaming
// (fitted on the R-MAT-22 shards of a 2-GPU run, round 2: 7.9 us per 10^6 blocks + 41 us per 10^6 matrix rows with a warp per block
// row; 23 us per 10^6 rows since short block rows are bundled four to a warp, i.e. a block row costs as much as ~330 bytes of
// streaming).  On that path every rank also stores its finished rows to every peer after the product (an all-gather written by
// the owner), and the step ends when the rank with the MOST rows has pushed them: 32 bytes per block row and peer at the ~750 GB/s
// a rank's NVLink egress sustains = 0.043 us per 10^6 block rows and peer = 76 byte units.  Without that term the rank that got the
// light tail of an R-MAT matrix (1.4 M of 4.2 M rows at 8 GPUs) pushed 40 MB per step while the others waited (round 2, N = 8:
// products of 75-103 us, steps of 161 us).
__global__ void spmv_weight_kernel(const int32_t* __restrict__ brp, const uint32_t* __restrict__ rvb, int nbr, int vsize,
                                   uint64_t row_cost, uint64_t* __restrict__ w) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nbr) return;
    w[r] = (uint64_t)(brp[r + 1] - brp[r]) * 12 + (uint64_t)(rvb[r + 1] - rvb[r]) * vsize + row_cost;
}

// candidate SpGEMM pairs per A block row (warp per row)
__global__ void __launch_bounds__(256) cand_weight_kernel(const int32_t* __restrict__ a_brp, const int32_t* __restrict__ a_bcol,
                                                          const int32_t* __restrict__ b_brp, int nbr, uint64_t* __restrict__ w) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= nbr) return;
    unsigned long long c = 0;
    for (int a = a_brp[row] + lane; a < a_brp[row + 1]; a += 32) {
        const int k = a_bcol[a];
        c += (unsigned long long)(b_brp[k + 1] - b_brp[k]);
    }
    c = warp_sum(c);
    if (lane == 0) w[row] = c + 4;   // + a little per-row overhead so empty rows still spread
}

__global__ void slice_rebase_kernel(uint64_t* __restrict__ keys, uint64_t* __restrict__ offsets, int64_t nblk, int64_t noff,
                                    uint64_t row_shift, uint64_t val_shift) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nblk) keys[i] -= row_shift << 32;
    if (i < noff) offsets[i] -= val_shift;
}

}  // namespace bmsp

using namespace bmsp;

extern "C" int bmsp_partition_block_rows(bmsp_matrix_t A, bmsp_matrix_t Bt, int32_t nparts, int32_t weight_spgemm,
                                         int32_t* bounds, void* stream) {
    if (!A || !bounds || nparts < 1 || (weight_spgemm && !Bt)) { set_error("bmsp_partition_block_rows: invalid argument"); return BMSP_ERR_INVALID; }
    if (weight_spgemm && A->cols != Bt->rows) { set_error("bmsp_partition_block_rows: inner dimensions differ"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    if (Bt) touch(Bt, st);
    const int nbr = A->nbr;
    bounds[0] = 0; bounds[nparts] = nbr;
    if (nbr == 0) { for (int p = 1; p < nparts; p++) bounds[p] = 0; return BMSP_OK; }
    DevBuf<uint64_t> w;
    BMSP_TRY(w.alloc((size_t)nbr + 2, st));
    if (weight_spgemm) cand_weight_kernel<<<(unsigned)ceil_div(nbr, 8), 256, 0, st>>>(A->brp, A->bcol, Bt->brp, nbr, w.get());
    else {
        const uint64_t row_cost = spmv_block_parallel(A) ? 330 + 76 * (uint64_t)(nparts - 1) : 40;
        spmv_weight_kernel<<<(unsigned)ceil_div(nbr, 256), 256, 0, st>>>(A->brp, A->rvb, nbr, (int)dtype_bytes(A->dtype), row_cost, w.get());
    }
    BMSP_KERNEL_CHECK();
    BMSP_TRY(exclusive_scan_u64(w.get(), w.get(), nbr, st));
    std::vector<uint64_t> h((size_t)nbr + 1);
    BMSP_CUDA(cudaMemcpyAsync(h.data(), w.get(), sizeof(uint64_t) * ((size_t)nbr + 1), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    const uint64_t total = h[nbr];
    for (int p = 1; p < nparts; p++) {
        const uint64_t target = (uint64_t)((long double)total * p / nparts);
        int r = (int)(std::lower_bound(h.begin(), h.end(), target) - h.begin());
        bounds[p] = std::min(std::max(r, bounds[p - 1]), nbr);
    }
    return BMSP_OK;
}

extern "C" int bmsp_slice_block_rows(bmsp_matrix_t A, int32_t r0, int32_t r1, int32_t rebase_rows, void* stream, bmsp_matrix_t* out) {
    if (!A || !out || r0 < 0 || r1 > A->nbr || r0 > r1) { set_error("bmsp_slice_block_rows: invalid argument"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    int32_t hb[2] = {0, 0}; uint32_t hv[2] = {0, 0};
    BMSP_CUDA(cudaMemcpyAsync(&hb[0], A->brp + r0, 4, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(&hb[1], A->brp + r1, 4, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(&hv[0], A->rvb + r0, 4, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(&hv[1], A->rvb + r1, 4, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    const int64_t nblk = hb[1] - hb[0], nnz = (int64_t)hv[1] - hv[0];
    const size_t vs = dtype_bytes(A->dtype);
    const int64_t rows = rebase_rows ? std::min<int64_t>((int64_t)(r1 - r0) * 8, (int64_t)A->rows - (int64_t)r0 * 8) : A->rows;
    HandlePtr m;
    BMSP_TRY(new_handle((int32_t)std::max<int64_t>(rows, 0), A->cols, nblk, nnz, A->dtype, A->transposed, st, m));
    if (nblk) {
        BMSP_CUDA(cudaMemcpyAsync(m->keys, A->keys + hb[0], 8 * nblk, cudaMemcpyDeviceToDevice, st));
        BMSP_CUDA(cudaMemcpyAsync(m->bmps, A->bmps + hb[0], 8 * nblk, cudaMemcpyDeviceToDevice, st));
        BMSP_CUDA(cudaMemcpyAsync(m->offsets, A->offsets + hb[0], 8 * nblk, cudaMemcpyDeviceToDevice, st));
        if (nnz) BMSP_CUDA(cudaMemcpyAsync(m->values, (const char*)A->values + (size_t)hv[0] * vs, (size_t)nnz * vs, cudaMemcpyDeviceToDevice, st));
        slice_rebase_kernel<<<(unsigned)ceil_div(nblk, 256), 256, 0, st>>>(m->keys, m->offsets, nblk, nblk, rebase_rows ? (uint64_t)r0 : 0, hv[0]);
        BMSP_KERNEL_CHECK();
    }
    BMSP_TRY(derive_compact(m.get(), st));
    *out = m.release();
    return BMSP_OK;
}
