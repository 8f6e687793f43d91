// add.cu -- C = alpha*A + beta*B for two matrices of the same shape and storage form (no counterpart in the reference).
//
// Both key arrays are sorted (br << 32 | bc), so C's keys are one merge of the two arrays with equal keys collapsed, and a
// block's bitmap is the OR of the two.  Two matrices in the same form number the cells of a block the same way, so the same code
// serves both forms.  The work is split over the merged sequence (merge path), not over block rows: every CTA gets the same number
// of input blocks however they fall over the rows (an R-MAT hub row, the one block row of a transposed dense column).
//   1. partition: the split of every tile boundary of the merged sequence, by a binary search along its diagonal;
//   2. count:     per tile, C's blocks that start in it (heads) and their values;
//   3. size:      two scans over the tile counts; the totals are read back (the call's one synchronisation) to allocate C;
//   4. fill:      the same merge again, each head writing its key, bitmap, value count and source blocks at the tile's base plus
//                 its rank in the tile; a scan of the value counts makes the offsets;
//   5. values:    a CTA per run of consecutive C blocks, its threads striding over the run's contiguous values.
// No atomic decides a position, so two calls give identical arrays.
#include "common.cuh"

namespace bmsp {

// Tile sizes.  The merge kernels stage a tile of 2048 keys (16 KB) in shared memory and give each of 256 threads 8 consecutive
// merge items, the tile of the library's scans and radix passes; a values CTA covers the values of 256 consecutive C blocks.
// Measured with these sizes on one B200 at 1000 W, A + A^T (DESIGN.md section 3.6): partition 0.02-0.05 ms and count 0.13-0.64 ms
// of 1.4-6.8 ms per call; the fill's scattered stores (up to 3.2 ms on RM22) and the values kernel (0.8 ms on P4096) hold the rest.
// No other sizes were measured.
constexpr int MERGE_T = 256, MERGE_ITEMS = 8, MERGE_TILE = MERGE_T * MERGE_ITEMS;
constexpr int VAL_T = 256, VAL_BLOCKS = VAL_T;
constexpr uint32_t NO_BLOCK = 0xFFFFFFFFu;
constexpr uint64_t NO_KEY = ~0ull;        // no valid key: a block row index is below 2^28

// split[t] = how many of A's blocks are among the first min(t * MERGE_TILE, na + nb) items of the merge; on equal keys A's block
// comes first, so the two blocks of a shared key are adjacent in merge order, A's first.
__global__ void add_partition_kernel(const uint64_t* __restrict__ ka, int64_t na, const uint64_t* __restrict__ kb, int64_t nb,
                                     int64_t ntiles, int64_t* __restrict__ split) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > ntiles) return;
    split[t] = merge_path(ka, na, kb, nb, min(t * MERGE_TILE, na + nb));
}

// One CTA per tile of the merge.  An item is a head (the first of C's block) when it comes from A, or when it comes from B and A's
// block just before it in merge order has another key; that test reads A's block before the tile when needed, so a pair split by a
// tile boundary is still collapsed.  An A head takes B's next block as its partner when the keys are equal.
// FILL false: tile_heads[t] / tile_nnz[t] = the tile's heads and the popcount of their bitmaps.
// FILL true:  tile_heads / tile_nnz hold their exclusive scans; each head writes its key, bitmap, popcount (into cnt) and source
//             blocks (NO_BLOCK when absent) at slot tile_heads[t] + its rank in the tile.
template <bool FILL>
__global__ void __launch_bounds__(MERGE_T) add_merge_kernel(const uint64_t* __restrict__ ka, const uint64_t* __restrict__ ba, int64_t na,
                                                            const uint64_t* __restrict__ kb, const uint64_t* __restrict__ bb, int64_t nb,
                                                            const int64_t* __restrict__ split, uint32_t* __restrict__ tile_heads,
                                                            uint64_t* __restrict__ tile_nnz, uint64_t* __restrict__ keys_out,
                                                            uint64_t* __restrict__ bmps_out, uint64_t* __restrict__ cnt,
                                                            uint32_t* __restrict__ src_a, uint32_t* __restrict__ src_b) {
    __shared__ uint64_t s[MERGE_TILE];        // A's keys of the tile, then B's
    __shared__ uint64_t s_prev_a, s_next_b;   // A's key before the tile, B's key after it (NO_KEY: none)
    const int64_t t = blockIdx.x;
    const int64_t d0 = t * MERGE_TILE, d1 = min(d0 + MERGE_TILE, na + nb);
    const int64_t i0 = split[t], i1 = split[t + 1], j0 = d0 - i0, j1 = d1 - i1;
    const int la = (int)(i1 - i0), lb = (int)(j1 - j0), len = la + lb;
    for (int e = threadIdx.x; e < len; e += MERGE_T) s[e] = e < la ? ka[i0 + e] : kb[j0 + e - la];
    if (threadIdx.x == 0) {
        s_prev_a = i0 > 0 ? ka[i0 - 1] : NO_KEY;
        s_next_b = j1 < nb ? kb[j1] : NO_KEY;
    }
    __syncthreads();
    // this thread's items: [diag, diag + MERGE_ITEMS) of the tile, starting at A's ia-th and B's jb-th block of the tile
    const int diag = min((int)threadIdx.x * MERGE_ITEMS, len);
    int ia = merge_path(s, la, s + la, lb, diag), jb = diag - ia;
    const int n_items = min(MERGE_ITEMS, len - diag);
    uint32_t sa[MERGE_ITEMS], sb[MERGE_ITEMS];
    uint32_t heads = 0;
    uint64_t pc = 0;
#pragma unroll
    for (int k = 0; k < MERGE_ITEMS; k++) {
        sa[k] = sb[k] = NO_BLOCK;
        if (k >= n_items) continue;
        if (ia < la && (jb >= lb || s[ia] <= s[la + jb])) {
            const uint64_t next_b = jb < lb ? s[la + jb] : s_next_b;
            sa[k] = (uint32_t)(i0 + ia);
            if (next_b == s[ia]) sb[k] = (uint32_t)(j0 + jb);
            ia++;
        } else {
            const uint64_t prev_a = ia > 0 ? s[ia - 1] : s_prev_a;
            if (prev_a != s[la + jb]) sb[k] = (uint32_t)(j0 + jb);
            jb++;
        }
        if (sa[k] != NO_BLOCK || sb[k] != NO_BLOCK) {
            heads++;
            if (!FILL) pc += __popcll((sa[k] != NO_BLOCK ? ba[sa[k]] : 0) | (sb[k] != NO_BLOCK ? bb[sb[k]] : 0));
        }
    }
    uint32_t total;
    uint32_t slot = cta_exclusive_scan(heads, &total);
    if (!FILL) {
        pc = cta_sum(pc);
        if (threadIdx.x == 0) { tile_heads[t] = total; tile_nnz[t] = pc; }
        return;
    }
    slot += tile_heads[t];
#pragma unroll
    for (int k = 0; k < MERGE_ITEMS; k++) {
        if (sa[k] == NO_BLOCK && sb[k] == NO_BLOCK) continue;
        const uint64_t bmp = (sa[k] != NO_BLOCK ? ba[sa[k]] : 0) | (sb[k] != NO_BLOCK ? bb[sb[k]] : 0);
        keys_out[slot] = sa[k] != NO_BLOCK ? ka[sa[k]] : kb[sb[k]];
        bmps_out[slot] = bmp;
        cnt[slot] = (uint64_t)__popcll(bmp);
        src_a[slot] = sa[k];
        src_b[slot] = sb[k];
        slot++;
    }
}

// the cell of bmp's r-th value (r from 0; cells numbered from the most significant bit)
__device__ __forceinline__ int nth_cell(uint64_t bmp, int r) {
    const uint32_t hi = (uint32_t)(bmp >> 32);
    const int h = __popc(hi);
    return r < h ? 31 - (int)__fns(hi, 31, -(r + 1)) : 63 - (int)__fns((uint32_t)bmp, 31, -(r - h + 1));
}

// the value of cell p in a block with bitmap bmp whose values start at v (0 when the cell is empty or there is no block: bmp 0)
template <typename T>
__device__ __forceinline__ float cell_value(uint64_t bmp, const T* __restrict__ v, uint32_t off, int p) {
    if (!((bmp >> (63 - p)) & 1)) return 0.0f;
    const int rank = p == 0 ? 0 : __popcll(bmp >> (64 - p));
    return val_to_f32(v[off + rank]);
}

// One CTA per VAL_BLOCKS consecutive blocks of C.  Their values are one contiguous range of vc; the CTA's threads stride over it,
// so the stores are coalesced.  A thread finds its block by a binary search over the run's offsets, its cell as the r-th set bit
// of the block's bitmap, and the values of that cell in A and B by popcounts of their bitmaps.  Every cell is
// fl(fl(alpha*a) + fl(beta*b)) in fp32 with a missing value = 0 (explicit _rn intrinsics: no FMA contraction), rounded once to TC.
template <typename TA, typename TB, typename TC>
__global__ void __launch_bounds__(VAL_T) add_values_kernel(const uint64_t* __restrict__ bmps, const uint64_t* __restrict__ offsets, int64_t nblk,
                                                           const uint32_t* __restrict__ src_a, const uint32_t* __restrict__ src_b,
                                                           const uint64_t* __restrict__ bmps_a, const uint64_t* __restrict__ offsets_a,
                                                           const TA* __restrict__ va, const uint64_t* __restrict__ bmps_b,
                                                           const uint64_t* __restrict__ offsets_b, const TB* __restrict__ vb,
                                                           float alpha, float beta, TC* __restrict__ vc) {
    __shared__ uint64_t s_off[VAL_BLOCKS + 1], s_bmp[VAL_BLOCKS], s_bmp_a[VAL_BLOCKS], s_bmp_b[VAL_BLOCKS];
    __shared__ uint32_t s_off_a[VAL_BLOCKS], s_off_b[VAL_BLOCKS];
    const int64_t b0 = (int64_t)blockIdx.x * VAL_BLOCKS;
    const int nb = (int)min((int64_t)VAL_BLOCKS, nblk - b0);
    const int tid = threadIdx.x;
    if (tid < nb) {
        const int64_t b = b0 + tid;
        const uint32_t a = src_a[b], bi = src_b[b];
        s_off[tid] = offsets[b];
        s_bmp[tid] = bmps[b];
        s_bmp_a[tid] = a != NO_BLOCK ? bmps_a[a] : 0;
        s_off_a[tid] = a != NO_BLOCK ? (uint32_t)offsets_a[a] : 0;
        s_bmp_b[tid] = bi != NO_BLOCK ? bmps_b[bi] : 0;
        s_off_b[tid] = bi != NO_BLOCK ? (uint32_t)offsets_b[bi] : 0;
    }
    if (tid == 0) s_off[nb] = offsets[b0 + nb];       // offsets[nblk] = nnz (the scan's total)
    __syncthreads();
    const uint64_t v1 = s_off[nb];
    for (uint64_t v = s_off[0] + tid; v < v1; v += VAL_T) {
        // the last block whose first value is at or before v; s_off[0] <= v < s_off[nb], so the search starts past block 0
        const int lo = upper_bound(s_off, 1, nb, v) - 1;
        const int p = nth_cell(s_bmp[lo], (int)(v - s_off[lo]));
        const float a = cell_value(s_bmp_a[lo], va, s_off_a[lo], p);
        const float b = cell_value(s_bmp_b[lo], vb, s_off_b[lo], p);
        vc[v] = conv<float, TC>(__fadd_rn(__fmul_rn(alpha, a), __fmul_rn(beta, b)));
    }
}

}  // namespace bmsp

using namespace bmsp;

extern "C" {

int bmsp_add(float alpha, bmsp_matrix_t A, float beta, bmsp_matrix_t B, int32_t out_dtype, void* stream, bmsp_matrix_t* C) {
    if (!A || !B || !C || A->rows != B->rows || A->cols != B->cols || (out_dtype != BMSP_F16 && out_dtype != BMSP_F32)) {
        set_error("bmsp_add: invalid argument");
        return BMSP_ERR_INVALID;
    }
    if (A->transposed != B->transposed) {
        set_error("bmsp_add: A and B are stored in different forms (bmsp_block_transpose converts one)");
        return BMSP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    touch(B, st);
    const int64_t na = A->nblk, nb = B->nblk;
    HandlePtr m;
    if (na + nb == 0) {
        BMSP_TRY(new_handle(A->rows, A->cols, 0, 0, out_dtype, A->transposed, st, m));
        BMSP_TRY(derive_compact(m.get(), st));
        *C = m.release();
        return BMSP_OK;
    }
    const int64_t ntiles = ceil_div(na + nb, MERGE_TILE);
    DevBuf<int64_t> split;
    DevBuf<uint32_t> tile_heads;
    DevBuf<uint64_t> tile_nnz;
    BMSP_TRY(split.alloc((size_t)ntiles + 1, st));
    BMSP_TRY(tile_heads.alloc((size_t)ntiles + 1, st));
    BMSP_TRY(tile_nnz.alloc((size_t)ntiles + 1, st));
    add_partition_kernel<<<(unsigned)ceil_div(ntiles + 1, 256), 256, 0, st>>>(A->keys, na, B->keys, nb, ntiles, split.get());
    BMSP_KERNEL_CHECK();
    add_merge_kernel<false><<<(unsigned)ntiles, MERGE_T, 0, st>>>(A->keys, A->bmps, na, B->keys, B->bmps, nb, split.get(), tile_heads.get(),
                                                                 tile_nnz.get(), nullptr, nullptr, nullptr, nullptr, nullptr);
    BMSP_KERNEL_CHECK();
    BMSP_TRY(exclusive_scan_u32(tile_heads.get(), tile_heads.get(), ntiles, st));
    BMSP_TRY(exclusive_scan_u64(tile_nnz.get(), tile_nnz.get(), ntiles, st));
    uint32_t nblk = 0;
    uint64_t nnz = 0;
    BMSP_CUDA(cudaMemcpyAsync(&nblk, tile_heads.get() + ntiles, sizeof(nblk), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(&nnz, tile_nnz.get() + ntiles, sizeof(nnz), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    if (nblk > 0x7FFFFFFFu || nnz > 0xFFFFFFFFull) {
        set_error("bmsp_add: the sum has %llu blocks and %llu values (limits 2^31-1 and 2^32-1)", (unsigned long long)nblk,
                  (unsigned long long)nnz);
        return BMSP_ERR_TOO_LARGE;
    }
    BMSP_TRY(new_handle(A->rows, A->cols, nblk, (int64_t)nnz, out_dtype, A->transposed, st, m));
    {
        DevBuf<uint32_t> src_a, src_b;
        BMSP_TRY(src_a.alloc(nblk, st));
        BMSP_TRY(src_b.alloc(nblk, st));
        add_merge_kernel<true><<<(unsigned)ntiles, MERGE_T, 0, st>>>(A->keys, A->bmps, na, B->keys, B->bmps, nb, split.get(), tile_heads.get(),
                                                                    tile_nnz.get(), m->keys, m->bmps, m->offsets, src_a.get(), src_b.get());
        BMSP_KERNEL_CHECK();
        BMSP_TRY(exclusive_scan_u64(m->offsets, m->offsets, m->nblk, st));       // offsets[nblk] = nnz: the values kernel reads it
        const unsigned grid = (unsigned)ceil_div(m->nblk, VAL_BLOCKS);
        BMSP_TRY(with_value_type(A->dtype, [&](auto ta) { return with_value_type(B->dtype, [&](auto tb) { return with_value_type(out_dtype, [&](auto tc) -> int {
            using TA = decltype(ta); using TB = decltype(tb); using TC = decltype(tc);
            add_values_kernel<TA, TB, TC><<<grid, VAL_T, 0, st>>>(m->bmps, m->offsets, m->nblk, src_a.get(), src_b.get(), A->bmps, A->offsets,
                                                                  (const TA*)A->values, B->bmps, B->offsets, (const TB*)B->values, alpha, beta,
                                                                  (TC*)m->values);
            BMSP_KERNEL_CHECK();
            return BMSP_OK;
        }); }); }));
    }
    BMSP_TRY(derive_compact(m.get(), st));
    *C = m.release();
    return BMSP_OK;
}

}  // extern "C"
