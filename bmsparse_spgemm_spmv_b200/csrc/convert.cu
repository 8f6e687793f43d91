// convert.cu -- CSR / COO / MatrixMarket -> bmSparse on the device, and the block transpose.
//
// Replaces the reference's ingest path src/bmSpMatrix.cu:111-219 (host parse -> thrust::sort with a
// 4-level comparator -> 2 reduce_by_key + scan + 2 transforms) and src/reader.cu:49-110.
// Same mapping (Appendix A of SURVEY.md), different algorithm: CSR rows are already sorted, so the
// block-row order of an entry is a sum of eight binary searches (an 8-way merge rank) -- no global
// sort.  Block ids are a CTA scan of the head flags, bitmaps a warp-segmented OR by shuffle, and values
// are compacted with 16-byte stores.
#include "common.cuh"
#include <vector>
#include <algorithm>
#include <numeric>
#include <fstream>
#include <string>
#include <cstring>
#include <cstdlib>
#include <cctype>
#include <thread>

namespace bmsp {

enum { FLAG_UNSORTED = 1, FLAG_DUP = 2, FLAG_RANGE = 4, FLAG_ROWPTR = 8 };

// row_ptr of a device CSR: starts at 0, ends at nnz, never decreases (rank_kernel binary-searches it and would read out of
// bounds on anything else)
__global__ void check_rowptr_kernel(const int32_t* __restrict__ rp, int32_t rows, int64_t nnz, int32_t* __restrict__ flags) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > rows) return;
    const int32_t v = rp[r];
    bool bad = v < 0 || (int64_t)v > nnz;
    if (r == 0) bad |= v != 0;
    if (r == rows) bad |= (int64_t)v != nnz;
    else bad |= rp[r + 1] < v;
    if (bad) atomicOr(flags, FLAG_ROWPTR);
}

// K0: the row of the first entry of every chunk of RANK_T entries (last r with rp[r] <= e), one thread per chunk.  The only
// place that searches all of row_ptr: a search per ENTRY was 24 dependent L2 round trips on a 16 M-row matrix and two thirds of the
// whole conversion (ncu launch list, profiles/r2_bench_launches_summary.txt).
constexpr int RANK_T = 256, RANK_SPAN = 1024;
__global__ void chunk_row_kernel(const int32_t* __restrict__ rp, int32_t rows, int64_t nnz, int32_t* __restrict__ chunk_row, int64_t nchunks) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b > nchunks) return;
    if (b == nchunks) { chunk_row[b] = rows - 1; return; }
    const int64_t e = b * RANK_T;
    chunk_row[b] = upper_bound(rp, 1, rows, e) - 1;   // rp[0] = 0 <= e < nnz = rp[rows]: the search starts past row 0
}

// K1: one thread per CSR entry, a CTA per chunk of RANK_T entries.  The chunk's rows lie between the rows of its first entry and
// of the next chunk's first entry: their row_ptr values go to shared memory and every thread finds its row there.  It then
// validates, computes its position in the block-row order (block column, then row-major or column-major inside the block:
// block_order, bmSpMatrix.cu:45-74) and scatters (key, cell position, source index) there.
template <bool TRANSPOSED>
__global__ void __launch_bounds__(RANK_T) rank_kernel(const int32_t* __restrict__ rp, const int32_t* __restrict__ ci, int32_t rows,
                                                      int32_t cols, int64_t nnz, const int32_t* __restrict__ chunk_row,
                                                      uint64_t* __restrict__ s_key, uint8_t* __restrict__ s_p, int32_t* __restrict__ s_src,
                                                      int32_t* __restrict__ flags) {
    __shared__ int32_t srp[RANK_SPAN + 1];
    const int r_lo = chunk_row[blockIdx.x], r_hi = chunk_row[blockIdx.x + 1];
    const int span = r_hi - r_lo + 1;                         // rows r_lo .. r_hi; rp[r_hi + 1] is past every entry of the chunk
    const bool in_smem = span <= RANK_SPAN;
    if (in_smem)
        for (int i = threadIdx.x; i <= span; i += RANK_T) srp[i] = __ldg(rp + r_lo + i);
    __syncthreads();
    int64_t e = (int64_t)blockIdx.x * RANK_T + threadIdx.x;
    if (e >= nnz) return;
    // row = last r with rp[r] <= e; rp[r_lo] <= e < rp[r_hi + 1], so the search starts past r_lo
    const int r = in_smem ? r_lo + upper_bound(srp, 1, span, e) - 1 : upper_bound(rp, r_lo + 1, r_hi + 1, e) - 1;
    const int c = ci[e];
    if (c < 0 || c >= cols) { atomicOr(flags, FLAG_RANGE); return; }
    const int rs = __ldg(rp + r);
    if (e > rs) {
        int prev = ci[e - 1];
        if (prev == c) atomicOr(flags, FLAG_DUP);
        else if (prev > c) atomicOr(flags, FLAG_UNSORTED);
    }
    const int br = r >> 3, bc = c >> 3, ri = r & 7, cidx = c & 7;
    const int r0 = br << 3;
    int pos = (int)(e - rs);   // entries of the own row with a smaller column
#pragma unroll
    for (int q = 0; q < 8; q++) {
        int rr = r0 + q;
        if (q == ri || rr >= rows) continue;
        int s = __ldg(rp + rr), t = __ldg(rp + rr + 1);
        int target;
        if (TRANSPOSED) target = q < ri ? c + 1 : c;                   // (bc, ci, ri) order
        else            target = q < ri ? (bc + 1) << 3 : bc << 3;      // (bc, ri, ci) order
        pos += lower_bound(ci, s, t, target) - s;
    }
    int64_t g = (int64_t)__ldg(rp + r0) + pos;
    s_key[g] = ((uint64_t)(uint32_t)br << 32) | (uint32_t)bc;
    s_p[g] = (uint8_t)(TRANSPOSED ? cidx * 8 + ri : ri * 8 + cidx);
    s_src[g] = (int32_t)e;
}

// K2: heads per tile of 1024 sorted entries.
__global__ void __launch_bounds__(1024) head_count_kernel(const uint64_t* __restrict__ s_key, int64_t nnz,
                                                          uint32_t* __restrict__ counts) {
    int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    bool head = false;
    if (i < nnz) head = (i == 0) || (s_key[i] != s_key[i - 1]);
    const uint32_t n = cta_sum(head);
    if (threadIdx.x == 0) counts[blockIdx.x] = n;
}

// K3: block ids from the scanned head counts; keys/offsets/block columns by the head lanes; bitmaps by
// a warp-segmented OR (entries of one block are contiguous) finished with one atomicOr per segment.
__global__ void __launch_bounds__(1024) emit_kernel(const uint64_t* __restrict__ s_key, const uint8_t* __restrict__ s_p,
                                                    int64_t nnz, const uint32_t* __restrict__ tile_base,
                                                    uint64_t* __restrict__ keys, uint64_t* __restrict__ bmps,
                                                    uint64_t* __restrict__ offsets) {
    int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    uint64_t key = 0;
    bool head = false;
    if (i < nnz) { key = s_key[i]; head = (i == 0) || (key != s_key[i - 1]); }
    uint32_t tile_heads;
    // inclusive head count up to this entry, minus one = block id
    int32_t blk = (int32_t)(tile_base[blockIdx.x] + cta_exclusive_scan(head, &tile_heads) + head) - 1;
    if (i >= nnz) blk = -1;
    uint32_t hi = 0, lo = 0;
    if (i < nnz) {
        int p = s_p[i];
        if (p < 32) hi = 0x80000000u >> p; else lo = 0x80000000u >> (p - 32);
        if (head) { keys[blk] = key; offsets[blk] = (uint64_t)i; }
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t th = __shfl_up_sync(0xffffffffu, hi, o), tl = __shfl_up_sync(0xffffffffu, lo, o);
        int32_t tb = __shfl_up_sync(0xffffffffu, blk, o);
        if (lane >= o && tb == blk) { hi |= th; lo |= tl; }
    }
    int32_t nb = __shfl_down_sync(0xffffffffu, blk, 1);
    if (blk >= 0 && (lane == 31 || nb != blk))
        atomicOr((unsigned long long*)(bmps + blk), ((unsigned long long)hi << 32) | lo);
}

// K4: values in sorted order, 8 per thread, 16-byte stores (conv: common.cuh).
template <typename Tin, typename Tout>
__global__ void __launch_bounds__(256) values_kernel(const Tin* __restrict__ vals, const int32_t* __restrict__ s_src, int64_t nnz,
                                                     Tout* __restrict__ out) {
    int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i0 >= nnz) return;
    Tout v[8];
    if (i0 + 8 <= nnz) {
        int4 a = *reinterpret_cast<const int4*>(s_src + i0), b = *reinterpret_cast<const int4*>(s_src + i0 + 4);
        int idx[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = conv<Tin, Tout>(vals[idx[k]]);
        if (sizeof(Tout) == 2) {
            *reinterpret_cast<int4*>(out + i0) = *reinterpret_cast<int4*>(v);
        } else {
            *reinterpret_cast<int4*>(out + i0) = *reinterpret_cast<int4*>(v);
            *reinterpret_cast<int4*>(out + i0 + 4) = *reinterpret_cast<int4*>(v + 4);
        }
    } else {
        for (int64_t i = i0; i < nnz; i++) out[i] = conv<Tin, Tout>(vals[s_src[i]]);
    }
}

// device CSR -> new matrix
static int convert_device_csr(int32_t rows, int32_t cols, int64_t nnz, const int32_t* rp, const int32_t* ci, const void* vals,
                              int vals_dtype, int transposed, int out_dtype, cudaStream_t st, bmsp_matrix_t* out) {
    if (nnz > 0xFFFFFFFFll) { set_error("nnz %lld exceeds 2^32-1", (long long)nnz); return BMSP_ERR_TOO_LARGE; }
    DevBuf<uint64_t> s_key; DevBuf<uint8_t> s_p; DevBuf<int32_t> s_src, flags, chunk_row; DevBuf<uint32_t> counts;
    int64_t tiles = ceil_div(nnz, 1024);
    uint32_t nblk32 = 0;
    BMSP_TRY(flags.alloc(1, st));
    BMSP_CUDA(cudaMemsetAsync(flags.get(), 0, sizeof(int32_t), st));
    {
        check_rowptr_kernel<<<(unsigned)ceil_div((int64_t)rows + 1, 256), 256, 0, st>>>(rp, rows, nnz, flags.get());
        BMSP_KERNEL_CHECK();
        int32_t hflags = 0;
        BMSP_CUDA(cudaMemcpyAsync(&hflags, flags.get(), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
        if (hflags & FLAG_ROWPTR) { set_error("row_ptr must start at 0, end at nnz and never decrease"); return BMSP_ERR_INVALID; }
    }
    if (nnz > 0) {
        BMSP_TRY(s_key.alloc((size_t)nnz, st));
        BMSP_TRY(s_p.alloc((size_t)nnz, st));
        BMSP_TRY(s_src.alloc((size_t)nnz + 8, st));
        BMSP_TRY(counts.alloc((size_t)tiles + 1, st));
        const int64_t nchunks = ceil_div(nnz, RANK_T);
        BMSP_TRY(chunk_row.alloc((size_t)nchunks + 1, st));
        chunk_row_kernel<<<(unsigned)ceil_div(nchunks + 1, 256), 256, 0, st>>>(rp, rows, nnz, chunk_row.get(), nchunks);
        BMSP_KERNEL_CHECK();
        unsigned grid = (unsigned)nchunks;
        if (transposed) rank_kernel<true><<<grid, RANK_T, 0, st>>>(rp, ci, rows, cols, nnz, chunk_row.get(), s_key.get(), s_p.get(), s_src.get(), flags.get());
        else            rank_kernel<false><<<grid, RANK_T, 0, st>>>(rp, ci, rows, cols, nnz, chunk_row.get(), s_key.get(), s_p.get(), s_src.get(), flags.get());
        BMSP_KERNEL_CHECK();
        int32_t hflags = 0;
        BMSP_CUDA(cudaMemcpyAsync(&hflags, flags.get(), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
        if (hflags & FLAG_RANGE) { set_error("column index outside [0, %d)", cols); return BMSP_ERR_RANGE; }
        if (hflags & FLAG_UNSORTED) { set_error("CSR column indices must ascend inside each row"); return BMSP_ERR_UNSORTED; }
        if (hflags & FLAG_DUP) { set_error("duplicate (row, col) entries are not supported"); return BMSP_ERR_DUPLICATE; }
        head_count_kernel<<<(unsigned)tiles, 1024, 0, st>>>(s_key.get(), nnz, counts.get());
        BMSP_KERNEL_CHECK();
        BMSP_TRY(exclusive_scan_u32(counts.get(), counts.get(), tiles, st));
        BMSP_CUDA(cudaMemcpyAsync(&nblk32, counts.get() + tiles, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
    }
    HandlePtr m;
    BMSP_TRY(new_handle(rows, cols, nblk32, nnz, out_dtype, transposed, st, m));
    if (nnz > 0) {
        BMSP_CUDA(cudaMemsetAsync(m->bmps, 0, sizeof(uint64_t) * m->nblk, st));
        emit_kernel<<<(unsigned)tiles, 1024, 0, st>>>(s_key.get(), s_p.get(), nnz, counts.get(), m->keys, m->bmps, m->offsets);
        BMSP_KERNEL_CHECK();
        const unsigned grid = (unsigned)ceil_div(ceil_div(nnz, 8), 256);
        BMSP_TRY(with_value_type(vals_dtype, [&](auto in) { return with_value_type(out_dtype, [&](auto out) -> int {
            using Tin = decltype(in); using Tout = decltype(out);
            values_kernel<Tin, Tout><<<grid, 256, 0, st>>>((const Tin*)vals, s_src.get(), nnz, (Tout*)m->values);
            BMSP_KERNEL_CHECK();
            return BMSP_OK;
        }); }));
    }
    BMSP_TRY(derive_compact(m.get(), st));
    *out = m.release();
    return BMSP_OK;
}

// ---------------------------------------------------------------------------- block transpose
// (transpose8x8: common.cuh)
// The values of one block in the other cell order: the value of cell p=(hi,lo) of bmp moves to the rank of cell (lo,hi) in
// t = transpose8x8(bmp).  vin / vout point at the block's first value.
template <typename Tin, typename Tout>
__device__ __forceinline__ void permute_block_values(uint64_t bmp, uint64_t t, const Tin* __restrict__ vin, Tout* __restrict__ vout) {
    uint64_t rem = bmp;
    int k = 0;
    while (rem) {
        int p = __clzll((long long)rem);
        rem &= ~(0x8000000000000000ull >> p);
        int q = ((p & 7) << 3) | (p >> 3);
        int rank = q == 0 ? 0 : __popcll(t >> (64 - q));
        vout[rank] = conv<Tin, Tout>(vin[k]);
        k++;
    }
}

// One thread per block: new bitmap = transpose, values permuted inside the block.
template <typename Tin, typename Tout>
__global__ void block_transpose_kernel(const uint64_t* __restrict__ bmps, const uint64_t* __restrict__ offsets,
                                       const Tin* __restrict__ vin, uint64_t* __restrict__ bmps_out,
                                       Tout* __restrict__ vout, int64_t nblk) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    uint64_t bmp = bmps[b], t = transpose8x8(bmp), off = offsets[b];
    bmps_out[b] = t;
    permute_block_values(bmp, t, vin + off, vout + off);
}

// ---------------------------------------------------------------------------- matrix transpose
// A^T's block (bc, br) is A's block (br, bc), so A^T's blocks in key order are A's blocks stably sorted by block column: A is
// sorted by (br, bc), and a stable sort keeps the blocks of one column in block-row order.  The sort is an LSD radix sort of
// (block column, block index) with 8-bit digits; each pass is a per-tile digit histogram, one scan over the [digit][tile] table
// and a scatter that ranks equal digits inside the tile in input order (match_any per warp, per-warp running counts).  No atomic
// decides a position, so the result is the same on every run.
constexpr int RADIX_T = 256, RADIX_ITEMS = 8, RADIX_TILE = RADIX_T * RADIX_ITEMS, RADIX_WARPS = RADIX_T / 32;

__global__ void __launch_bounds__(RADIX_T) radix_hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, uint32_t* __restrict__ hist,
                                                             int64_t ntiles) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * RADIX_TILE;
#pragma unroll
    for (int i = 0; i < RADIX_ITEMS; i++) {
        const int64_t e = base + i * RADIX_T + threadIdx.x;
        if (e < n) atomicAdd(&h[(keys[e] >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    hist[(int64_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

// pos: the exclusive scan of radix_hist_kernel's table.  vals_in nullptr: the value of an element is its index (the first pass);
// keys_out nullptr: the keys are not needed after this pass (the last one).
__global__ void __launch_bounds__(RADIX_T) radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, int64_t n,
                                                                int shift, const uint32_t* __restrict__ pos, int64_t ntiles,
                                                                uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
    __shared__ uint32_t cnt[RADIX_WARPS][256];      // per warp and digit: elements seen so far, then the warp's first output slot
    for (int i = threadIdx.x; i < RADIX_WARPS * 256; i += RADIX_T) (&cnt[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t wbase = (int64_t)blockIdx.x * RADIX_TILE + (int64_t)w * 32 * RADIX_ITEMS;   // each warp owns a contiguous run
    uint32_t key[RADIX_ITEMS], rank[RADIX_ITEMS];
#pragma unroll
    for (int i = 0; i < RADIX_ITEMS; i++) {
        const int64_t e = wbase + i * 32 + lane;
        const bool valid = e < n;                   // the invalid elements are the tile's last ones: they rank after every valid one
        key[i] = valid ? keys_in[e] : 0u;
        const uint32_t d = (key[i] >> shift) & 0xFFu;
        const uint32_t peers = __match_any_sync(0xffffffffu, valid ? d : 256u);
        rank[i] = cnt[w][d] + __popc(peers & ((1u << lane) - 1u));
        __syncwarp();
        if (valid && lane == __ffs(peers) - 1) cnt[w][d] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    {
        uint32_t run = pos[(int64_t)threadIdx.x * ntiles + blockIdx.x];      // RADIX_T == 256: one thread per digit
#pragma unroll
        for (int q = 0; q < RADIX_WARPS; q++) { const uint32_t c = cnt[q][threadIdx.x]; cnt[q][threadIdx.x] = run; run += c; }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < RADIX_ITEMS; i++) {
        const int64_t e = wbase + i * 32 + lane;
        if (e >= n) continue;
        const uint32_t slot = cnt[w][(key[i] >> shift) & 0xFFu] + rank[i];
        if (keys_out) keys_out[slot] = key[i];
        vals_out[slot] = vals_in ? vals_in[e] : (uint32_t)e;
    }
}

// One thread per block of A^T: src[j] is its block in A (src nullptr: the same index).  Key (br, bc) -> (bc, br) is a rotation
// by 32 bits; the bitmap is transposed when A's form and A^T's are the same (flip); the block's value count goes to cnt for the
// scan that makes the offsets.
__global__ void transpose_blocks_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ bmps, const uint32_t* __restrict__ src,
                                        int64_t nblk, int flip, uint64_t* __restrict__ keys_out, uint64_t* __restrict__ bmps_out,
                                        uint64_t* __restrict__ cnt) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nblk) return;
    const int64_t s = src ? (int64_t)src[j] : j;
    const uint64_t key = keys[s], bmp = bmps[s];
    keys_out[j] = (key << 32) | (key >> 32);
    bmps_out[j] = flip ? transpose8x8(bmp) : bmp;
    cnt[j] = (uint64_t)__popcll(bmp);
}

// One thread per block of A^T: its values from A's block src[j], copied in order or permuted (flip), converted to Tout.
template <typename Tin, typename Tout>
__global__ void transpose_values_kernel(const uint64_t* __restrict__ bmps, const uint64_t* __restrict__ offsets, const Tin* __restrict__ vin,
                                        const uint32_t* __restrict__ src, int64_t nblk, int flip, const uint64_t* __restrict__ offsets_out,
                                        Tout* __restrict__ vout) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nblk) return;
    const int64_t s = src ? (int64_t)src[j] : j;
    const uint64_t bmp = bmps[s];
    const Tin* in = vin + offsets[s];
    Tout* out = vout + offsets_out[j];
    if (flip) {
        permute_block_values(bmp, transpose8x8(bmp), in, out);
    } else {
        const int n = __popcll(bmp);
        for (int k = 0; k < n; k++) out[k] = conv<Tin, Tout>(in[k]);
    }
}

// src[j] = A's block that becomes A^T's block j; *src nullptr when A has at most one block column (the order is A's)
static int transpose_block_order(const bmsp_matrix_s* A, cudaStream_t st, DevBuf<uint32_t> (&kbuf)[2], DevBuf<uint32_t> (&vbuf)[2],
                                 const uint32_t** src) {
    *src = nullptr;
    const int64_t n = A->nblk, nbc = ceil_div(A->cols, 8);
    int bits = 0;
    while (bits < 32 && ((uint64_t)(nbc - 1) >> bits)) bits++;
    const int passes = (bits + 7) / 8;
    if (n == 0 || passes == 0) return BMSP_OK;
    const int64_t ntiles = ceil_div(n, RADIX_TILE);
    DevBuf<uint32_t> pos;
    BMSP_TRY(pos.alloc((size_t)ntiles * 256 + 1, st));
    for (int b = 0; b < 2; b++) {
        if (passes > 1 + b) BMSP_TRY(kbuf[b].alloc((size_t)n, st));
        if (passes > b) BMSP_TRY(vbuf[b].alloc((size_t)n, st));
    }
    const uint32_t* keys = (const uint32_t*)A->bcol;
    const uint32_t* vals = nullptr;
    for (int p = 0; p < passes; p++) {
        const int shift = 8 * p;
        radix_hist_kernel<<<(unsigned)ntiles, RADIX_T, 0, st>>>(keys, n, shift, pos.get(), ntiles);
        BMSP_KERNEL_CHECK();
        BMSP_TRY(exclusive_scan_u32(pos.get(), pos.get(), ntiles * 256, st));
        uint32_t* kout = p + 1 < passes ? kbuf[p & 1].get() : nullptr;
        radix_scatter_kernel<<<(unsigned)ntiles, RADIX_T, 0, st>>>(keys, vals, n, shift, pos.get(), ntiles, kout, vbuf[p & 1].get());
        BMSP_KERNEL_CHECK();
        keys = kout; vals = vbuf[p & 1].get();
    }
    *src = vals;
    return BMSP_OK;
}

}  // namespace bmsp

using namespace bmsp;

extern "C" {

int bmsp_create_from_csr(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_ptr, const int32_t* col_idx,
                         const void* vals, int32_t vals_dtype, int32_t mem, int32_t transposed, int32_t out_dtype,
                         void* stream, bmsp_matrix_t* out) {
    if (!out || rows < 0 || cols < 0 || nnz < 0 || !row_ptr || (nnz > 0 && (!col_idx || !vals)) ||
        (vals_dtype != BMSP_F16 && vals_dtype != BMSP_F32) || (out_dtype != BMSP_F16 && out_dtype != BMSP_F32)) {
        set_error("bmsp_create_from_csr: invalid argument");
        return BMSP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (mem != BMSP_DEVICE && !host_row_ptr_spans(row_ptr, rows, nnz)) { set_error("row_ptr[0] must be 0 and row_ptr[rows] == nnz"); return BMSP_ERR_INVALID; }
    DevBuf<char> d_rp, d_ci, d_v;
    BMSP_TRY(stage(d_rp, row_ptr, sizeof(int32_t) * ((size_t)rows + 1), mem, st));
    BMSP_TRY(stage(d_ci, col_idx, sizeof(int32_t) * (size_t)nnz, mem, st));
    BMSP_TRY(stage(d_v, vals, (size_t)nnz * dtype_bytes(vals_dtype), mem, st));
    BMSP_TRY(convert_device_csr(rows, cols, nnz, row_ptr, col_idx, vals, vals_dtype, transposed, out_dtype, st, out));
    if (mem != BMSP_DEVICE) BMSP_CUDA(cudaStreamSynchronize(st));      // host buffers may be freed by the caller
    return BMSP_OK;
}

// host COO -> matrix; duplicates summed when `merge`
static int coo_to_matrix(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_idx, const int32_t* col_idx, const double* vals,
                         int32_t transposed, int32_t out_dtype, int32_t flags, void* stream, bmsp_matrix_t* out) {
    std::vector<int32_t> rp, ci;
    std::vector<double> dv;
    if (coo_to_csr_host(rows, nnz, row_idx, col_idx, vals, rp, ci, dv)) { set_error("row index outside [0, %d)", rows); return BMSP_ERR_RANGE; }
    int64_t n = nnz;
    if (flags & BMSP_MERGE_DUPLICATES) {
        // repeated (row, col) entries are summed in file order (what assembling a finite-element matrix means by them); the
        // reference keeps them apart and corrupts its offsets (SURVEY Appendix B), without this flag they are rejected
        std::vector<int32_t> nrp((size_t)rows + 1, 0);
        int64_t w = 0;
        for (int32_t r = 0; r < rows; r++) {
            for (int64_t i = rp[r]; i < rp[r + 1]; i++) {
                if (i > rp[r] && ci[i] == ci[w - 1] && w > nrp[r]) dv[w - 1] += dv[i];
                else { ci[w] = ci[i]; dv[w] = dv[i]; w++; }
            }
            nrp[r + 1] = (int32_t)w;
        }
        rp.swap(nrp); n = w;
    }
    if (out_dtype == BMSP_F16) {
        std::vector<__half> v((size_t)n);
        for (int64_t i = 0; i < n; i++) v[i] = __double2half(dv[i]);
        return bmsp_create_from_csr(rows, cols, n, rp.data(), ci.data(), v.data(), BMSP_F16, BMSP_HOST, transposed, BMSP_F16, stream, out);
    }
    std::vector<float> v((size_t)n);
    for (int64_t i = 0; i < n; i++) v[i] = (float)dv[i];
    return bmsp_create_from_csr(rows, cols, n, rp.data(), ci.data(), v.data(), BMSP_F32, BMSP_HOST, transposed, out_dtype, stream, out);
}

int bmsp_create_from_coo_ex(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_idx, const int32_t* col_idx,
                            const double* vals, int32_t transposed, int32_t out_dtype, int32_t flags, void* stream, bmsp_matrix_t* out) {
    if (!out || rows < 0 || cols < 0 || nnz < 0 || (nnz > 0 && (!row_idx || !col_idx || !vals))) {
        set_error("bmsp_create_from_coo: invalid argument");
        return BMSP_ERR_INVALID;
    }
    // values cast straight from double (bmSpMatrix.cu:136-157 casts the parsed double to valueType in one rounding)
    return coo_to_matrix(rows, cols, nnz, row_idx, col_idx, vals, transposed, out_dtype, flags, stream, out);
}

int bmsp_create_from_coo(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_idx, const int32_t* col_idx,
                         const double* vals, int32_t transposed, int32_t out_dtype, void* stream, bmsp_matrix_t* out) {
    return bmsp_create_from_coo_ex(rows, cols, nnz, row_idx, col_idx, vals, transposed, out_dtype, 0, stream, out);
}

// MatrixMarket coordinate files.  Banner rules follow cusp's reader (cusp/io/detail/matrix_market.inl:70-95): five tokens,
// storage coordinate | array, type real | integer | pattern | complex, symmetry general | symmetric | skew-symmetric | hermitian.
//   pattern            value 1 (:171)                       integer           parsed like real (:177-190)
//   symmetric          off-diagonal entries mirrored (:257-279; bmSpMatrix.cu:113-149 does the same)
//   skew-symmetric     mirrored with the sign flipped (cusp throws not_implemented :286-290; the reference's own reader would mirror it
//                      with the SAME sign because "skew-symmetric" contains "symmetric", bmSpMatrix.cu:113-120)
//   complex, hermitian, array storage: BMSP_ERR_UNSUPPORTED (a real-valued bmSpMatrix cannot hold them; cusp keeps only the real part)
// Indices are checked against the size line (:222-235).  The body is parsed by all host cores: the text is cut at line ends into
// one slice per thread (strtol / strtod, no streams).
int bmsp_create_from_mtx_ex(const char* path, int32_t transposed, int32_t out_dtype, int32_t flags, void* stream, bmsp_matrix_t* out) {
    if (!path || !out) { set_error("bmsp_create_from_mtx: null argument"); return BMSP_ERR_INVALID; }
    std::ifstream f(path, std::ios::binary);
    if (!f) { set_error("cannot open %s", path); return BMSP_ERR_IO; }
    std::string content((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    const char* p = content.c_str();
    const char* end = p + content.size();
    auto line_end = [&](const char* q) { while (q < end && *q != '\n') q++; return q; };
    const char* le = line_end(p);
    std::string banner(p, le);
    std::vector<std::string> tok;
    {
        size_t i = 0;
        while (i < banner.size()) {
            while (i < banner.size() && isspace((unsigned char)banner[i])) i++;
            size_t j = i;
            while (j < banner.size() && !isspace((unsigned char)banner[j])) j++;
            if (j > i) tok.push_back(banner.substr(i, j - i));
            i = j;
        }
        for (auto& t : tok) for (auto& ch : t) ch = (char)tolower((unsigned char)ch);
    }
    bool symmetric = false, skew = false, pattern = false;
    if (tok.size() == 5 && tok[0] == "%%matrixmarket") {
        if (tok[1] != "matrix") { set_error("%s: invalid MatrixMarket banner", path); return BMSP_ERR_IO; }
        if (tok[2] == "array") { set_error("%s: array storage is not supported (coordinate files only)", path); return BMSP_ERR_UNSUPPORTED; }
        if (tok[2] != "coordinate") { set_error("%s: invalid MatrixMarket storage format [%s]", path, tok[2].c_str()); return BMSP_ERR_IO; }
        if (tok[3] == "complex") { set_error("%s: complex matrices are not supported", path); return BMSP_ERR_UNSUPPORTED; }
        if (tok[3] == "pattern") pattern = true;
        else if (tok[3] != "real" && tok[3] != "integer") { set_error("%s: invalid MatrixMarket data type [%s]", path, tok[3].c_str()); return BMSP_ERR_IO; }
        if (tok[4] == "hermitian") { set_error("%s: hermitian matrices are not supported", path); return BMSP_ERR_UNSUPPORTED; }
        if (tok[4] == "symmetric") symmetric = true;
        else if (tok[4] == "skew-symmetric") skew = true;
        else if (tok[4] != "general") { set_error("%s: invalid MatrixMarket symmetry [%s]", path, tok[4].c_str()); return BMSP_ERR_IO; }
    } else {
        // no well-formed banner: the reference's rule -- "symmetric" anywhere in the first line (bmSpMatrix.cu:113-120)
        symmetric = banner.find("symmetric") != std::string::npos;
        pattern = banner.find("pattern") != std::string::npos;
        if (!banner.empty() && banner[0] != '%') le = p - 1;          // the first line already is the size line
    }
    p = le < end ? le + 1 : end;
    while (p < end && (*p == '%' || *p == '\n' || *p == '\r')) { le = line_end(p); p = le < end ? le + 1 : end; }
    char* q = nullptr;
    long nr = strtol(p, &q, 10); p = q;
    long nc = strtol(p, &q, 10); p = q;
    long long nl = strtoll(p, &q, 10); p = q;
    if (nr <= 0 || nc <= 0 || nl < 0 || nr > 0x7FFFFFFFl || nc > 0x7FFFFFFFl) { set_error("%s: bad size line", path); return BMSP_ERR_IO; }
    le = line_end(p); p = le < end ? le + 1 : end;
    // slices of whole lines, one per thread
    int nth = (int)std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
    if ((end - p) < (1 << 20)) nth = 1;
    std::vector<const char*> cut((size_t)nth + 1);
    cut[0] = p; cut[nth] = end;
    for (int t = 1; t < nth; t++) { const char* c = p + (end - p) * t / nth; c = line_end(c); cut[t] = c < end ? c + 1 : end; }
    struct Part { std::vector<int32_t> r, c; std::vector<double> v; int err = 0; long long lines = 0; };
    std::vector<Part> parts((size_t)nth);
    auto parse = [&](int t) {
        Part& P = parts[(size_t)t];
        const char* s = cut[t]; const char* e = cut[t + 1];
        P.r.reserve((size_t)((e - s) / 12 + 16)); P.c.reserve(P.r.capacity()); P.v.reserve(P.r.capacity());
        char* qq = nullptr;
        while (s < e) {
            while (s < e && (*s == ' ' || *s == '\t' || *s == '\r' || *s == '\n')) s++;
            if (s >= e) break;
            if (*s == '%') { while (s < e && *s != '\n') s++; continue; }
            long i = strtol(s, &qq, 10); if (qq == s) { P.err = BMSP_ERR_IO; return; } s = qq;
            long j = strtol(s, &qq, 10); if (qq == s) { P.err = BMSP_ERR_IO; return; } s = qq;
            double x = 1.0;
            if (!pattern) { x = strtod(s, &qq); if (qq == s) { P.err = BMSP_ERR_IO; return; } s = qq; }
            if (i < 1 || i > nr || j < 1 || j > nc) { P.err = BMSP_ERR_RANGE; return; }
            P.lines++;
            P.r.push_back((int32_t)(i - 1)); P.c.push_back((int32_t)(j - 1)); P.v.push_back(x);
            if ((symmetric || skew) && i != j) { P.r.push_back((int32_t)(j - 1)); P.c.push_back((int32_t)(i - 1)); P.v.push_back(skew ? -x : x); }
            while (s < e && *s != '\n') s++;
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 1; t < nth; t++) th.emplace_back(parse, t);
        parse(0);
        for (auto& t : th) t.join();
    }
    size_t total = 0; long long lines = 0;
    for (auto& P : parts) {
        if (P.err == BMSP_ERR_RANGE) { set_error("%s: index outside the %ld x %ld matrix", path, nr, nc); return BMSP_ERR_RANGE; }
        if (P.err) { set_error("%s: malformed entry line", path); return BMSP_ERR_IO; }
        total += P.r.size(); lines += P.lines;
    }
    std::vector<int32_t> r(total), c(total); std::vector<double> v(total);
    size_t w = 0;
    for (auto& P : parts) {
        std::copy(P.r.begin(), P.r.end(), r.begin() + w); std::copy(P.c.begin(), P.c.end(), c.begin() + w); std::copy(P.v.begin(), P.v.end(), v.begin() + w);
        w += P.r.size();
    }
    if (lines != nl) { set_error("%s: %lld entry lines, the size line announces %lld", path, lines, nl); return BMSP_ERR_IO; }
    return coo_to_matrix((int32_t)nr, (int32_t)nc, (int64_t)total, r.data(), c.data(), v.data(), transposed, out_dtype, flags, stream, out);
}

int bmsp_create_from_mtx(const char* path, int32_t transposed, int32_t out_dtype, void* stream, bmsp_matrix_t* out) {
    return bmsp_create_from_mtx_ex(path, transposed, out_dtype, 0, stream, out);
}

int bmsp_block_transpose(bmsp_matrix_t A, int32_t out_dtype, void* stream, bmsp_matrix_t* At) {
    if (!A || !At || (out_dtype != BMSP_F16 && out_dtype != BMSP_F32)) { set_error("bmsp_block_transpose: invalid argument"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    HandlePtr m;
    BMSP_TRY(new_handle(A->rows, A->cols, A->nblk, A->nnz, out_dtype, !A->transposed, st, m));
    m->offsets_len = A->offsets_len;
    if (m->nblk) {
        BMSP_CUDA(cudaMemcpyAsync(m->keys, A->keys, sizeof(uint64_t) * m->nblk, cudaMemcpyDeviceToDevice, st));
        BMSP_CUDA(cudaMemcpyAsync(m->offsets, A->offsets, sizeof(uint64_t) * m->offsets_len, cudaMemcpyDeviceToDevice, st));
        const unsigned grid = (unsigned)ceil_div(m->nblk, 128);
        BMSP_TRY(with_value_type(A->dtype, [&](auto in) { return with_value_type(out_dtype, [&](auto out) -> int {
            using Tin = decltype(in); using Tout = decltype(out);
            block_transpose_kernel<Tin, Tout><<<grid, 128, 0, st>>>(A->bmps, A->offsets, (const Tin*)A->values, m->bmps, (Tout*)m->values, m->nblk);
            BMSP_KERNEL_CHECK();
            return BMSP_OK;
        }); }));
    }
    BMSP_TRY(derive_compact(m.get(), st));
    *At = m.release();
    return BMSP_OK;
}

// A^T: the block order (transpose_block_order), then keys / bitmaps / value counts per block, the offsets by a scan, the values,
// the derived arrays.  Every step is enqueued on st; nothing is read back.
int bmsp_matrix_transpose(bmsp_matrix_t A, int32_t out_dtype, int32_t out_transposed, void* stream, bmsp_matrix_t* At) {
    if (!A || !At || (out_dtype != BMSP_F16 && out_dtype != BMSP_F32)) { set_error("bmsp_matrix_transpose: invalid argument"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    HandlePtr m;
    BMSP_TRY(new_handle(A->cols, A->rows, A->nblk, A->nnz, out_dtype, out_transposed ? 1 : 0, st, m));
    m->offsets_len = A->offsets_len;
    const int flip = (A->transposed != 0) == (out_transposed != 0);     // same form: the cells of a block move, so the bitmap does
    {
        DevBuf<uint32_t> kbuf[2], vbuf[2];
        const uint32_t* src = nullptr;
        BMSP_TRY(transpose_block_order(A, st, kbuf, vbuf, &src));
        const unsigned grid = (unsigned)ceil_div(m->nblk, 256);
        if (m->nblk) {
            transpose_blocks_kernel<<<grid, 256, 0, st>>>(A->keys, A->bmps, src, m->nblk, flip, m->keys, m->bmps, m->offsets);
            BMSP_KERNEL_CHECK();
        }
        BMSP_TRY(exclusive_scan_u64(m->offsets, m->offsets, m->nblk, st));       // offsets[nblk] = nnz, kept when offsets_len says so
        if (m->nblk) {
            BMSP_TRY(with_value_type(A->dtype, [&](auto in) { return with_value_type(out_dtype, [&](auto out) -> int {
                using Tin = decltype(in); using Tout = decltype(out);
                transpose_values_kernel<Tin, Tout><<<grid, 256, 0, st>>>(A->bmps, A->offsets, (const Tin*)A->values, src, m->nblk, flip,
                                                                         m->offsets, (Tout*)m->values);
                BMSP_KERNEL_CHECK();
                return BMSP_OK;
            }); }));
        }
    }
    BMSP_TRY(derive_compact(m.get(), st));
    *At = m.release();
    return BMSP_OK;
}

}  // extern "C"
