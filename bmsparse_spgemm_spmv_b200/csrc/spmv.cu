// spmv.cu -- y = A x on the bmSparse form, HBM-streaming, no tensor cores.
//
// Replaces bmSparse_SpMV / spmv_kernel (src/bmSparse_SPMV.cu:153-230).  The reference rebuilds the
// block-row pointers with reduce_by_key + scan on every call (:196-206), runs one 64-thread CTA per
// block row with thread <-> cell and re-reads key/bitmap/offset (24 B) from all 64 threads per block.
// Here the matrix is streamed exactly once through the compact surface (8 B bitmap + 4 B block column
// per block, 2 B per value, 8 B per block row):
//
//   path 0 "row-tiled"  (dense-ish blocks: Poisson, block-clustered)
//       one CTA per tile of 64 (32, 16 for heavy rows) block rows.  A per-matrix tile plan lists, for every tile, the
//       distinct 32-column lines of x its blocks touch and gives every block a 16-bit offset into the tile's staged
//       copy of those lines.  The tile's bitmaps / x offsets / values / row pointers are bulk-copied (cp.async.bulk +
//       mbarrier, SASS UBLKCP) into shared memory while all threads gather the x lines with coalesced 16-byte loads;
//       12+ CTAs are resident per SM, each in a different phase, which is what hides the copy latency.  Two threads
//       per block row, one per 32-bit bitmap half (4 matrix rows, 4 fp32 accumulators): each walks the blocks of its
//       block row, ranks with popc, and consumes set bits two rows at a time in predicated rounds (one PTX block per
//       row pair, no branches except the early exit); every per-value read (fp16 value, fp32 x) is a shared-memory
//       load; y is stored as one float4 per thread.  Tiles that exceed the shared-memory capacities are read from
//       global memory by the same threads.
//   path 1 "block-parallel" (about one value per block: uniform random, R-MAT)
//       one warp per work item (a block row, or a 512-block slice of a long one); lane <-> block, 4 x 32 blocks per step,
//       coalesced 8 B + 4 B metadata loads, value offsets by a warp scan of popc, eight per-row partial
//       sums per lane kept in shared memory, shuffle reduction at the end; sliced rows are finished by
//       a deterministic fix-up kernel.
#include "common.cuh"
#include <cstdlib>
#include <algorithm>
#include <vector>
#include <cstring>
#include <utility>
#include <type_traits>

namespace bmsp {

constexpr int SLICE = 512;         // blocks per work item (path 1): 4 steps of 128 blocks; longer block rows are sliced and summed by the fix-up

template <typename X> __device__ __forceinline__ float ld_xp(const X* p);
template <> __device__ __forceinline__ float ld_xp<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld_xp<__half>(const __half* p) { return __half2float(__ldg(p)); }
template <typename X> __device__ __forceinline__ float ld_x(const X* x, uint32_t i);
template <> __device__ __forceinline__ float ld_x<float>(const float* x, uint32_t i) { return __ldg(x + i); }
template <> __device__ __forceinline__ float ld_x<__half>(const __half* x, uint32_t i) { return __half2float(__ldg(x + i)); }

// One 8-bit row mask, MSB-aligned in `t` (column 0 = bit 31): walk its set bits in column order; the
// values are consecutive from vp.  xq points 24 elements before the block's x segment so that the
// leading-zero count of the right-aligned form indexes it directly.
template <typename T, typename X>
__device__ __forceinline__ void row_bits(uint32_t t, const T*& vp, const X* __restrict__ xs, float& acc) {
    while (t) {
        uint32_t c;                                      // column = leading zeros (FLO.U32.SH)
        asm("bfind.shiftamt.u32 %0, %1;" : "=r"(c) : "r"(t));
        const X* px;                                     // xs + c in one IMAD.WIDE
        asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(px) : "r"(c), "n"(sizeof(X)), "l"(xs));
        acc = fmaf(val_to_f32(*vp), ld_xp<X>(px), acc);
        vp++;
        t ^= 0x80000000u >> c;
    }
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// The blocks [pb, pe) of one block row, seen by the thread that owns bitmap half `h` (rows 4h..4h+3).
// bm / bc / vals are indexed relative to the tile's aligned bases (shared memory for staged tiles).
template <typename T, typename X>
__device__ __forceinline__ void half_block_row(const uint64_t* __restrict__ bm, const int32_t* __restrict__ bc,
                                               const T* __restrict__ vals, int pb, int pe, uint32_t k, const int h,
                                               const X* __restrict__ x, float (&acc)[4]) {
    if (pb < pe) prefetch_l1(x + (uint32_t)bc[pb] * 8u + 4u * h);
    for (int b = pb; b < pe; b++) {
        const uint2 w2 = *reinterpret_cast<const uint2*>(bm + b);     // .y = rows 0-3, .x = rows 4-7
        const uint32_t nhi = __popc(w2.y), nlo = __popc(w2.x);
        const uint32_t w = h ? w2.x : w2.y;
        const T* vp = vals + (k + (h ? nhi : 0u));
        k += nhi + nlo;
        // the next block's x segment is touched one block ahead: its L2 latency hides behind this block
        if (b + 1 < pe) prefetch_l1(x + (uint32_t)bc[b + 1] * 8u + 4u * h);
        if (w) {
            const X* xs = x + (uint32_t)bc[b] * 8u;
            row_bits<T, X>(w & 0xFF000000u, vp, xs, acc[0]);
            row_bits<T, X>((w << 8) & 0xFF000000u, vp, xs, acc[1]);
            row_bits<T, X>((w << 16) & 0xFF000000u, vp, xs, acc[2]);
            row_bits<T, X>(w << 24, vp, xs, acc[3]);
        }
    }
}

// ---- explicit 32-bit shared addresses (no generic-pointer arithmetic) ----
__device__ __forceinline__ uint2 lds_v2(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// ===================================================================================== path 0, tile plan
// Built once per matrix (plan_spmv): for every tile of RT block rows, the sorted distinct x "lines" (32 columns
// = 4 block columns = 128 B of fp32 x) its blocks touch, and per block a 16-bit offset of its 8-column x segment
// inside the tile's staged copy of those lines.  The kernel then never reads block_col: it streams bitmaps
// (8 B), x offsets (2 B) and values per block, gathers each distinct x line ONCE per tile with coalesced
// 16-byte loads (8 threads per line) and serves every per-value x read from shared memory.  Staged lines
// have a pitch of 33 elements: when the 16 block rows of a warp read the same column of consecutive block
// columns (stencils, bands) the 16 addresses fall into 16 different banks.
constexpr int XL_STRIDE = 33;      // staged x line pitch, elements (32 + 1 skew)
constexpr int PLAN_MAXB = 2048;    // blocks per tile the planner sorts in shared memory
constexpr int XL_MAX = 1900;       // distinct lines per tile (16-bit element offsets)

// 64 bytes; [lmin, lmax] = x lines touched.  The distinct lines of a stencil / band / cluster tile form a few runs of consecutive
// lines: up to three runs (first line, line count) are kept in the descriptor so that the streaming kernel can fetch the tile's
// x with one bulk copy per run without reading the line list (nruns = 0: more than three runs, copy line by line).
struct __align__(16) TileDesc { int32_t p0, nb; uint32_t v0; int32_t nv, nl, flags, lmin, lmax; int32_t nruns; uint32_t run_line[3], run_count[3]; int32_t pad; };
static_assert(sizeof(TileDesc) == 64, "TileDesc is four 16-byte words");

// ---- bitmap palette (streaming kernel) ----
// A stencil or banded matrix has a handful of distinct bitmaps among millions of blocks (P4096: 4).  When a matrix has at most
// PALETTE_MAX of them, the streaming kernel does not stream bitmaps (8 B per block), x offsets (2 B) and row pointers (8 B per block
// row): it streams one 32-bit word per block -- the x offset and the byte offset of the block's palette entry -- and one u16 pair
// per block row relative to its tile, and keeps the palette in shared memory.  An entry holds, per 32-bit bitmap half (rows 4h ..
// 4h+3), the half itself and what the consumer would otherwise derive from it for every block: the value offsets and the shape.
constexpr int PALETTE_MAX = 256;
constexpr int PAL_SLOTS = 1024, PAL_GSLOTS = 2048;   // open-addressing tables: per CTA (shared) and per matrix (global)
// entry = {half 0 bits, half 0 meta, half 1 bits, half 1 meta}; meta = value offset of the half * sizeof(T) (bits 0-7) | shape, one bit
// each (bits 8-11, none: empty half) | PAL_SINGLE: 8 * row + column of the cell (bits 12-16) | values of the block * sizeof(T) (bits 20-31).
// One-hot shapes are tested one bit at a time; a small integer would be compiled into an indirect jump.
enum : uint32_t { PAL_DIAG = 1u << 8, PAL_TRI = 1u << 9, PAL_SINGLE = 1u << 10, PAL_GENERIC = 1u << 11 };
struct PalScan { unsigned long long key[PAL_GSLOTS]; uint32_t count, has_zero, overflow, pad; };

__device__ __forceinline__ uint32_t pal_hash(uint64_t b, int bits) { return (uint32_t)((b * 0x9E3779B97F4A7C15ull) >> (64 - bits)); }
// insert the non-zero key b: 1 = inserted, 0 = already present, -1 = table full; *at = its slot
__device__ __forceinline__ int pal_insert(unsigned long long* tab, int bits, uint64_t b, uint32_t* at = nullptr) {
    const uint32_t mask = (1u << bits) - 1u;
    uint32_t i = pal_hash(b, bits);
    for (uint32_t n = 0; n <= mask; n++, i = (i + 1u) & mask) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(tab + i);
        if (at) *at = i;
        if (cur == b) return 0;
        if (cur == 0ull) {
            cur = atomicCAS(tab + i, 0ull, (unsigned long long)b);
            if (cur == 0ull) return 1;
            if (cur == b) return 0;
        }
    }
    return -1;
}

// One pass over the bitmaps: every CTA collects its distinct bitmaps in shared memory, then merges them into the global table.  Gives up
// (overflow) as soon as any table holds more than PALETTE_MAX; the order of the table is irrelevant (the host sorts the bitmaps).
__global__ void __launch_bounds__(256) palette_scan_kernel(const uint64_t* __restrict__ bmps, int64_t nblk, PalScan* __restrict__ ps) {
    __shared__ unsigned long long s_tab[PAL_SLOTS];
    __shared__ uint32_t s_cnt, s_zero, s_over;
    const int tid = threadIdx.x;
    for (int i = tid; i < PAL_SLOTS; i += 256) s_tab[i] = 0ull;
    if (tid == 0) { s_cnt = 0; s_zero = 0; s_over = 0; }
    __syncthreads();
    // a thread inserts at most one bitmap between two looks at the count: the table never holds more than PALETTE_MAX + 256 < PAL_SLOTS
    uint32_t it = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + tid; i < nblk; i += (int64_t)gridDim.x * 256, it++) {
        if (*reinterpret_cast<volatile uint32_t*>(&s_cnt) > (uint32_t)PALETTE_MAX) break;
        if ((it & 15u) == 0 && *reinterpret_cast<volatile uint32_t*>(&ps->overflow)) break;
        const uint64_t b = ld_stream_u64(bmps + i);
        if (b == 0ull) { s_zero = 1; continue; }
        const int r = pal_insert(s_tab, 10, b);
        if (r > 0) atomicAdd(&s_cnt, 1u);
        else if (r < 0) { s_over = 1; break; }
    }
    __syncthreads();
    if (s_over || s_cnt > (uint32_t)PALETTE_MAX) { if (tid == 0) atomicExch(&ps->overflow, 1u); return; }
    if (tid == 0 && s_zero) ps->has_zero = 1;
    for (int j = tid; j < PAL_SLOTS; j += 256) {
        const uint64_t b = s_tab[j];
        if (b == 0ull) continue;
        if (*reinterpret_cast<volatile uint32_t*>(&ps->overflow)) break;
        const int r = pal_insert(ps->key, 11, b);
        if (r < 0 || (r > 0 && atomicAdd(&ps->count, 1u) >= (uint32_t)PALETTE_MAX)) { atomicExch(&ps->overflow, 1u); break; }
    }
}

// pal / npal: the sorted palette (streaming kernel with a palette: per block `word`, per block row `rowrel`; otherwise `xoff`)
__global__ void __launch_bounds__(256) tile_plan_kernel(const int32_t* __restrict__ brp, const int32_t* __restrict__ bcol,
                                                        const uint32_t* __restrict__ rvb, int nbr, int ncols, int rt, int pitch, TileDesc* __restrict__ desc,
                                                        uint32_t* __restrict__ lines, uint16_t* __restrict__ xoff,
                                                        unsigned long long* __restrict__ stats, const uint64_t* __restrict__ bmps,
                                                        const uint4* __restrict__ pal, int npal, uint32_t* __restrict__ word,
                                                        uint32_t* __restrict__ rowrel) {
    __shared__ uint32_t s_key[PLAN_MAXB];
    __shared__ uint32_t s_uniq[PLAN_MAXB];
    __shared__ uint64_t s_pal[PALETTE_MAX];
    const int t = blockIdx.x, tid = threadIdx.x;
    const int r0 = t * rt, r1 = min(r0 + rt, nbr);
    const int p0 = brp[r0], nb = brp[r1] - p0;
    const uint32_t v0 = rvb[r0], v1 = rvb[r1];
    if (word) {
        // tile-relative row pairs: read for staged tiles only, whose block and value counts are far below 65536 (shared memory)
        for (int r = r0 + tid; r < r1; r += 256) rowrel[r] = (uint32_t)(brp[r] - p0) | ((rvb[r] - v0) << 16);
        for (int i = tid; i < npal; i += 256) s_pal[i] = (uint64_t)pal[i].x << 32 | pal[i].z;
    }
    TileDesc d;
    d.p0 = p0; d.nb = nb; d.v0 = v0; d.nv = (int32_t)(v1 - v0); d.nl = 0; d.flags = 0; d.lmin = 0; d.lmax = nb > 0 ? 0x7FFFFFFF : -1;
    d.nruns = 0; d.pad = 0;
    for (int k = 0; k < 3; k++) { d.run_line[k] = 0; d.run_count[k] = 0; }
    if (nb > PLAN_MAXB) {          // too many blocks to plan: the kernel reads this tile straight from global memory
        if (tid == 0) { desc[t] = d; atomicAdd(stats + 4, 1ull); }
        return;
    }
    int n2 = 32;
    while (n2 < nb) n2 <<= 1;
    for (int i = tid; i < n2; i += 256) s_key[i] = i < nb ? ((uint32_t)bcol[p0 + i] >> 2) : 0xFFFFFFFFu;
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < n2; i += 256) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint32_t a = s_key[i], b = s_key[ixj];
                    if ((a > b) == ((i & k) == 0)) { s_key[i] = b; s_key[ixj] = a; }
                }
            }
            __syncthreads();
        }
    // distinct keys, order kept: thread t owns `per` consecutive sorted slots
    const int per = n2 >= 256 ? n2 / 256 : 1;
    const int i0 = tid * per, i1 = min(i0 + per, nb);
    uint32_t cnt = 0;
    for (int i = i0; i < i1; i++) cnt += (i == 0 || s_key[i] != s_key[i - 1]) ? 1u : 0u;
    uint32_t total;
    uint32_t run = cta_exclusive_scan(cnt, &total);
    for (int i = i0; i < i1; i++)
        if (i == 0 || s_key[i] != s_key[i - 1]) s_uniq[run++] = s_key[i];
    const int nl = (int)total;
    __syncthreads();
    for (int j = tid; j < nl; j += 256) lines[p0 + j] = s_uniq[j];
    const bool ok = nl <= XL_MAX;
    if (ok)
        for (int i = tid; i < nb; i += 256) {
            const uint32_t c = (uint32_t)bcol[p0 + i];
            const int lo = lower_bound(s_uniq, 0, nl, c >> 2);
            const uint32_t xo = (uint32_t)(lo * pitch + (int)(c & 3u) * 8);
            if (word) {
                const int pl = lower_bound(s_pal, 0, npal, bmps[p0 + i]);
                word[p0 + i] = xo | (uint32_t)pl << 20;              // entry byte offset (16 * code) in bits 16-31
            } else {
                xoff[p0 + i] = (uint16_t)xo;
            }
        }
    if (tid == 0) {
        // flags: bit 0 = planned (x offsets valid), bit 1 = the last line reaches past the last column (guarded gather)
        if (nb > 0) { d.lmin = (int32_t)s_uniq[0]; d.lmax = (int32_t)s_uniq[nl - 1]; }
        d.nl = nl; d.flags = (ok ? 1 : 0) | ((nl > 0 && (uint64_t)s_uniq[nl - 1] * 32u + 32u > (uint64_t)ncols) ? 2 : 0);
        // runs of consecutive lines (at most three are kept; a fourth makes the tile a line-by-line one)
        int nruns = 0;
        for (int j = 0; j < nl && nruns <= 3; j++) {
            if (j == 0 || s_uniq[j] != s_uniq[j - 1] + 1u) { if (nruns < 3) { d.run_line[nruns] = s_uniq[j]; d.run_count[nruns] = 0; } nruns++; }
            if (nruns <= 3) d.run_count[nruns - 1]++;
        }
        d.nruns = nruns <= 3 ? nruns : 0;
        desc[t] = d;
        atomicMax(stats + 0, (unsigned long long)nb);
        atomicMax(stats + 1, (unsigned long long)(v1 - v0));
        atomicMax(stats + 2, (unsigned long long)nl);
        atomicAdd(stats + 3, (unsigned long long)nl);
        if (!ok) atomicAdd(stats + 4, 1ull);
    }
}

// ---- row shapes (streaming kernel with a palette) ----
// On a stencil or band matrix the block words of a block row repeat from row to row once the x offset is taken relative to the row:
// a block column c of block row lbr in a tile whose lines are consecutive sits at x offset 8 c - 32 (first line), so xo - 8 lbr is
// the same for every interior row (P4096: 14 distinct rows in all 32 768 tiles).  When the staged rows of a matrix have at most
// SHAPE_MAX distinct such sequences ("shapes"), the streaming kernel keeps them in one table in shared memory next to the palette
// and streams no block words: a row's 4-byte word names its shape instead of its first block.
//   shape word  = x offset - 8 lbr + SHAPE_BIAS (bits 0-15) | palette entry byte offset (bits 16-31), as in `word`.  The bias keeps
//                 the field positive: a row can touch a line that lies before the lines of the tile's earlier rows (xo < 8 lbr), and
//                 xo + SHAPE_BIAS - 8 lbr lies in [8, 61304] for every planned tile (xo < XL_MAX * 32, lbr < 64).
//   row word    = shape's first word in the table (bits 0-10) | its block count (bits 11-15) | first value relative to the tile
//                 (bits 16-31, as in `rowrel`).  An empty row is {0, 0}.
// The consumer moves its staged-x base by (8 lbr - SHAPE_BIAS) elements and walks the shape with tile_half_row_pal unchanged.
constexpr int SHAPE_MAX = 128;         // distinct shapes per matrix
constexpr int SHAPE_NB = 31;           // blocks per shape (5-bit count)
constexpr int SHAPE_WORDS = 1024;      // words in the table (4 KB of shared memory per CTA at most)
constexpr uint32_t SHAPE_BIAS = 512;   // > 8 * (STREAM_RT - 1)
constexpr int SHP_SLOTS = 512, SHP_GSLOTS = 1024;   // open-addressing tables of row hashes: per CTA (shared) and per matrix (global)
struct ShapeScan { unsigned long long key[SHP_GSLOTS]; uint32_t rep[SHP_GSLOTS]; uint32_t count, overflow, nout, pad; };

__device__ __forceinline__ uint32_t shape_word(uint32_t w, int lbr) { return (w & 0xFFFF0000u) | ((w & 0xFFFFu) + SHAPE_BIAS - 8u * (uint32_t)lbr); }
__device__ __forceinline__ unsigned long long shape_hash(const uint32_t* __restrict__ w, int nb, int lbr) {
    unsigned long long h = 0x243F6A8885A308D3ull ^ (uint32_t)nb;
    for (int i = 0; i < nb; i++) { h = (h ^ shape_word(__ldg(w + i), lbr)) * 0x9E3779B97F4A7C15ull; h ^= h >> 29; }
    return h | 1ull;
}
// the rows of a tile the streaming kernel stages (the test of its producer); the others read brp / bcol / bmps from global memory
__device__ __forceinline__ bool shape_row_staged(const TileDesc* __restrict__ desc, int r, int cb, int cv, int cl) {
    const int4 d0 = __ldg(reinterpret_cast<const int4*>(desc + r / 64)), d1 = __ldg(reinterpret_cast<const int4*>(desc + r / 64) + 1);
    return (d1.y & 1) && d0.y <= cb && d0.w <= cv && d1.x <= cl;
}

// One pass over the staged block rows: every CTA collects the hashes of its distinct non-empty shapes (and one row of each) in
// shared memory, then merges them into the global table; gives up (overflow) as soon as a table holds more than SHAPE_MAX or a row
// has more than SHAPE_NB blocks.  Two shapes with one hash become one entry here: shape_assign_kernel compares every row's words.
__global__ void __launch_bounds__(256) shape_scan_kernel(const int32_t* __restrict__ brp, const uint32_t* __restrict__ word,
                                                         const TileDesc* __restrict__ desc, int nbr, int cb, int cv, int cl,
                                                         ShapeScan* __restrict__ ss) {
    __shared__ unsigned long long s_tab[SHP_SLOTS];
    __shared__ uint32_t s_rep[SHP_SLOTS];
    __shared__ uint32_t s_cnt, s_over;
    const int tid = threadIdx.x;
    for (int i = tid; i < SHP_SLOTS; i += 256) s_tab[i] = 0ull;
    if (tid == 0) { s_cnt = 0; s_over = 0; }
    __syncthreads();
    // as palette_scan_kernel: the table never holds more than SHAPE_MAX + 256 < SHP_SLOTS keys
    uint32_t it = 0;
    for (int r = blockIdx.x * 256 + tid; r < nbr; r += gridDim.x * 256, it++) {
        if (*reinterpret_cast<volatile uint32_t*>(&s_cnt) > (uint32_t)SHAPE_MAX) break;
        if ((it & 15u) == 0 && *reinterpret_cast<volatile uint32_t*>(&ss->overflow)) break;
        if (!shape_row_staged(desc, r, cb, cv, cl)) continue;
        const int p = __ldg(brp + r), nb = __ldg(brp + r + 1) - p;
        if (nb == 0) continue;
        if (nb > SHAPE_NB) { s_over = 1; break; }
        uint32_t at = 0;
        const int res = pal_insert(s_tab, 9, shape_hash(word + p, nb, r & 63), &at);
        if (res > 0) { s_rep[at] = (uint32_t)r; atomicAdd(&s_cnt, 1u); }
        else if (res < 0) { s_over = 1; break; }
    }
    __syncthreads();
    if (s_over || s_cnt > (uint32_t)SHAPE_MAX) { if (tid == 0) atomicExch(&ss->overflow, 1u); return; }
    for (int j = tid; j < SHP_SLOTS; j += 256) {
        const uint64_t k = s_tab[j];
        if (k == 0ull) continue;
        if (*reinterpret_cast<volatile uint32_t*>(&ss->overflow)) break;
        uint32_t at = 0;
        const int res = pal_insert(ss->key, 10, k, &at);
        if (res > 0) ss->rep[at] = s_rep[j];
        if (res < 0 || (res > 0 && atomicAdd(&ss->count, 1u) >= (uint32_t)SHAPE_MAX)) { atomicExch(&ss->overflow, 1u); break; }
    }
}

// the words of every shape, from the row the scan kept for it: out[k] = {global slot | block count << 16, words ...}
__global__ void shape_gather_kernel(const int32_t* __restrict__ brp, const uint32_t* __restrict__ word, ShapeScan* __restrict__ ss,
                                    uint32_t* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= SHP_GSLOTS || ss->overflow || ss->key[j] == 0ull) return;
    const uint32_t k = atomicAdd(&ss->nout, 1u);
    if (k >= (uint32_t)SHAPE_MAX) return;
    const int r = (int)ss->rep[j], p = brp[r], nb = brp[r + 1] - p;
    uint32_t* o = out + (size_t)k * (SHAPE_NB + 1);
    o[0] = (uint32_t)j | (uint32_t)nb << 16;
    for (int i = 0; i < nb; i++) o[1 + i] = shape_word(word[p + i], r & 63);
}

// Row words of the shape layout (into srow; rowrel stays as it is).  Exactness does not rest on the hash: every staged row's words
// are compared with the words of the shape its hash names, and any difference -- or a hash the table does not hold -- sets *bad,
// which keeps the matrix in the word layout.
__global__ void __launch_bounds__(256) shape_assign_kernel(const int32_t* __restrict__ brp, const uint32_t* __restrict__ word,
                                                           const uint32_t* __restrict__ rowrel, const TileDesc* __restrict__ desc,
                                                           int nbr, int cb, int cv, int cl, const unsigned long long* __restrict__ gkey,
                                                           const uint32_t* __restrict__ gval, const uint32_t* __restrict__ table,
                                                           uint32_t* __restrict__ srow, uint32_t* __restrict__ bad) {
    const int r = blockIdx.x * 256 + threadIdx.x;
    if (r >= nbr) return;
    uint32_t f = 0;
    if (shape_row_staged(desc, r, cb, cv, cl)) {
        const int p = __ldg(brp + r), nb = __ldg(brp + r + 1) - p;
        if (nb > SHAPE_NB) { atomicExch(bad, 1u); return; }
        if (nb > 0) {
            const unsigned long long k = shape_hash(word + p, nb, r & 63);
            uint32_t i = pal_hash(k, 10), n = 0;
            while (n < SHP_GSLOTS && gkey[i] != k && gkey[i] != 0ull) { i = (i + 1u) & (SHP_GSLOTS - 1); n++; }
            if (n == SHP_GSLOTS || gkey[i] != k) { atomicExch(bad, 1u); return; }
            f = gval[i];
            const uint32_t* s = table + (f & 0x7FFu);
            bool same = (int)(f >> 11) == nb;
            for (int b = 0; b < nb && same; b++) same = __ldg(s + b) == shape_word(__ldg(word + p + b), r & 63);
            if (!same) { atomicExch(bad, 1u); return; }
        }
    }
    srow[r] = f | (rowrel[r] & 0xFFFF0000u);
}

// shared-memory carve-up of spmv_tile_kernel (cap_blk and cap_val are multiples of 8); computed on the host
struct TileSmem { uint32_t xo, val, row, xs, bar, total; };
inline TileSmem tile_smem(int rt, int cap_blk, int cap_val, int cap_lines, int vsize, int xsize) {
    TileSmem s;
    s.xo = (uint32_t)(cap_blk + 2) * 8;
    s.val = s.xo + (uint32_t)(cap_blk + 16) * 2;
    s.row = s.val + (uint32_t)(cap_val + 16) * vsize;
    s.xs = s.row + (uint32_t)(rt + 2) * 8;
    s.bar = (s.xs + (uint32_t)cap_lines * XL_STRIDE * xsize + 15u) & ~15u;
    s.total = s.bar + 16;
    return s;
}

template <typename T>
struct TileArgs {
    const uint64_t* bmps; const int32_t* bcol; const T* values; const int2* rowpair;   // rowpair[r] = (block_row_ptr[r], first value of row r)
    const TileDesc* desc; const uint32_t* lines; const uint16_t* xoff;
    const uint32_t* word; const uint32_t* rowrel; const uint4* palette; int32_t npal;   // streaming kernel with a palette (tile_plan_kernel)
    int32_t shape_words;                                                                 // ... and row shapes: table words behind the palette
    const int32_t* brp; const uint32_t* rvb;                                             // ... whose unstaged tiles read their row pointers here
    int32_t rows, nbr, cols, cap_blk, cap_val, cap_lines;
    int32_t tile0;       // first tile of this launch (row-range launches of the host-buffer pipeline)
    TileSmem so;
};

__global__ void zip_rows_kernel(const int32_t* __restrict__ brp, const uint32_t* __restrict__ rvb, int n, int2* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_int2(brp[i], (int)rvb[i]);
}

__device__ __forceinline__ uint32_t lds_u16(uint32_t a) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return v;
}

// Two 8-bit row masks b0, b1 of one bitmap half (left in place: row r of the half occupies bits 31-8r..24-8r)
// advance together: every round takes the highest set bit p of each mask, multiplies the row's next value
// (shared address va + round * sizeof(T)) with x[column] (shared address xb - p * sizeof(X) - 8 r sizeof(X),
// the row term folded into the load's immediate) and clears the bit.  The whole walk is one PTX block so that
// the predicates stay in predicate registers from round to round: per value FLO, IMAD, 2 LDS, BMSK, LOP3,
// (cvt,) FFMA, and no branch other than the early exit once both masks are empty.  Value loads are not
// predicated (their addresses stay inside the staged tile), x loads and the FMAs are.
#define BMSP_RND(OFF, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)                                        \
    "bfind.u32 p0, %2;\n\tbfind.u32 p1, %3;\n\t"                                                          \
    "mad.lo.s32 a0, p0, " XMUL ", %6;\n\tmad.lo.s32 a1, p1, " XMUL ", %6;\n\t"                            \
    VLD "0, [%4+" #OFF "];\n\t" VLD "1, [%5+" #OFF "];\n\t"                                               \
    "@q0 " XLD "0, [a0+" XA "];\n\t@q1 " XLD "1, [a1+" XB "];\n\t"                                        \
    "bmsk.clamp.b32 m0, p0, 1;\n\tbmsk.clamp.b32 m1, p1, 1;\n\t" VC0 VC1 XC0 XC1                          \
    "@q0 fma.rn.f32 %0, f0, x0, %0;\n\t@q1 fma.rn.f32 %1, f1, x1, %1;\n\t"                                \
    "not.b32 m0, m0;\n\tnot.b32 m1, m1;\n\tand.b32 %2, %2, m0;\n\tand.b32 %3, %3, m1;\n\t"                \
    "setp.ne.u32 q0, %2, 0;\n\tsetp.ne.u32 q1, %3, 0;\n\tor.pred qa, q0, q1;\n\t@!qa bra DONE;\n\t"
#define BMSP_PAIR(O0, O1, O2, O3, O4, O5, O6, O7, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)            \
    asm("{\n\t.reg .pred q0, q1, qa;\n\t.reg .u32 p0, p1, m0, m1, a0, a1, h0, h1, g0, g1;\n\t"            \
        ".reg .f32 x0, x1, f0, f1;\n\t.reg .b16 lo, hi;\n\t"                                              \
        "setp.ne.u32 q0, %2, 0;\n\tsetp.ne.u32 q1, %3, 0;\n\tor.pred qa, q0, q1;\n\t@!qa bra DONE;\n\t"   \
        BMSP_RND(O0, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB) BMSP_RND(O1, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)  \
        BMSP_RND(O2, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB) BMSP_RND(O3, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)  \
        BMSP_RND(O4, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB) BMSP_RND(O5, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)  \
        BMSP_RND(O6, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB) BMSP_RND(O7, VLD, VC0, VC1, XLD, XC0, XC1, XMUL, XA, XB)  \
        "DONE:\n\t}"                                                                                      \
        : "+f"(acc0), "+f"(acc1), "+r"(b0), "+r"(b1) : "r"(va0), "r"(va1), "r"(xb))
#define BMSP_CVT16(dst, src) "mov.b32 {lo, hi}, " src ";\n\tcvt.f32.f16 " dst ", lo;\n\t"
// PAIR 0: rows 0,1 of the half (x immediates 0 and -8 columns); PAIR 1: rows 2,3 (-16 and -24 columns)
template <typename T, typename X, int PAIR> struct RowPair;
#define BMSP_ROWPAIR(TT, XX, PP, ...)                                                                                             \
    template <> struct RowPair<TT, XX, PP> {                                                                                      \
        static __device__ __forceinline__ void run(float& acc0, float& acc1, uint32_t b0, uint32_t b1, uint32_t va0, uint32_t va1, \
                                                   uint32_t xb) {                                                                 \
            BMSP_PAIR(__VA_ARGS__);                                                                                               \
        }                                                                                                                         \
    };
#define BMSP_V16 0, 2, 4, 6, 8, 10, 12, 14, "ld.shared.u16 h", BMSP_CVT16("f0", "h0"), BMSP_CVT16("f1", "h1")
#define BMSP_V32 0, 4, 8, 12, 16, 20, 24, 28, "ld.shared.f32 f", "", ""
#define BMSP_X32 "ld.shared.f32 x", "", "", "-4"
#define BMSP_X16 "ld.shared.u16 g", BMSP_CVT16("x0", "g0"), BMSP_CVT16("x1", "g1"), "-2"
BMSP_ROWPAIR(__half, float, 0, BMSP_V16, BMSP_X32, "0", "-32")
BMSP_ROWPAIR(__half, float, 1, BMSP_V16, BMSP_X32, "-64", "-96")
BMSP_ROWPAIR(__half, __half, 0, BMSP_V16, BMSP_X16, "0", "-16")
BMSP_ROWPAIR(__half, __half, 1, BMSP_V16, BMSP_X16, "-32", "-48")
BMSP_ROWPAIR(float, float, 0, BMSP_V32, BMSP_X32, "0", "-32")
BMSP_ROWPAIR(float, float, 1, BMSP_V32, BMSP_X32, "-64", "-96")
BMSP_ROWPAIR(float, __half, 0, BMSP_V32, BMSP_X16, "0", "-16")
BMSP_ROWPAIR(float, __half, 1, BMSP_V32, BMSP_X16, "-32", "-48")
#undef BMSP_RND
#undef BMSP_PAIR
#undef BMSP_CVT16
#undef BMSP_ROWPAIR
#undef BMSP_V16
#undef BMSP_V32
#undef BMSP_X32
#undef BMSP_X16

template <typename V> __device__ __forceinline__ float lds_as_f32(uint32_t a);
template <> __device__ __forceinline__ float lds_as_f32<float>(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
template <> __device__ __forceinline__ float lds_as_f32<__half>(uint32_t a) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return __half2float(__ushort_as_half(v));
}

// The blocks of one block row seen by the thread that owns bitmap half h (rows 4h..4h+3).  Everything lives in
// shared memory: bitmaps at a_bm, 16-bit x offsets at a_xo, the row's values from a_v on; xs31 = staged x + 31
// elements.
template <typename X> __device__ __forceinline__ void lds_x4(uint32_t a, float (&o)[4]);
template <> __device__ __forceinline__ void lds_x4<float>(uint32_t a, float (&o)[4]) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]) : "r"(a));
}
template <> __device__ __forceinline__ void lds_x4<__half>(uint32_t a, float (&o)[4]) {
    uint32_t lo, hi;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(a));
    const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&lo)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    o[0] = f0.x; o[1] = f0.y; o[2] = f1.x; o[3] = f1.y;
}

// The four shapes of one bitmap half, each on its half's values from va0 on and its 8-column x segment at element offset xo of the
// staged lines (xs31 = staged x + 31 elements).
// XV: the staged x lines are dense (pitch 32) and 16-byte aligned, so the four x elements of a bitmap half are one vector load
template <typename T, typename X, bool XV>
__device__ __forceinline__ void half_diag(uint32_t va0, uint32_t xo, const int h, const uint32_t xs31, float (&acc)[4]) {
    // diagonal block (the +-m neighbours of a stencil, any band at a multiple of 8): row i of the half holds exactly
    // column 4h + i -- four straight multiply-adds, no bit walk (20 instructions instead of ~50)
    constexpr uint32_t SV = sizeof(T), SX = sizeof(X);
    const uint32_t xa = xs31 - 31u * SX + (xo + 4u * (uint32_t)h) * SX;
    float x4[4];
    if constexpr (XV) lds_x4<X>(xa, x4);
    else {
#pragma unroll
        for (int i = 0; i < 4; i++) x4[i] = lds_as_f32<X>(xa + i * SX);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) acc[i] = fmaf(lds_as_f32<T>(va0 + i * SV), x4[i], acc[i]);
}
template <typename T, typename X, bool XV>
__device__ __forceinline__ void half_tri(uint32_t va0, uint32_t xo, const int h, const uint32_t xs31, float (&acc)[4]) {
    // tridiagonal block (the diagonal block of a stencil, any 3-wide band): row i of the half holds columns
    // 4h+i-1 .. 4h+i+1, clipped to the block -- 11 values.  Written as 12 slots (3 per row) over the six x elements
    // 4h-1 .. 4h+4 so that the code does not depend on h: slot 0 of the upper half (column -1) and slot 11 of the
    // lower half (column 8) do not exist and are predicated off (their loads stay inside the staged tile).
    constexpr uint32_t SV = sizeof(T), SX = sizeof(X);
    const uint32_t vb = va0 + ((uint32_t)h - 1u) * SV;                       // slot s at vb + s * SV
    const uint32_t xa = xs31 - 31u * SX + (xo + 4u * (uint32_t)h - 1u) * SX;   // x[4h-1+j] at xa + j * SX
    float xl[6], v[12];
    if constexpr (XV) {
        float x4[4];
        lds_x4<X>(xa + SX, x4);
        xl[0] = lds_as_f32<X>(xa); xl[1] = x4[0]; xl[2] = x4[1]; xl[3] = x4[2]; xl[4] = x4[3]; xl[5] = lds_as_f32<X>(xa + 5 * SX);
    } else {
#pragma unroll
        for (int j = 0; j < 6; j++) xl[j] = lds_as_f32<X>(xa + j * SX);
    }
#pragma unroll
    for (int s = 0; s < 12; s++) v[s] = lds_as_f32<T>(vb + s * SV);
    if (h) acc[0] = fmaf(v[0], xl[0], acc[0]);
    acc[0] = fmaf(v[1], xl[1], acc[0]); acc[0] = fmaf(v[2], xl[2], acc[0]);
    acc[1] = fmaf(v[3], xl[1], acc[1]); acc[1] = fmaf(v[4], xl[2], acc[1]); acc[1] = fmaf(v[5], xl[3], acc[1]);
    acc[2] = fmaf(v[6], xl[2], acc[2]); acc[2] = fmaf(v[7], xl[3], acc[2]); acc[2] = fmaf(v[8], xl[4], acc[2]);
    acc[3] = fmaf(v[9], xl[3], acc[3]); acc[3] = fmaf(v[10], xl[4], acc[3]);
    if (!h) acc[3] = fmaf(v[11], xl[5], acc[3]);
}
template <typename T, typename X>
__device__ __forceinline__ void half_single(uint32_t va0, uint32_t xo, const uint32_t t, const uint32_t xs31, float (&acc)[4]) {
    // one value in this half, cell t = 8 * row + column (the +-1 neighbours of a stencil: a single cell in the whole block): one
    // product, added to the row it belongs to
    constexpr uint32_t SX = sizeof(X);
    const float prod = lds_as_f32<T>(va0) * lds_as_f32<X>(xs31 - 31u * SX + (xo + (t & 7u)) * SX);
    const uint32_t rr = t >> 3;
    acc[0] += rr == 0u ? prod : 0.f; acc[1] += rr == 1u ? prod : 0.f;
    acc[2] += rr == 2u ? prod : 0.f; acc[3] += rr == 3u ? prod : 0.f;
}
template <typename T, typename X>
__device__ __forceinline__ void half_generic(uint32_t w, uint32_t va0, uint32_t xo, const uint32_t xs31, float (&acc)[4]) {
    constexpr uint32_t SV = sizeof(T), SX = sizeof(X);
    const uint32_t xb = xs31 + xo * SX;
    const uint32_t b0 = w & 0xFF000000u, b1 = w & 0x00FF0000u, b2 = w & 0x0000FF00u, b3 = w & 0x000000FFu;
    const uint32_t va1 = va0 + __popc(b0) * SV, va2 = va1 + __popc(b1) * SV, va3 = va2 + __popc(b2) * SV;
    RowPair<T, X, 0>::run(acc[0], acc[1], b0, b1, va0, va1, xb);
    RowPair<T, X, 1>::run(acc[2], acc[3], b2, b3, va2, va3, xb);
}

// The blocks of one block row seen by the thread that owns bitmap half h (rows 4h..4h+3).  Everything lives in
// shared memory: bitmaps at a_bm, 16-bit x offsets at a_xo, the row's values from a_v on; xs31 = staged x + 31
// elements.
template <typename T, typename X, bool XV = false>
__device__ __forceinline__ void tile_half_row(uint32_t a_bm, uint32_t a_xo, uint32_t a_v, int nb, const int h, const uint32_t xs31,
                                              float (&acc)[4]) {
    constexpr uint32_t SV = sizeof(T);
    const uint32_t hm = 0u - (uint32_t)h;
#pragma unroll 1
    for (int i = 0; i < nb; i++) {
        const uint2 w2 = lds_v2(a_bm);                  // .y = rows 0-3, .x = rows 4-7
        const uint32_t xo = lds_u16(a_xo);
        a_bm += 8; a_xo += 2;
        const uint32_t nhi = __popc(w2.y), nlo = __popc(w2.x);
        const uint32_t w = (w2.x & hm) | (w2.y & ~hm);
        const uint32_t va0 = a_v + (nhi & hm) * SV;
        a_v += (nhi + nlo) * SV;
        if (w == (0x80402010u >> (4 * h))) half_diag<T, X, XV>(va0, xo, h, xs31, acc);
        else if (w == (h ? 0x1C0E0703u : 0xC0E07038u)) half_tri<T, X, XV>(va0, xo, h, xs31, acc);
        else if (w && !(w & (w - 1u))) half_single<T, X>(va0, xo, 31u - (uint32_t)(31 - __clz((int)w)), xs31, acc);
        else if (w) half_generic<T, X>(w, va0, xo, xs31, acc);
    }
}

// The same walk over a palette matrix: per block one 32-bit word (x offset | entry byte offset << 16) at a_w and the half's 8 bytes of
// the palette entry at pal_h + entry offset {bits, meta}: no popc and no shape tests, the entry says it all.  The products and their
// order per row are those of tile_half_row.
template <typename T, typename X>
__device__ __forceinline__ void tile_half_row_pal(uint32_t a_w, const uint32_t pal_h, uint32_t a_v, int nb, const int h, const uint32_t xs31,
                                                  float (&acc)[4]) {
#pragma unroll 1
    for (int i = 0; i < nb; i++) {
        const uint32_t wd = lds_u32(a_w);
        a_w += 4;
        const uint2 e = lds_v2(pal_h + (wd >> 16));
        const uint32_t xo = wd & 0xFFFFu, m = e.y;
        const uint32_t va0 = a_v + (m & 0xFFu);
        a_v += m >> 20;
        if (m & PAL_DIAG) half_diag<T, X, true>(va0, xo, h, xs31, acc);
        else if (m & PAL_TRI) half_tri<T, X, true>(va0, xo, h, xs31, acc);
        else if (m & PAL_SINGLE) half_single<T, X>(va0, xo, (m >> 12) & 31u, xs31, acc);
        else if (m & PAL_GENERIC) half_generic<T, X>(e.x, va0, xo, xs31, acc);
    }
}

template <typename X> __device__ __forceinline__ void sts_x(uint32_t a, X v);
template <> __device__ __forceinline__ void sts_x<float>(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
template <> __device__ __forceinline__ void sts_x<__half>(uint32_t a, __half v) {
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"(__half_as_ushort(v)) : "memory");
}
template <typename X> struct alignas(4 * sizeof(X)) XQuad { X e[4]; };

// ---- multi-GPU: halo exchange over peer memory (NVLink) fused into the product, SURVEY.md section 8e -------------
// Every rank keeps x for its extended column range in three peer-mapped buffers (rotating) plus an inbox of epoch
// flags, one slot per peer.  A product reads x[cur] (own slice + halo slices the peers pushed), writes y into the
// own slice of x[nxt] and -- in the same kernel -- stores the rows a peer needs straight into that peer's x[nxt]
// (P2P stores); the last pushing CTA then publishes `signal_epoch` in the peers' inboxes (st.release.sys after a
// system fence).  Only tiles whose x lines leave the rank's own columns wait (spin on the inbox until every peer's
// slot reached `wait_epoch`), and the tile order is rotated by half a grid so that these boundary tiles -- which
// are also the ones that push -- run mid-kernel: the peers' rows of the previous product arrived long before, and
// this product's rows are on their way long before the peers need them, so the exchange costs no time at all.
// Peers signal each other in both directions even when one direction carries no data.  Write-after-read: the
// buffer a peer overwrites during its product e was last read by my product e-2, which finished before my product
// e-1 (whose epoch the peer waited for) started -- hence three buffers.
constexpr int HALO_MAX = 8;
struct HaloDev {
    int32_t n_push, n_peer;
    int32_t lo[HALO_MAX], hi[HALO_MAX];      // local row ranges [lo, hi) pushed to a peer (lo a multiple of 4)
    float* dst[HALO_MAX];                    // peer address of row lo[i] (16-byte aligned)
    uint32_t* peer_flag[HALO_MAX];           // my slot in each peer's inbox
    const uint32_t* my_flag[HALO_MAX];       // the peers' slots in my inbox
    uint32_t* scratch;                       // [0] pushing CTAs that finished, [1] error: a wait timed out
    uint32_t wait_epoch, signal_epoch, n_sig;
    int32_t solo_tile;                       // tile that signals when no tile pushes anything (-1: none)
    int32_t n_iv, iv_lo[HALO_MAX], iv_hi[HALO_MAX];   // the tiles that own pushed rows, as disjoint tile intervals [lo, hi] (host-computed:
                                             // the streaming kernel's producer tests a tile against these instead of the row ranges)
    int32_t own_c0, own_c1;                  // columns [own_c0, own_c1) of x_ext are this rank's own slice: tiles that stay inside never wait
    int32_t rot;                             // tile order rotation: CTA b runs tile (b + rot) mod ntiles, so that the boundary tiles
                                             // (which need the peers' rows and produce the rows the peers need) run mid-kernel
};
struct NoHalo {};

__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// one thread per peer: spin until the peer's slot reached wait_epoch; gives up after 4 s (error flag, no hang)
__device__ __forceinline__ void halo_wait(const HaloDev& h, int i, bool full_fence = true) {
    const uint32_t* f = h.my_flag[i];
    if ((int32_t)(ld_relaxed_sys(f) - h.wait_epoch) < 0) {
        const uint64_t t0 = globaltimer_ns();
        while ((int32_t)(ld_relaxed_sys(f) - h.wait_epoch) < 0) {
            if (*(volatile uint32_t*)(h.scratch + 1)) return;
            if (globaltimer_ns() - t0 > 4000000000ull) { atomicExch(h.scratch + 1, 1u); return; }
            __nanosleep(64);
        }
    }
    // The peer released its flag after fencing its rows.  Readers that go through L1 (the per-tile kernel's x gather, unstaged
    // tiles) need the full fence: it also drops the SM's L1 lines (SASS CCTL.IVALL), and a 32-column line that straddles the own /
    // halo boundary may have been cached before the peer's part of it arrived.  The streaming kernel reads x with bulk copies
    // (L2): an acquire load of the flag pairs with the peer's st.release.sys and does not stall the warp for microseconds.
    if (full_fence) fence_acq_rel_sys();
    else (void)ld_acquire_sys(f);
}
// one thread of every pushing CTA, after the CTA's remote stores were fenced (system scope) and barriered
__device__ __forceinline__ void halo_signal(const HaloDev& h) {
    const uint32_t old = atomicAdd(h.scratch, 1u);
    if (old + 1u == h.n_sig) {
        *(volatile uint32_t*)h.scratch = 0u;             // ready for the next launch
        __threadfence_system();
        for (int p = 0; p < h.n_peer; p++) st_release_sys(h.peer_flag[p], h.signal_epoch);
    }
}
// rows [row, row + 4) of y (row a multiple of 4; the ragged tail stops at `rows`) to every peer range that contains them.
// Compared as row <= hi - 4, not row + 4 <= hi: row + 4 overflows int for the last quad of a matrix of 2^31 - 1 rows.
__device__ __forceinline__ void halo_store(const HaloDev& h, int row, int rows, const float (&acc)[4]) {
    for (int i = 0; i < h.n_push; i++) {
        const int lo = h.lo[i], hi = h.hi[i];
        if (row >= hi || row <= lo - 4) continue;
        float* d = h.dst[i] + (row - lo);
        if (row >= lo && row <= hi - 4 && row <= rows - 4) {
            *reinterpret_cast<float4*>(d) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++) if (row + q >= lo && row + q < hi && row + q < rows) d[q] = acc[q];
        }
    }
}

__global__ void halo_wait_kernel(const HaloDev h) {
    if ((int)threadIdx.x < h.n_peer) halo_wait(h, threadIdx.x);
}
// stand-alone push (first exchange after set_x, and products that run the block-parallel kernel): every thread reads four rows of y
// once and stores them to every peer range that contains them -- 16-byte stores, 512 contiguous bytes per warp and peer, all
// peers' links busy at the same time (for a scattered matrix every peer needs the whole slice: an all-gather written by the owner)
// The loop counter is 64-bit: a range that ends at 2^31 - 1 would step an int counter past INT_MAX, and with no range at all
// (lo_all = INT_MAX) the first row would already overflow.  Inside the loop r < hi_all <= rows fits in int; the quad tests
// compare against hi - 4 and rows - 4 for the same reason as halo_store.
__global__ void __launch_bounds__(256) halo_push_kernel(const float* __restrict__ y, int rows, const HaloDev h) {
    int lo_all = 0x7FFFFFFF, hi_all = 0;
    for (int i = 0; i < h.n_push; i++) { lo_all = min(lo_all, h.lo[i]); hi_all = max(hi_all, h.hi[i]); }
    const int64_t step = 4 * (int64_t)(gridDim.x * blockDim.x);
    for (int64_t r64 = lo_all + 4 * (int64_t)(blockIdx.x * blockDim.x + threadIdx.x); r64 < hi_all; r64 += step) {
        const int r = (int)r64;
        float v[4];
        if (r <= rows - 4) { const float4 t = *reinterpret_cast<const float4*>(y + r); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
        else { for (int q = 0; q < 4; q++) v[q] = r + q < rows ? y[r + q] : 0.f; }
        for (int i = 0; i < h.n_push; i++) {
            const int lo = h.lo[i], hi = h.hi[i];
            if (r >= hi || r <= lo - 4) continue;
            float* d = h.dst[i] + (r - lo);
            if (r >= lo && r <= hi - 4) *reinterpret_cast<float4*>(d) = make_float4(v[0], v[1], v[2], v[3]);
            else { for (int q = 0; q < 4; q++) if (r + q >= lo && r + q < hi) d[q] = v[q]; }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) halo_signal(h);
}

// One CTA per tile of RTT block rows, two threads per block row (one per 32-bit bitmap half, 4 matrix rows each).  One thread
// per block row (all 8 matrix rows) was measured slower on P4096: 103.5 us against 92.7 us -- fewer instructions, but too few
// warps to hide the staging latency.  Every thread reads the 32-byte tile descriptor; thread 0 arms the mbarrier and issues the
// bulk copies (row pointers, bitmaps, x offsets, values) while all threads gather the tile's distinct x lines (coalesced 16-byte
// loads, stored at a 33-element pitch); latency is hidden by the CTAs resident per SM, each in a different phase.
// H = HaloDev: the multi-GPU variant (waits for the peers' halo slices before gathering x, pushes its boundary rows).
template <typename T, typename X, int RTT, int MINB, typename H = NoHalo>
__global__ void __launch_bounds__(RTT * 2, MINB) spmv_tile_kernel(const TileArgs<T> a, const X* __restrict__ x, float* __restrict__ y, const H hd) {
    constexpr bool DIST = !std::is_same<H, NoHalo>::value;
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int VA = 16 / sizeof(T);   // values per 16 bytes
    constexpr int LPI = RTT * 2 / 8;     // x lines per gather step (8 threads per line)
    constexpr int GB = 4;                // gather steps in flight
    constexpr uint32_t SX = sizeof(X);
    const int tid = threadIdx.x;
    int t = blockIdx.x + a.tile0;
    if constexpr (DIST) { t += hd.rot; if (t >= (int)gridDim.x) t -= (int)gridDim.x; }
    const uint32_t sbase = smem_u32(smem);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + a.so.bar);

    const int4* dp = reinterpret_cast<const int4*>(a.desc + t);
    const int4 d0 = __ldg(dp);
    const int4 d1 = __ldg(dp + 1);       // nl, flags, lmin, lmax
    const int p0 = d0.x, nb = d0.y, nv = d0.w, nl = d1.x;
    const uint32_t v0 = (uint32_t)d0.z, v0a = v0 & ~(uint32_t)(VA - 1);
    const bool staged = (d1.y & 1) && nb <= a.cap_blk && nv <= a.cap_val && nl <= a.cap_lines;
    const int r0 = t * RTT, nrow = min(RTT, a.nbr - r0);

    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
        const uint32_t nrb = (uint32_t)((nrow + 1 + 1) & ~1) * 8;
        const int p0a = p0 & ~1, p0x = p0 & ~7;
        uint32_t n8 = 0, n2 = 0, nvb = 0;
        if (staged && nb > 0) {
            n8 = (uint32_t)((p0 + nb - p0a + 1) & ~1) * 8;
            n2 = (uint32_t)((p0 + nb - p0x + 7) & ~7) * 2;
            nvb = ((v0 + (uint32_t)nv - v0a + (uint32_t)(VA - 1)) & ~(uint32_t)(VA - 1)) * (uint32_t)sizeof(T);
        }
        mbar_arrive_expect_tx(bar, n8 + n2 + nvb + nrb);
        bulk_g2s(smem + a.so.row, a.rowpair + r0, nrb, bar);
        if (n8) bulk_g2s(smem, a.bmps + p0a, n8, bar);
        if (n2) bulk_g2s(smem + a.so.xo, a.xoff + p0x, n2, bar);
        if (nvb) bulk_g2s(smem + a.so.val, a.values + v0a, nvb, bar);
    }
    bool part = false;               // DIST: this tile owns rows a peer needs (CTA-uniform)
    if constexpr (DIST) {
        // trow1 in 64 bits: (r0 + nrow) * 8 is 2^31 for the last tile of a matrix of 2^31 - 1 rows
        const int trow0 = r0 * 8;
        const int64_t trow1 = min((int64_t)a.rows, (int64_t)(r0 + nrow) * 8);
        part = t == hd.solo_tile;
        for (int i = 0; i < hd.n_push; i++) part |= hd.lo[i] < trow1 && hd.hi[i] > trow0;
        // A tile depends on the peers when its x lines leave this rank's own columns (it reads rows they pushed) or when it
        // pushes rows itself: the peers' epoch is the back-pressure that keeps this rank from overwriting a buffer a slower
        // peer still reads, also for one-directional patterns (triangular, directed graphs) where a pushing tile reads nothing
        // remote.  The matrix copies above are already in flight; x must not be touched before the halo is in.
        if (part || (nb > 0 && ((int64_t)d1.z * 32 < hd.own_c0 || ((int64_t)d1.w + 1) * 32 > hd.own_c1))) {
            if (tid < hd.n_peer) halo_wait(hd, tid);
            __syncthreads();
        }
    }
    if (staged) {
        // x lines -> shared: 8 threads per line (4 elements each), GB steps of LPI lines in flight before the first store
        const uint32_t j4 = (uint32_t)(tid & 7) * 4u;
        const int l0 = tid >> 3;
        const uint32_t* lp = a.lines + p0 + l0;
        uint32_t dst = sbase + a.so.xs + ((uint32_t)l0 * XL_STRIDE + j4) * SX;
        const X* xj = x + j4;
        if (!(d1.y & 2)) {
            for (int l = l0; l < nl; l += LPI * GB) {
                XQuad<X> buf[GB];
#pragma unroll
                for (int g = 0; g < GB; g++)
                    if (l + g * LPI < nl) buf[g] = *reinterpret_cast<const XQuad<X>*>(xj + (size_t)__ldg(lp + g * LPI) * 32u);
#pragma unroll
                for (int g = 0; g < GB; g++)
                    if (l + g * LPI < nl) {
#pragma unroll
                        for (int e = 0; e < 4; e++) sts_x<X>(dst + (uint32_t)(g * LPI * XL_STRIDE + e) * SX, buf[g].e[e]);
                    }
                lp += LPI * GB;
                dst += (uint32_t)(LPI * GB * XL_STRIDE) * SX;
            }
        } else {      // the tile's last line reaches past the last column: element-wise guarded loads
            for (int l = l0; l < nl; l += LPI) {
                const uint32_t col = __ldg(lp) * 32u + j4;
#pragma unroll
                for (int e = 0; e < 4; e++) sts_x<X>(dst + e * SX, col + e < (uint32_t)a.cols ? x[col + e] : X(0.f));
                lp += LPI;
                dst += (uint32_t)(LPI * XL_STRIDE) * SX;
            }
        }
    }
    __syncthreads();                 // barrier initialised and armed, x lines visible
    mbar_wait(bar, 0);

    const int lbr = tid >> 1, h = tid & 1;
    const int row = (r0 + lbr) * 8 + h * 4;
    const bool active = lbr < nrow && row < a.rows;
    if (!DIST && !active) return;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (active) {
        const uint2 rp = lds_v2(sbase + a.so.row + 8u * lbr);          // (first block, first value) of this block row
        const uint32_t pe = lds_u32(sbase + a.so.row + 8u * lbr + 8u);
        const uint32_t pb = rp.x, kv = rp.y;
        if (staged) {
            const uint32_t rel = pb - (uint32_t)p0;
            const uint32_t a_bm = sbase + ((uint32_t)(p0 & 1) + rel) * 8u, a_xo = sbase + a.so.xo + ((uint32_t)(p0 & 7) + rel) * 2u;
            const uint32_t a_v = sbase + a.so.val + (kv - v0a) * (uint32_t)sizeof(T), xs31 = sbase + a.so.xs + 31u * SX;
            tile_half_row<T, X>(a_bm, a_xo, a_v, (int)(pe - pb), h, xs31, acc);
        } else {
            half_block_row<T, X>(a.bmps, a.bcol, a.values, (int)pb, (int)pe, kv, h, x, acc);
        }
        float* yr = y + row;
        // row <= rows - 4, not row + 4 <= rows: row + 4 overflows int for the last four rows of a matrix of 2^31 - 1 rows
        if (row <= a.rows - 4) *reinterpret_cast<float4*>(yr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        else {
#pragma unroll
            for (int q = 0; q < 4; q++) if (row + q < a.rows) yr[q] = acc[q];
        }
    }
    if constexpr (DIST) {
        if (part) {
            if (active) halo_store(hd, row, a.rows, acc);
            __threadfence_system();
            __syncthreads();
            if (tid == 0) halo_signal(hd);
        }
    }
}


// ===================================================================================== path 0, streaming kernel
// Persistent CTAs, warp-specialised.  The one-CTA-per-tile kernel above holds a tile's shared memory through three dependent
// global latencies (descriptor -> line list -> x lines) before it computes anything: with shared memory as the limiting
// resource that idle time is what caps the bytes in flight (ncu, round 1: 58 % of the stall samples sit in that prologue).
// Here a CTA is one producer warp plus 2 * STREAM_RT consumer threads (two per block row, one per 32-bit bitmap half) and owns
// `spg` tile-sized stages of shared memory.  CTA b takes the tiles b + k gridDim.x, k = 0, 1, .. -- the SMs sweep the matrix
// together, so the x lines shared by neighbouring tiles are in L2 at the same time.  The kernel runs 64-row tiles only: on the
// 16- and 32-row tiles of heavy rows it is slower than the per-tile kernel (plan_tiles).
//   producer (one elected lane): keeps the 64-byte descriptors of its next tiles arriving by cp.async in a small ring, and as
//     soon as a stage is released issues the tile's bulk copies -- row pointers, bitmaps, x offsets, values, and the tile's x
//     lines as one copy per run of consecutive lines (three runs for a 5-point stencil; line by line, all lanes, for scattered
//     tiles) -- all completing on the stage's `full` mbarrier.  A stage waits for ONE memory latency, not three.
//   consumers: wait for `full`, multiply out of shared memory, store y, arrive on the stage's `empty` mbarrier.
// No CTA-wide barrier after start-up.  Every 128 consumers need a producer warp of their own: a warp issues its ~200 instructions
// per tile at one every few cycles, so one producer for seven such consumer groups caps the SM at one tile per 0.7 us (measured).
// Several groups with a producer each per CTA were slower than one group per CTA (P4096: 6 groups x 1 CTA 69.7 us, 1 x 7 67.8 us).
constexpr int STREAM_RT = 64;      // block rows per tile
constexpr int STREAM_CTAS = 7;     // CTAs per SM the kernel's registers must allow (P4096: 7 x 2 stages, the measured optimum)
static_assert(STREAM_RT == 64 && SHAPE_BIAS > 8u * (STREAM_RT - 1), "row shapes: 64-row tiles (r & 63), positive biased x offsets");
// pal: the palette variant -- a 32-byte header (the second 16 bytes: the tile's block and value counts as the last row's end), one
// 32-bit word per block in place of bitmaps and x offsets (`bm`; `xo` unused), 4-byte relative row pairs; shp: the palette variant
// with row shapes -- no block words at all
struct StageLayout { uint32_t bm, xo, val, row, xs, stride; };
inline StageLayout stage_layout(int cap_blk, int cap_val, int cap_lines, int vsize, int xsize, bool pal, bool shp) {
    constexpr uint32_t rt = STREAM_RT;
    auto up16 = [](uint32_t v) { return (v + 15u) & ~15u; };
    StageLayout s;
    if (pal) {
        s.bm = 32;
        s.xo = s.val = shp ? s.bm : up16(s.bm + (uint32_t)(cap_blk + 4) * 4);
        s.row = up16(s.val + (uint32_t)(cap_val + 16) * vsize);
        s.xs = up16(s.row + (rt + 4) * 4);
    } else {
        s.bm = 16;                                               // 16-byte header: {p0, v0, staged, -}
        s.xo = up16(s.bm + (uint32_t)(cap_blk + 2) * 8);
        s.val = up16(s.xo + (uint32_t)(cap_blk + 16) * 2);
        s.row = up16(s.val + (uint32_t)(cap_val + 16) * vsize);
        s.xs = up16(s.row + (rt + 2) * 8);
    }
    s.stride = (s.xs + (uint32_t)cap_lines * 32u * xsize + 16u + 127u) & ~127u;   // + 16: the tridiagonal path reads one element past
    return s;
}

template <typename T>
struct StreamArgs {
    TileArgs<T> t;
    StageLayout so;
    int32_t spg, ntiles;         // stages per CTA; tiles of this launch (tile0 .. tile0 + ntiles)
    int32_t n_static;            // a CTA's first n_static tiles are its static share (tile slot blockIdx.x + k * gridDim.x) ...
    int32_t* sched;              // ... the rest it claims one at a time from sched[0]; sched[1] counts finished CTAs.  nullptr: all static
};

__device__ __forceinline__ int4 lds_v4(uint32_t a) {
    int4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bar_sync_named(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

constexpr int SCHED_SLOTS = 16;
constexpr int STREAM_DR = 8, STREAM_PD = 4;      // descriptor ring slots / prefetch distance of a producer

// The rare multi-GPU actions of the streaming kernel, out of line: a tile in 2000 waits for the peers or pushes rows, and inlined
// these bodies (spin loops, system fences, a named barrier) cost the multiply loop its schedule.
__device__ __noinline__ void halo_wait_all(const HaloDev* hd, int lane, bool full_fence) {
    if (lane < hd->n_peer) halo_wait(*hd, lane, full_fence);
}
__device__ __noinline__ void halo_push_tile(const HaloDev* hd, int row, int rows, bool active, float a0, float a1, float a2, float a3, int gt, int bar_id, int nthreads) {
    if (active) { const float acc[4] = {a0, a1, a2, a3}; halo_store(*hd, row, rows, acc); }
    // the consumers' remote stores happen-before their barrier, the barrier before thread 0's system fence (cumulative), the fence
    // before the counter / flag: one fence per pushing tile instead of one per thread -- a system fence stalls its warp for
    // microseconds, and a CTA that stalls finishes its static share of the tiles that much later than everybody else
    asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nthreads) : "memory");
    if (gt == 0) { __threadfence_system(); halo_signal(*hd); }
}

// PAL: the matrix has a bitmap palette (see palette_scan_kernel); it is loaded once per CTA, behind the descriptor ring.
// SHP (with PAL): row shapes (see shape_scan_kernel); their table follows the palette in the same buffer and the same bulk copy.
template <typename T, typename X, typename H = NoHalo, bool PAL = false, bool SHP = false>
__global__ void __launch_bounds__(32 + STREAM_RT * 2, STREAM_CTAS) spmv_stream_kernel(const __grid_constant__ StreamArgs<T> sa, const X* __restrict__ x,
                                                                                    float* __restrict__ y, const __grid_constant__ H hd) {
    static_assert(PAL || !SHP, "row shapes come with a palette");
    constexpr bool DIST = !std::is_same<H, NoHalo>::value;
    constexpr int GT = STREAM_RT * 2;      // consumer threads: two per block row
    constexpr int VA = 16 / sizeof(T);
    constexpr uint32_t SX = sizeof(X);
    constexpr int DR = STREAM_DR, PD = STREAM_PD;
    extern __shared__ __align__(128) unsigned char smem[];
    const TileArgs<T>& a = sa.t;
    const StageLayout so = sa.so;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int spg = sa.spg;
    const uint32_t sbase = smem_u32(smem);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)spg * so.stride);      // full[spg], empty[spg]
    uint64_t* empty = full + spg;
    const uint32_t pal_off = (uint32_t)spg * (so.stride + 16u) + DR * 64u + 64u;        // PAL: barrier, then the entries
    uint64_t* pal_bar = reinterpret_cast<uint64_t*>(smem + pal_off);
    if (tid == 0) {
        for (int s = 0; s < spg; s++) { mbar_init(full + s, 1); mbar_init(empty + s, GT / 32); }
        if constexpr (PAL) mbar_init(pal_bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if constexpr (PAL) {
        if (tid == 0) {
            const uint32_t nbytes = (uint32_t)a.npal * 16u + (SHP ? (uint32_t)a.shape_words * 4u : 0u);    // shape_words: a multiple of 4
            mbar_arrive_expect_tx(pal_bar, nbytes);
            bulk_g2s(smem + pal_off + 16, a.palette, nbytes, pal_bar);
        }
    }
    const int grid = (int)gridDim.x;
    // Tile slots q = 0 .. ntiles - 1 in launch order.  A CTA's sequence of slots: blockIdx.x + k * grid for its static share, then
    // slots claimed from a counter (sa.sched).  Static shares alone leave the kernel as slow as its slowest CTA: a CTA that stalled
    // -- a system fence after pushing rows to a peer costs microseconds, a tile of a clustered matrix can be several times the
    // average -- finishes its share that much later than the rest.  With the last part of the tiles handed out on demand the others
    // absorb it.
    const int q0 = (int)blockIdx.x;
    auto tile_at = [&](int q) {
        if constexpr (DIST) { q += hd.rot; if (q >= sa.ntiles) q -= sa.ntiles; }
        return a.tile0 + q;
    };

    if (warp == 0) {
        // ------------------------------------------------------------------------------------------ producer
        // The descriptors of the next PD tiles travel global -> shared with cp.async (no register is waited on), one commit group
        // per tile; group k is complete once at most PD newer groups are pending.
        const uint32_t ring = sbase + (uint32_t)spg * (so.stride + 16u);
        static_assert(DR * 4 <= 64, "tile ids of the ring live in the 64 spare bytes behind it");
        const uint32_t tq = ring + DR * 64u;
        const int n_static = sa.sched ? sa.n_static : 0x7fffffff;
        const int dyn_base = sa.sched ? sa.n_static * grid : 0;
        int pending = 0;                  // lane 0: the slot claimed for the next dynamic sequence number, asked for one iteration ahead
        bool ended = false;               // lane 0: a slot past the last tile has been seen (every later one is past it too)
        // descriptor of sequence number k (slot q) -> ring, its tile id -> tq; a slot past the end leaves the end marker (-1)
        auto issue = [&](int k, int q) {
            int t = -1;
            if (q < sa.ntiles) {
                t = tile_at(q);
                const char* src = reinterpret_cast<const char*>(a.desc + t);
                const uint32_t dst = ring + (uint32_t)(k % DR) * 64u;
#pragma unroll
                for (int c = 0; c < 4; c++) cp_async16(dst + 16u * c, src + 16 * c);
            } else ended = true;
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(tq + (uint32_t)(k % DR) * 4u), "r"(t) : "memory");
            cp_async_commit();
        };
        if (lane == 0) {
            for (int k = 0; k < PD; k++) issue(k, k < n_static ? q0 + k * grid : (ended ? sa.ntiles : dyn_base + atomicAdd(sa.sched, 1)));
            if (PD >= n_static && !ended) pending = dyn_base + atomicAdd(sa.sched, 1);
        }
        int s = 0; uint32_t round = 0;
        for (int k = 0;; k++) {
            int4 d0, d1, d2, d3;
            if (lane == 0) {
                // refill the ring, then make sure tile k's descriptor has landed.  The claim for the sequence number after this one
                // goes out now and is looked at in the next iteration: the atomic's round trip never stalls the warp.
                const int kk = k + PD;
                const int q = kk < n_static ? q0 + kk * grid : (ended ? sa.ntiles : pending);
                issue(kk, q);
                if (kk + 1 >= n_static && !ended) pending = dyn_base + atomicAdd(sa.sched, 1);
                cp_async_wait<PD>();
            }
            __syncwarp();
            const int t = (int)lds_u32(tq + (uint32_t)(k % DR) * 4u);
            if (t < 0) {
                // no more tiles: tell the consumers through the next stage's header
                if (round) mbar_wait(empty + s, (round - 1u) & 1u);
                if (lane == 0) {
                    *reinterpret_cast<int4*>(smem + (size_t)s * so.stride) = make_int4(0, 0, 0, -1);
                    mbar_arrive(full + s);
                }
                break;
            }
            const uint32_t dsl = ring + (uint32_t)(k % DR) * 64u;
            d0 = lds_v4(dsl); d1 = lds_v4(dsl + 16); d2 = lds_v4(dsl + 32); d3 = lds_v4(dsl + 48);
            const int p0 = d0.x, nb = d0.y, nv = d0.w, nl = d1.x;
            const uint32_t v0 = (uint32_t)d0.z, v0a = v0 & ~(uint32_t)(VA - 1);
            const bool staged = (d1.y & 1) && nb <= a.cap_blk && nv <= a.cap_val && nl <= a.cap_lines;
            const int r0 = t * STREAM_RT, nrow = min(STREAM_RT, a.nbr - r0);
            const uint32_t sp32 = sbase + (uint32_t)s * so.stride;
            unsigned char* sp = smem + (size_t)s * so.stride;
            // PAL: nrb = relative row pairs (4 B per block row), n8 = block words from p0a = p0 & ~3; otherwise int2 row pairs (one past
            // the tile's last row), bitmaps from p0 & ~1 and x offsets from p0 & ~7
            const uint32_t nrb = PAL ? (uint32_t)((nrow + 3) & ~3) * 4 : (uint32_t)((nrow + 1 + 1) & ~1) * 8;
            const int p0a = PAL ? p0 & ~3 : p0 & ~1, p0x = p0 & ~7;
            uint32_t n8 = 0, n2 = 0, nvb = 0;
            int nlc = 0;                                                  // x lines that arrive by bulk copy
            if (staged && nb > 0) {
                if constexpr (SHP) {}                                     // no block words: the shapes are in shared memory
                else if constexpr (PAL) n8 = (uint32_t)((p0 + nb - p0a + 3) & ~3) * 4;
                else {
                    n8 = (uint32_t)((p0 + nb - p0a + 1) & ~1) * 8;
                    n2 = (uint32_t)((p0 + nb - p0x + 7) & ~7) * 2;
                }
                nvb = ((v0 + (uint32_t)nv - v0a + (uint32_t)(VA - 1)) & ~(uint32_t)(VA - 1)) * (uint32_t)sizeof(T);
                nlc = (d1.y & 2) ? nl - 1 : nl;                          // a last line that reaches past the last column is loaded by hand
            }
            bool part = false;                                            // DIST: this tile owns rows a peer needs
            if constexpr (DIST) {
                // A tile whose x lines leave this rank's own columns must not read x before the peers' rows are in, and a tile that
                // pushes rows waits too (back-pressure, see spmv_tile_kernel).  The producer waits on the tile's behalf before it
                // completes `full`; the rotated tile order puts these tiles mid-kernel, where the wait is over before it starts.
                // Whether the tile pushes goes to the consumers through the stage header: evaluated by them, the loop over the push
                // ranges cost every warp ~100 instructions per tile (ncu: 64.5 M warp instructions against 51.9 M).
                part = t == hd.solo_tile;
                for (int i = 0; i < hd.n_iv; i++) part |= t >= hd.iv_lo[i] && t <= hd.iv_hi[i];
                if (part || (nb > 0 && ((int64_t)d1.z * 32 < hd.own_c0 || ((int64_t)d1.w + 1) * 32 > hd.own_c1))) {
                    halo_wait_all(&hd, lane, !staged);
                    __syncwarp();
                    // the x lines are fetched by the async proxy (bulk copies): order them behind the acquire made above
                    asm volatile("fence.proxy.async;" ::: "memory");
                }
            }
            // everything above is ready before the stage is: what follows the wait is the stage's critical path (a CTA has two
            // stages; a microsecond between a stage's release and its next copies is a microsecond without loads in flight)
            if (round) mbar_wait(empty + s, (round - 1u) & 1u);          // the stage's previous tile has been consumed
            if (staged && nlc < nl) {
                const uint32_t col = (uint32_t)d1.w * 32u + (uint32_t)lane;          // lmax is the tile's last line
                sts_x<X>(sp32 + so.xs + ((uint32_t)(nl - 1) * 32u + (uint32_t)lane) * SX, col < (uint32_t)a.cols ? x[col] : X(0.f));
                __syncwarp();
            }
            const bool by_runs = d2.x > 0;
            if (lane == 0) {
                *reinterpret_cast<int4*>(sp) = make_int4(p0, (int)v0, (staged ? 1 : 0) | (part ? 2 : 0), t);     // the consumers take the tile from here
                if constexpr (PAL) *reinterpret_cast<uint32_t*>(sp + 16) = (uint32_t)nb | (uint32_t)nv << 16;
                mbar_arrive_expect_tx(full + s, n8 + n2 + nvb + nrb + (uint32_t)nlc * 32u * SX);
                if constexpr (PAL) {
                    bulk_g2s(sp + so.row, a.rowrel + r0, nrb, full + s);
                    if (n8) bulk_g2s(sp + so.bm, a.word + p0a, n8, full + s);
                } else {
                    bulk_g2s(sp + so.row, a.rowpair + r0, nrb, full + s);
                    if (n8) bulk_g2s(sp + so.bm, a.bmps + p0a, n8, full + s);
                    if (n2) bulk_g2s(sp + so.xo, a.xoff + p0x, n2, full + s);
                }
                if (nvb) bulk_g2s(sp + so.val, a.values + v0a, nvb, full + s);
                if (nlc > 0 && by_runs) {                                 // up to three runs of consecutive lines
                    unsigned char* xs = sp + so.xs;
                    const uint32_t rl[3] = {(uint32_t)d2.y, (uint32_t)d2.z, (uint32_t)d2.w}, rc[3] = {(uint32_t)d3.x, (uint32_t)d3.y, (uint32_t)d3.z};
                    uint32_t first = 0;
#pragma unroll
                    for (int r = 0; r < 3; r++) {
                        if (r < d2.x) {
                            uint32_t cnt = rc[r];
                            if (first + cnt > (uint32_t)nlc) cnt = (uint32_t)nlc - first;     // the hand-loaded last line
                            if (cnt) bulk_g2s(xs + (size_t)first * 32u * SX, x + (size_t)rl[r] * 32u, cnt * 32u * SX, full + s);
                            first += rc[r];
                        }
                    }
                }
            }
            if (nlc > 0 && !by_runs) {                                    // scattered lines: one copy per line, all lanes
                __syncwarp();                                             // after lane 0's expect_tx
                unsigned char* xs = sp + so.xs;
                for (int j = lane; j < nlc; j += 32)
                    bulk_g2s(xs + (size_t)j * 32u * SX, x + (size_t)__ldg(a.lines + p0 + j) * 32u, 32u * SX, full + s);
            }
            if (++s == spg) { s = 0; round++; }
        }
        if (sa.sched && lane == 0) {
            // the last CTA to finish claiming re-arms the counters for the next launch that takes this slot
            __threadfence();
            if (atomicAdd(sa.sched + 1, 1) == grid - 1) { sa.sched[0] = 0; sa.sched[1] = 0; }
        }
    } else {
        // ------------------------------------------------------------------------------------------ consumers
        const int gt = tid - 32;
        const int lbr = gt >> 1, h = gt & 1;
        const uint32_t pal_h = sbase + pal_off + 16u + 8u * (uint32_t)h;    // PAL: this half's 8 bytes of entry 0
        const uint32_t shp_t = sbase + pal_off + 16u + (uint32_t)a.npal * 16u;   // SHP: the shape table
        if constexpr (PAL) mbar_wait(pal_bar, 0);
        int s = 0; uint32_t par = 0;
        for (;;) {
            mbar_wait(full + s, par);
            const uint32_t sb = sbase + (uint32_t)s * so.stride;
            const int4 hdr = lds_v4(sb);                                  // {first block, first value, staged | pushes << 1, tile}
            const int t = hdr.w;
            if (t < 0) break;                                             // the producer ran out of tiles
            const int r0 = t * STREAM_RT, nrow = min(STREAM_RT, a.nbr - r0);
            const int p0 = hdr.x; const uint32_t v0a = (uint32_t)hdr.y & ~(uint32_t)(VA - 1);
            const bool staged = (hdr.z & 1) != 0;
            const int row = (r0 + lbr) * 8 + h * 4;
            const bool active = lbr < nrow && row < a.rows;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            if (active) {
                if constexpr (SHP) {
                    if (staged) {
                        // {shape, block count, first value relative to the tile}; the shape's x offsets are relative to this row (biased)
                        const uint32_t rp = lds_u32(sb + so.row + 4u * lbr);
                        const uint32_t a_v = sb + so.val + ((uint32_t)hdr.y - v0a + (rp >> 16)) * (uint32_t)sizeof(T);
                        const uint32_t xs31 = sb + so.xs + (31u + 8u * (uint32_t)lbr - SHAPE_BIAS) * SX;
                        tile_half_row_pal<T, X>(shp_t + (rp & 0x7FFu) * 4u, pal_h, a_v, (int)((rp >> 11) & 31u), h, xs31, acc);
                    } else {
                        const int br = r0 + lbr;
                        half_block_row<T, X>(a.bmps, a.bcol, a.values, __ldg(a.brp + br), __ldg(a.brp + br + 1), __ldg(a.rvb + br), h, x, acc);
                    }
                } else if constexpr (PAL) {
                    if (staged) {
                        // (first block, first value) of this block row and of the next one, relative to the tile; the tile's counts end the last row
                        const uint32_t rp = lds_u32(sb + so.row + 4u * lbr);
                        const uint32_t re = lbr + 1 < nrow ? lds_u32(sb + so.row + 4u * lbr + 4u) : lds_u32(sb + 16u);
                        const uint32_t rb = rp & 0xFFFFu;
                        const uint32_t a_w = sb + so.bm + ((uint32_t)(p0 & 3) + rb) * 4u;
                        const uint32_t a_v = sb + so.val + ((uint32_t)hdr.y - v0a + (rp >> 16)) * (uint32_t)sizeof(T), xs31 = sb + so.xs + 31u * SX;
                        tile_half_row_pal<T, X>(a_w, pal_h, a_v, (int)((re & 0xFFFFu) - rb), h, xs31, acc);
                    } else {
                        const int br = r0 + lbr;
                        half_block_row<T, X>(a.bmps, a.bcol, a.values, __ldg(a.brp + br), __ldg(a.brp + br + 1), __ldg(a.rvb + br), h, x, acc);
                    }
                } else {
                    const uint2 rp = lds_v2(sb + so.row + 8u * lbr);          // (first block, first value) of this block row
                    const uint32_t pe = lds_u32(sb + so.row + 8u * lbr + 8u);
                    const uint32_t pb = rp.x, kv = rp.y;
                    if (staged) {
                        const uint32_t rel = pb - (uint32_t)p0;
                        const uint32_t a_bm = sb + so.bm + ((uint32_t)(p0 & 1) + rel) * 8u, a_xo = sb + so.xo + ((uint32_t)(p0 & 7) + rel) * 2u;
                        const uint32_t a_v = sb + so.val + (kv - v0a) * (uint32_t)sizeof(T), xs31 = sb + so.xs + 31u * SX;
                        tile_half_row<T, X, true>(a_bm, a_xo, a_v, (int)(pe - pb), h, xs31, acc);
                    } else {
                        half_block_row<T, X>(a.bmps, a.bcol, a.values, (int)pb, (int)pe, kv, h, x, acc);
                    }
                }
                float* yr = y + row;
                if (row <= a.rows - 4) *reinterpret_cast<float4*>(yr) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                else {
#pragma unroll
                    for (int q = 0; q < 4; q++) if (row + q < a.rows) yr[q] = acc[q];
                }
            }
            if constexpr (DIST) {
                if (hdr.z & 2)                                           // the producer found rows of this tile in a push range
                    halo_push_tile(&hd, row, a.rows, active, acc[0], acc[1], acc[2], acc[3], gt, 1, GT);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + s);
            if (++s == spg) { s = 0; par ^= 1u; }
        }
    }
}

// ------------------------------------------------------------------------------------ path 1
// work item: x = block row, y = first block, z = end block, w = 1 when the block row is sliced.
// One warp per item, UNR x 32 blocks per step: every lane issues the metadata loads of its UNR blocks together, the UNR
// warp scans of popc (value offsets) interleave, and the first value / x element of each of the UNR blocks -- with
// about one value per block that is nearly all of them -- are loaded back to back before any of them is used, so a
// step has 4 * UNR independent loads in flight per lane instead of a chain of four dependent ones.
// Multi-GPU: the product itself is unchanged; a wait kernel before it and halo_push_kernel after it do the exchange (bmsp_spmv_halo).
// Two in-kernel variants were measured and dropped.  Every warp storing its finished block row to the peers (32-byte pieces):
// 3.78x at 8 GPUs on R-MAT-22 -- NVLink wants 256-byte writes.  Collecting a CTA's eight block rows in shared memory and storing
// 256 bytes per peer: the CTA-wide barrier keeps seven warps waiting for the one that drew a hub-row slice (2 GPUs: 404 us against
// 368 us).  And a system fence per CTA invalidates the SM's L1 (SASS: MEMBAR.SYS + CCTL.IVALL), which this kernel lives on: with
// fences at the start and the end of every CTA the 2-GPU product took 1161 us against 600 us on one GPU.
template <typename T, typename X>
__global__ void __launch_bounds__(256) spmv_blockpar_kernel(const uint64_t* __restrict__ bmps, const int32_t* __restrict__ bcol,
                                                           const uint64_t* __restrict__ offsets, const T* __restrict__ values,
                                                           const int4* __restrict__ work, int n_work, int rows,
                                                           const X* __restrict__ x, float* __restrict__ y,
                                                           float* __restrict__ partial, const int32_t* __restrict__ brp) {
    constexpr int UNR = 4;
    __shared__ float s_acc[8][8][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int item = blockIdx.x * 8 + wid;
    if (item >= n_work) return;
    const int4 w = work[item];
    float (*acc)[32] = s_acc[wid];
#pragma unroll
    for (int r = 0; r < 8; r++) acc[r][lane] = 0.f;
    if (w.w == 2) {
        // bundle: lanes 8q .. 8q+7 take block row w.x + q, one block per lane (at most 8 per row); the eight per-row sums are
        // reduced over the 8 lanes of the group (3 shuffle steps each) and lane 8q + r stores row r: 128 contiguous bytes per warp
        const int sub = lane >> 3, l8 = lane & 7, br = w.x + sub;
        const int b = __ldg(brp + br) + l8;
        if (b < __ldg(brp + br + 1)) {
            uint64_t rem = ld_stream_u64(bmps + b);
            const uint32_t xb = (uint32_t)ld_stream_s32(bcol + b) * 8u;
            uint64_t k = offsets[b];
            while (rem) {
                const int p = __clzll((long long)rem);
                rem &= ~(0x8000000000000000ull >> p);
                acc[p >> 3][lane] += val_to_f32(values[k++]) * ld_x<X>(x, xb + (uint32_t)(p & 7));
            }
        }
        float res = 0.f;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            float v = acc[r][lane];
            v += __shfl_xor_sync(0xffffffffu, v, 1); v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 4);
            if (l8 == r) res = v;
        }
        const int64_t row = (int64_t)br * 8 + l8;
        if (row < rows) y[row] = res;
        return;
    }
    uint64_t vbase = w.y < w.z ? offsets[w.y] : 0;
    for (int b0 = w.y; b0 < w.z; b0 += 32 * UNR) {
        uint64_t bmp[UNR]; uint32_t xb[UNR], cnt[UNR], inc[UNR];
#pragma unroll
        for (int g = 0; g < UNR; g++) {
            const int b = b0 + g * 32 + lane;
            const bool valid = b < w.z;
            bmp[g] = valid ? ld_stream_u64(bmps + b) : 0ull;
            xb[g] = valid ? (uint32_t)ld_stream_s32(bcol + b) * 8u : 0u;
        }
#pragma unroll
        for (int g = 0; g < UNR; g++) { cnt[g] = __popcll(bmp[g]); inc[g] = cnt[g]; }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int g = 0; g < UNR; g++) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc[g], o);
                if (lane >= o) inc[g] += t;
            }
        }
        uint64_t k[UNR];
#pragma unroll
        for (int g = 0; g < UNR; g++) {
            k[g] = vbase + inc[g] - cnt[g];
            vbase += __shfl_sync(0xffffffffu, inc[g], 31);
        }
        // first value of every block: independent loads, issued together
        float v0[UNR], x0[UNR]; int p0[UNR];
#pragma unroll
        for (int g = 0; g < UNR; g++) {
            p0[g] = bmp[g] ? __clzll((long long)bmp[g]) : 0;
            v0[g] = bmp[g] ? val_to_f32(values[k[g]]) : 0.f;
            x0[g] = bmp[g] ? ld_x<X>(x, xb[g] + (uint32_t)(p0[g] & 7)) : 0.f;
        }
#pragma unroll
        for (int g = 0; g < UNR; g++) {
            if (bmp[g]) {
                acc[p0[g] >> 3][lane] += v0[g] * x0[g];
                uint64_t rem = bmp[g] & ~(0x8000000000000000ull >> p0[g]);
                uint64_t kk = k[g] + 1;
                while (rem) {
                    const int p = __clzll((long long)rem);
                    rem &= ~(0x8000000000000000ull >> p);
                    acc[p >> 3][lane] += val_to_f32(values[kk]) * ld_x<X>(x, xb[g] + (uint32_t)(p & 7));
                    kk++;
                }
            }
        }
    }
    float res = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        float v = acc[r][lane];
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == r) res = v;
    }
    if (lane < 8) {
        if (w.w) partial[(int64_t)item * 8 + lane] = res;
        else {
            const int64_t row = (int64_t)w.x * 8 + lane;
            if (row < rows) y[row] = res;
        }
    }
}

// sliced block rows (more than one work item): listed once per plan; spmv_fixup_kernel sums their slices
__global__ void split_list_kernel(const int32_t* __restrict__ item_ofs, int nbr, int32_t* __restrict__ list, int32_t* __restrict__ count) {
    const int br = blockIdx.x * blockDim.x + threadIdx.x;
    if (br < nbr && item_ofs[br + 1] - item_ofs[br] > 1) list[atomicAdd(count, 1)] = br;
}

// One warp per sliced block row: lane l sums the slices l, l + 32, ... (two 16-byte loads per slice: its eight row partials), then
// a fixed shuffle tree adds the lanes -- the order of the additions depends on nothing but the slice count, so the result is
// deterministic.  (One thread per matrix row walking all slices in turn took 12 us on R-MAT-22, whose heaviest block row has ~800
// slices: 10 % of a product at 8 GPUs.)
__global__ void __launch_bounds__(256) spmv_fixup_kernel(const int32_t* __restrict__ item_ofs, const float* __restrict__ partial,
                                                         const int32_t* __restrict__ split_list, int n_split_rows, int rows, float* __restrict__ y) {
    const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= n_split_rows) return;
    const int br = split_list[w];
    const int i0 = item_ofs[br], i1 = item_ofs[br + 1];
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int i = i0 + lane; i < i1; i += 32) {
        const float4 a = *reinterpret_cast<const float4*>(partial + (int64_t)i * 8), b = *reinterpret_cast<const float4*>(partial + (int64_t)i * 8 + 4);
        s[0] += a.x; s[1] += a.y; s[2] += a.z; s[3] += a.w; s[4] += b.x; s[5] += b.y; s[6] += b.z; s[7] += b.w;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
#pragma unroll
        for (int r = 0; r < 8; r++) s[r] += __shfl_xor_sync(0xffffffffu, s[r], o);
    }
    float mine = 0.f;
#pragma unroll
    for (int r = 0; r < 8; r++) if (lane == r) mine = s[r];
    const int64_t row = (int64_t)br * 8 + lane;
    if (lane < 8 && row < rows) y[row] = mine;
}

// Four consecutive block rows (an aligned group) with at most 8 blocks each form ONE work item, a "bundle" (w = 2): eight lanes per
// block row instead of a warp.  R-MAT-22 has 4.2 M matrix rows, 52 % of them empty: a warp per block row cost 41 ns per row -- 29 %
// of the product -- mostly its 40 reduction shuffles.
constexpr int BUNDLE_ROWS = 4, BUNDLE_MAXB = 8;
__device__ __forceinline__ bool is_bundle(const int32_t* __restrict__ brp, int nbr, int br) {
    const int g0 = br & ~(BUNDLE_ROWS - 1);
    if (g0 + BUNDLE_ROWS > nbr) return false;
    bool ok = true;
#pragma unroll
    for (int q = 0; q < BUNDLE_ROWS; q++) ok &= brp[g0 + q + 1] - brp[g0 + q] <= BUNDLE_MAXB;
    return ok;
}
__global__ void work_count_kernel(const int32_t* __restrict__ brp, int nbr, uint32_t* __restrict__ cnt) {
    int br = blockIdx.x * blockDim.x + threadIdx.x;
    if (br >= nbr) return;
    if (is_bundle(brp, nbr, br)) { cnt[br] = (br & (BUNDLE_ROWS - 1)) == 0 ? 1u : 0u; return; }
    int nb = brp[br + 1] - brp[br];
    cnt[br] = nb <= SLICE ? 1u : (uint32_t)((nb + SLICE - 1) / SLICE);
}
__global__ void work_fill_kernel(const int32_t* __restrict__ brp, int nbr, const uint32_t* __restrict__ ofs, int4* __restrict__ work) {
    int br = blockIdx.x * blockDim.x + threadIdx.x;
    if (br >= nbr) return;
    if (is_bundle(brp, nbr, br)) {
        if ((br & (BUNDLE_ROWS - 1)) == 0) work[ofs[br]] = make_int4(br, brp[br], brp[br + BUNDLE_ROWS], 2);
        return;
    }
    int b0 = brp[br], b1 = brp[br + 1];
    uint32_t o = ofs[br], n = ofs[br + 1] - o;
    for (uint32_t i = 0; i < n; i++) {
        int s = b0 + (int)i * SLICE;
        work[o + i] = make_int4(br, s, min(s + SLICE, b1), n > 1 ? 1 : 0);
    }
}

static int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }

// ------------------------------------------------------------------------------------ host-buffer pipeline
// y_host = A x_host with both vectors in (pinned) host memory: the block rows are cut into chunks of whole tiles;
// chunk c needs the columns [0, x_need[c]) of x (running maximum of the tile plan's line ranges -- for a banded matrix
// the frontier advances with the rows, for a scattered one the first chunk needs everything and only the y copies
// overlap).  Three streams: s_in feeds x slices (H2D), the caller's stream runs the row-range launches, s_out drains
// y slices (D2H); PCIe is full duplex, so the step costs max(x, y) bytes over the link instead of their sum.
struct HostPipe {
    DevBuf<char> x_dev;
    DevBuf<float> y_dev;
    Stream s_in, s_out;
    Event ev_start, ev_done;
    std::vector<Event> ev_x, ev_k;
    // the whole pipeline of one (x_host, y_host) pair captured as a CUDA graph: one launch instead of ~7 API calls per chunk
    Stream s_cap;
    GraphExec gexec;
    const void* g_x = nullptr; const void* g_y = nullptr; int32_t g_xdt = -1;      // what gexec was captured for
    const void* seen_x = nullptr; const void* seen_y = nullptr; int32_t seen_xdt = -1;   // the previous call's buffers
    std::vector<int> tile_lo;        // [nchunks+1] first tile of every chunk (row-tiled path); {0, 0} for the block-parallel path
    std::vector<int64_t> x_need;     // [nchunks]  columns that must be resident before the chunk runs
};

// Everything the first product on a matrix builds (plan_spmv), owned by the handle (bmsp_matrix_s::spmv).  Which members mean
// anything depends on the path, and on the row-tiled path on the kernel and on whether there is a palette.
struct SpmvPlan {
    enum Path { ROW_TILED, BLOCK_PARALLEL } path = ROW_TILED;   // row-tiled: dense-ish blocks; block-parallel: sparse blocks
    // row-tiled path (plan_tiles).  kernel 0 = streaming kernel (persistent CTAs, staged tiles in a shared-memory ring; 64-row tiles
    // only), 1 = one CTA per tile; tiles of 64, 32 or 16 block rows; per-tile shared-memory capacities in blocks, values, x lines
    int32_t kernel = 0, tile_rows = 64, cap_blk = 0, cap_val = 0, cap_lines = 0;
    int32_t npal = 0;            // palette entries (distinct bitmaps), 0 = no palette
    uint32_t sched_next = 0;     // the scheduler slot the streaming kernel's next launch over all tiles takes
    DevBuf<TileDesc> desc;       // [ntiles] block / value / x-line ranges of every tile
    DevBuf<uint32_t> lines;      // [nblk] distinct x lines (32 columns) of every tile, stored from the tile's first block index
    DevBuf<int32_t> sched;       // streaming kernel: SCHED_SLOTS x {next tile to claim, CTAs done}; a launch takes the next slot
    DevBuf<uint16_t> xoff;       // no palette: [nblk] per block, offset of its 8-column x segment inside the tile's staged lines
    DevBuf<int2> rowpair;        // no palette: [nbr+1] (block_row_ptr, first value) zipped for one bulk copy per tile
    // streaming kernel, matrices with at most PALETTE_MAX distinct bitmaps (stencils, bands): the bitmaps are replaced by a palette
    // and xoff / rowpair by word / rowrel ("bitmap palette")
    DevBuf<uint4> palette;       // [npal] 16-byte entries, sorted by bitmap (row shapes: then the shape table, shape_words words)
    DevBuf<uint32_t> word;       // [nblk] per block: x offset (bits 0-15) | palette entry byte offset (bits 16-31); freed with shapes
    DevBuf<uint32_t> rowrel;     // [nbr] per block row: (first block - tile's first block) | (first value - tile's first value) << 16
                                 // (row shapes: {shape, block count} in bits 0-15, see shape_scan_kernel)
    bool shapes = false;         // palette matrices whose staged rows have at most SHAPE_MAX distinct shapes ("row shapes")
    int32_t nshapes = 0, shape_words = 0;   // shapes; table words, padded to a multiple of 4 (one bulk copy with the palette)
    // block-parallel path (plan_block_parallel): n_work int4 work items; the block rows sliced into several items are listed for
    // the fix-up kernel, which sums their items' row sums (split_partial, allocated only when there are such rows)
    int32_t n_work = 0, n_split_rows = 0;
    DevBuf<int4> work;
    DevBuf<uint32_t> item_ofs;   // [nbr+1] first work item of every block row
    DevBuf<int32_t> split_list;
    DevBuf<float> split_partial;
    // bmsp_spmv_host's pipeline, built by its first call.  Declared last so that it is destroyed first: the pipeline's streams
    // drain before any of the plan's memory is freed.
    std::unique_ptr<HostPipe> host;
};

// The streaming kernel's bitmap palette: collect the distinct bitmaps (palette_scan_kernel), sort them here and upload one 16-byte
// entry per bitmap (layout at PalScan) into `palette`.  Leaves pal empty when the matrix has more than PALETTE_MAX distinct bitmaps.
static int build_palette(const bmsp_matrix_s* m, int vsize, cudaStream_t st, std::vector<uint4>& pal, DevBuf<uint4>& palette) {
    DevBuf<PalScan> ps;
    BMSP_TRY(ps.alloc(1, st));
    BMSP_CUDA(cudaMemsetAsync(ps.get(), 0, sizeof(PalScan), st));
    const int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, ceil_div(m->nblk, 256 * 16)));
    palette_scan_kernel<<<grid, 256, 0, st>>>(m->bmps, m->nblk, ps.get());
    BMSP_KERNEL_CHECK();
    std::vector<PalScan> h(1);
    BMSP_CUDA(cudaMemcpyAsync(h.data(), ps.get(), sizeof(PalScan), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    ps.reset();
    if (h[0].overflow) return BMSP_OK;
    std::vector<uint64_t> keys;
    for (int i = 0; i < PAL_GSLOTS; i++) if (h[0].key[i]) keys.push_back(h[0].key[i]);
    if (h[0].has_zero) keys.push_back(0ull);
    if (keys.empty() || keys.size() > (size_t)PALETTE_MAX) return BMSP_OK;
    std::sort(keys.begin(), keys.end());
    for (const uint64_t b : keys) {
        const uint32_t hw[2] = {(uint32_t)(b >> 32), (uint32_t)b};      // half 0 = rows 0-3 (high word), half 1 = rows 4-7
        const uint32_t nhi = (uint32_t)__builtin_popcount(hw[0]), ntot = nhi + (uint32_t)__builtin_popcount(hw[1]);
        uint32_t meta[2];
        for (int h2 = 0; h2 < 2; h2++) {
            const uint32_t w = hw[h2];
            // the tests of tile_half_row, in its order
            uint32_t cls = 0, cell = 0;
            if (w == (0x80402010u >> (4 * h2))) cls = PAL_DIAG;
            else if (w == (h2 ? 0x1C0E0703u : 0xC0E07038u)) cls = PAL_TRI;
            else if (w && !(w & (w - 1u))) { cls = PAL_SINGLE; cell = (uint32_t)__builtin_clz(w); }
            else if (w) cls = PAL_GENERIC;
            meta[h2] = (h2 ? nhi : 0u) * (uint32_t)vsize | cls | cell << 12 | ntot * (uint32_t)vsize << 20;
        }
        pal.push_back(make_uint4(hw[0], meta[0], hw[1], meta[1]));
    }
    BMSP_TRY(palette.alloc(pal.size(), st));
    BMSP_CUDA(cudaMemcpyAsync(palette.get(), pal.data(), sizeof(uint4) * pal.size(), cudaMemcpyHostToDevice, st));
    return BMSP_OK;
}

// Row shapes of a palette matrix (layout at shape_scan_kernel): collect them on the device, sort them here and lay them out behind
// the palette, then rewrite the row words and compare every staged row with its shape.  The word layout stays when the matrix has
// more than SHAPE_MAX shapes or SHAPE_WORDS words in all, a staged row has more than SHAPE_NB blocks, or a row differs from the
// shape of its hash.  Otherwise the per-block words are freed.
static int build_shapes(const bmsp_matrix_s* m, SpmvPlan& p, cudaStream_t st) {
    const int nbr = m->nbr, cb = p.cap_blk, cv = p.cap_val, cl = p.cap_lines, npal = p.npal;
    constexpr int OUTW = SHAPE_NB + 1;
    DevBuf<ShapeScan> ss;
    DevBuf<uint32_t> out;
    BMSP_TRY(ss.alloc(1, st));
    BMSP_TRY(out.alloc((size_t)SHAPE_MAX * OUTW, st));
    BMSP_CUDA(cudaMemsetAsync(ss.get(), 0, sizeof(ShapeScan), st));
    const int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, ceil_div(nbr, 256 * 8)));
    shape_scan_kernel<<<grid, 256, 0, st>>>(m->brp, p.word.get(), p.desc.get(), nbr, cb, cv, cl, ss.get());
    BMSP_KERNEL_CHECK();
    shape_gather_kernel<<<SHP_GSLOTS / 256, 256, 0, st>>>(m->brp, p.word.get(), ss.get(), out.get());
    BMSP_KERNEL_CHECK();
    uint32_t cnt[3];                                     // count, overflow, nout
    std::vector<uint32_t> h((size_t)SHAPE_MAX * OUTW);
    BMSP_CUDA(cudaMemcpyAsync(cnt, &ss.get()->count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(h.data(), out.get(), sizeof(uint32_t) * h.size(), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    out.reset();
    if (cnt[1] || cnt[2] > (uint32_t)SHAPE_MAX) return BMSP_OK;
    const int ns = (int)cnt[2];
    std::vector<std::vector<uint32_t>> shp((size_t)ns);
    std::vector<int> order((size_t)ns);
    for (int k = 0; k < ns; k++) {
        const uint32_t* o = h.data() + (size_t)k * OUTW;
        shp[k].assign(o + 1, o + 1 + (o[0] >> 16));
        order[k] = k;
    }
    std::sort(order.begin(), order.end(), [&](int i, int j) { return shp[i] < shp[j]; });
    std::vector<uint32_t> gval(SHP_GSLOTS, 0u), words;
    for (const int k : order) {
        gval[h[(size_t)k * OUTW] & 0xFFFFu] = (uint32_t)words.size() | (uint32_t)shp[k].size() << 11;
        words.insert(words.end(), shp[k].begin(), shp[k].end());
    }
    if (words.size() > (size_t)SHAPE_WORDS) return BMSP_OK;
    words.resize((words.size() + 3) & ~(size_t)3, 0u);
    DevBuf<uint4> comb;                                  // palette, then the table: one bulk copy per CTA
    DevBuf<uint32_t> gv, srow, bad;
    BMSP_TRY(comb.alloc((size_t)npal + words.size() / 4 + 1, st));
    BMSP_TRY(gv.alloc(SHP_GSLOTS, st));
    BMSP_TRY(srow.alloc((size_t)nbr + 8, st));
    BMSP_TRY(bad.alloc(1, st));
    BMSP_CUDA(cudaMemcpyAsync(comb.get(), p.palette.get(), sizeof(uint4) * npal, cudaMemcpyDeviceToDevice, st));
    if (!words.empty())
        BMSP_CUDA(cudaMemcpyAsync(comb.get() + npal, words.data(), sizeof(uint32_t) * words.size(), cudaMemcpyHostToDevice, st));
    BMSP_CUDA(cudaMemcpyAsync(gv.get(), gval.data(), sizeof(uint32_t) * SHP_GSLOTS, cudaMemcpyHostToDevice, st));
    BMSP_CUDA(cudaMemsetAsync(bad.get(), 0, sizeof(uint32_t), st));
    shape_assign_kernel<<<(unsigned)ceil_div(nbr, 256), 256, 0, st>>>(m->brp, p.word.get(), p.rowrel.get(), p.desc.get(), nbr, cb, cv, cl,
                                                                      ss.get()->key, gv.get(), reinterpret_cast<const uint32_t*>(comb.get() + npal),
                                                                      srow.get(), bad.get());
    BMSP_KERNEL_CHECK();
    uint32_t hbad = 1;
    BMSP_CUDA(cudaMemcpyAsync(&hbad, bad.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));                // also the end of the pageable uploads above
    if (hbad) return BMSP_OK;
    p.palette = std::move(comb); p.rowrel = std::move(srow); p.word.reset();
    p.shapes = true; p.nshapes = ns; p.shape_words = (int32_t)words.size();
    return BMSP_OK;
}

// path 0 plan: tile descriptors, x lines and per-block x offsets; shared-memory capacities from the tile maxima
// when they fit the per-CTA budget, else from the averages (larger tiles are then read from global memory).
static int plan_tiles(const bmsp_matrix_s* m, SpmvPlan& p, cudaStream_t st) {
    const int vsize = (int)dtype_bytes(m->dtype);
    // tile height: 64 block rows unless an average tile (bitmaps, x offsets, values, ~x lines) would not fit ~20 KB
    int rt = 64;
    const double row_bytes = ((double)m->nblk * (8 + 2 + 16) + (double)m->nnz * vsize) / m->nbr + 8;
    while (rt > 16 && row_bytes * rt > 20.0 * 1024) rt >>= 1;
    // Light rows (64-block-row tiles: stencils, bands) stream through the persistent kernel, which runs STREAM_RT-row tiles only.
    // Heavy rows (dense blocks: 16- or 32-row tiles of 17 KB) are bound by the bit walk, not by memory: a stage then feeds only one
    // or two consumer warps and the one-CTA-per-tile kernel, which keeps 13 such tiles computing per SM, is faster (BC4M: 280 us vs
    // 479 us).  BMSP_SPMV_KERNEL=1 is a test hook: it puts the per-tile kernel behind a light matrix, the bit-exact reference of the
    // streaming kernel.
    const int kernel = (rt == STREAM_RT && env_int("BMSP_SPMV_KERNEL", 0) != 1) ? 0 : 1;
    const int xl_pitch = kernel == 1 ? XL_STRIDE : 32;
    const int ntiles = (int)ceil_div(m->nbr, rt);
    std::vector<uint4> pal;                    // kept until the synchronisation below (pageable source of the palette upload)
    if (kernel == 0) BMSP_TRY(build_palette(m, vsize, st, pal, p.palette));
    const int npal = p.npal = (int)pal.size();
    const bool use_pal = npal > 0;
    DevBuf<unsigned long long> stats;
    BMSP_TRY(p.desc.alloc((size_t)ntiles, st));
    BMSP_TRY(p.lines.alloc((size_t)m->nblk + 8, st));
    if (use_pal) {
        BMSP_TRY(p.word.alloc((size_t)m->nblk + 8, st));
        BMSP_TRY(p.rowrel.alloc((size_t)m->nbr + 8, st));
    } else {
        BMSP_TRY(p.xoff.alloc((size_t)m->nblk + 16, st));
        BMSP_TRY(p.rowpair.alloc((size_t)m->nbr + 1 + 8, st));
        zip_rows_kernel<<<(unsigned)ceil_div(m->nbr + 1, 256), 256, 0, st>>>(m->brp, m->rvb, m->nbr + 1, p.rowpair.get());
        BMSP_KERNEL_CHECK();
    }
    BMSP_TRY(stats.alloc(8, st));
    BMSP_CUDA(cudaMemsetAsync(stats.get(), 0, 8 * sizeof(unsigned long long), st));
    if (kernel == 0) {
        // tile-claim counters of the streaming kernel (zero before the plan's synchronisation below, so that no later launch -- on
        // whatever stream, captured in a graph or not -- has to wait for them)
        BMSP_TRY(p.sched.alloc((size_t)SCHED_SLOTS * 2, st));
        BMSP_CUDA(cudaMemsetAsync(p.sched.get(), 0, sizeof(int32_t) * SCHED_SLOTS * 2, st));
    }
    tile_plan_kernel<<<ntiles, 256, 0, st>>>(m->brp, m->bcol, m->rvb, m->nbr, m->cols, rt, xl_pitch, p.desc.get(), p.lines.get(),
                                             p.xoff.get(), stats.get(), m->bmps, p.palette.get(), npal, p.word.get(), p.rowrel.get());
    BMSP_KERNEL_CHECK();
    unsigned long long h[8];
    BMSP_CUDA(cudaMemcpyAsync(h, stats.get(), sizeof(h), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    stats.reset();
    // capacities: the tile maxima when they fit the per-CTA budget, else 1.25 x the averages (larger tiles are then
    // read from global memory by the kernel)
    auto up8 = [](long long v) { return (int)((v + 7) & ~7ll); };
    int cb = up8((long long)h[0]), cv = up8((long long)h[1]), cl = (int)h[2];
    const size_t budget = 40 * 1024;
    if (tile_smem(rt, cb, cv, cl, vsize, 4).total > budget) {
        const double ab = (double)m->nblk / ntiles, av = (double)m->nnz / ntiles, al = (double)h[3] / ntiles;
        cb = std::min(cb, up8((long long)(ab * 1.25) + 16)); cv = std::min(cv, up8((long long)(av * 1.25) + 64));
        cl = std::min(cl, (int)(al * 1.25) + 4);
        while (tile_smem(rt, cb, cv, cl, vsize, 4).total > budget && (cb > 64 || cv > 256 || cl > 16)) {
            cb = std::max(64, up8(cb * 3 / 4)); cv = std::max(256, up8(cv * 3 / 4)); cl = std::max(16, cl * 3 / 4);
        }
    }
    cb = std::max(cb, 8); cv = std::max(cv, 8);
    // the palette variant's relative row pairs are 16-bit: a staged tile has fewer than 65536 blocks and values (the 40 KB budget
    // above keeps both far below that already)
    if (use_pal) { cb = std::min(cb, 65528); cv = std::min(cv, 65528); }
    p.cap_blk = cb; p.cap_val = cv; p.cap_lines = std::max(cl, 1); p.tile_rows = rt; p.kernel = kernel;
    if (use_pal) BMSP_TRY(build_shapes(m, p, st));      // which tiles are staged is known from here on
    return BMSP_OK;
}

// block-parallel plan: work items of at most SLICE blocks (or bundles of four short block rows), and the list of sliced block rows
static int plan_block_parallel(const bmsp_matrix_s* m, SpmvPlan& p, cudaStream_t st) {
    p.path = SpmvPlan::BLOCK_PARALLEL;
    BMSP_TRY(p.item_ofs.alloc((size_t)m->nbr + 1, st));
    work_count_kernel<<<(unsigned)ceil_div(m->nbr, 256), 256, 0, st>>>(m->brp, m->nbr, p.item_ofs.get());
    BMSP_KERNEL_CHECK();
    BMSP_TRY(exclusive_scan_u32(p.item_ofs.get(), p.item_ofs.get(), m->nbr, st));
    uint32_t total = 0;
    BMSP_CUDA(cudaMemcpyAsync(&total, p.item_ofs.get() + m->nbr, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    BMSP_TRY(p.work.alloc((size_t)total, st));
    work_fill_kernel<<<(unsigned)ceil_div(m->nbr, 256), 256, 0, st>>>(m->brp, m->nbr, p.item_ofs.get(), p.work.get());
    BMSP_KERNEL_CHECK();
    // sliced block rows (more than one item): listed on the device.  (Items minus block rows no longer says whether there are any:
    // a bundle is one item for four block rows.)  A sliced row has at least two items, so there are at most total / 2 of them.
    const size_t cap = (size_t)total / 2 + 1;
    BMSP_TRY(p.split_list.alloc(cap + 1, st));
    int32_t* cntr = p.split_list.get() + cap;
    BMSP_CUDA(cudaMemsetAsync(cntr, 0, sizeof(int32_t), st));
    split_list_kernel<<<(unsigned)ceil_div(m->nbr, 256), 256, 0, st>>>((const int32_t*)p.item_ofs.get(), m->nbr, p.split_list.get(), cntr);
    BMSP_KERNEL_CHECK();
    BMSP_CUDA(cudaMemcpyAsync(&p.n_split_rows, cntr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    if (p.n_split_rows > 0) BMSP_TRY(p.split_partial.alloc((size_t)total * 8, st));
    p.n_work = (int32_t)total;
    return BMSP_OK;
}

// m->spmv, built on st by the first product and published only when complete.  m is neither transposed nor empty: the entry
// points reject those before they plan.
static int plan_spmv(bmsp_matrix_s* m, cudaStream_t st) {
    if (m->spmv) return BMSP_OK;
    std::unique_ptr<SpmvPlan> p(new SpmvPlan());
    BMSP_TRY(spmv_block_parallel(m) ? plan_block_parallel(m, *p, st) : plan_tiles(m, *p, st));
    m->spmv = p.release();
    return BMSP_OK;
}

// The plan's buffers free on the stream it was built on (DevBuf), not on the handle's last stream.  That is the same order:
// either the handle was used on that stream only, or bmsp_destroy synchronised the device before it calls this.
void spmv_release(bmsp_matrix_s* m) { delete m->spmv; m->spmv = nullptr; }

template <typename T, typename X, int RTT, int MINB, typename H>
static int launch_tile_kernel(const TileArgs<T>& a, const X* x, float* y, const H& hd, int grid, size_t smem, cudaStream_t st) {
    auto kern = spmv_tile_kernel<T, X, RTT, MINB, H>;
    BMSP_TRY(kernel_smem((const void*)kern, smem, true));
    kern<<<(unsigned)grid, RTT * 2, smem, st>>>(a, x, y, hd);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

// Streaming kernel launch.  STREAM_CTAS bounds the CTAs per SM the registers allow.  Shared memory decides the rest: as many CTAs
// per SM as fit with two stages each (a CTA needs a second stage to have its next tile arriving while it multiplies the current
// one; P4096: 7 CTAs x 2 stages of 15.4 KB -- the measured optimum, see DESIGN.md section 7).
// The last STREAM_DYN_PCT per cent of every CTA's share are claimed at run time (P4096: 0 % 68.6 us, 12-25 % 66.5 us, 50 % 67.6 us,
// 100 % 75.6 us -- 32 768 atomics on one address are too many).
constexpr int STREAM_DYN_PCT = 25;
template <typename T, typename X, typename H, bool PAL, bool SHP>
static int launch_stream_kernel(const TileArgs<T>& a, const X* x, float* y, const H& hd, int ntiles, cudaStream_t st, int32_t* sched) {
    auto kern = spmv_stream_kernel<T, X, H, PAL, SHP>;
    const DeviceInfo* dev = nullptr;
    BMSP_TRY(current_device(&dev));
    StreamArgs<T> sa;
    sa.t = a;
    sa.so = stage_layout(a.cap_blk, a.cap_val, a.cap_lines, sizeof(T), sizeof(X), PAL, SHP);
    sa.ntiles = ntiles;
    // descriptor ring (+ palette, + shape table)
    const size_t fixed = (size_t)STREAM_DR * 64 + 64 + (PAL ? 16 + (size_t)a.npal * 16 : 0) + (SHP ? (size_t)a.shape_words * 4 : 0);
    const size_t per_stage = (size_t)sa.so.stride + 16;
    int ctas = 0, spg = 0;
    size_t per_cta = 0;
    for (int c = STREAM_CTAS; c >= 1; c--) {
        per_cta = std::min<size_t>(dev->smem_per_sm / c - 1024 - 256, 227 * 1024);   // 1 KB per resident CTA is the system's; 256 B allocation granule
        const int fit = per_cta > fixed ? (int)((per_cta - fixed) / per_stage) : 0;
        if (fit >= 2 || (c == 1 && fit >= 1)) { ctas = c; spg = std::min(fit, 8); break; }
    }
    if (ctas < 1 || spg < 1) { set_error("spmv: a tile stage of %u bytes does not fit shared memory", sa.so.stride); return BMSP_ERR_CUDA; }
    sa.spg = spg;
    const size_t smem = (size_t)spg * per_stage + fixed;
    BMSP_TRY(kernel_smem((const void*)kern, smem, true));
    const int grid = std::max(1, std::min(ntiles, dev->sms * ctas));
    const int share = ntiles / grid;
    sa.sched = (sched && share >= 2) ? sched : nullptr;
    sa.n_static = sa.sched ? (int)((int64_t)share * (100 - STREAM_DYN_PCT) / 100) : 0;
    kern<<<(unsigned)grid, 32 + STREAM_RT * 2, smem, st>>>(sa, x, y, hd);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

// tile0 / ntiles: row-tiled path only -- launch the tiles [tile0, tile0 + ntiles) (ntiles < 0: all of them).
// hd: NoHalo, or HaloDev for the fused multi-GPU product (row-tiled path, fp32 x, all tiles).
template <typename T, typename X, typename H = NoHalo>
static int launch_spmv(const bmsp_matrix_s* A, SpmvPlan& p, const X* x, float* y, cudaStream_t st, int tile0 = 0, int ntiles = -1, const H& hd = H()) {
    if (p.path == SpmvPlan::ROW_TILED) {
        TileArgs<T> a;
        a.tile0 = tile0;
        a.bmps = A->bmps; a.bcol = A->bcol; a.values = (const T*)A->values; a.rowpair = p.rowpair.get();
        a.desc = p.desc.get(); a.lines = p.lines.get(); a.xoff = p.xoff.get();
        a.word = p.word.get(); a.rowrel = p.rowrel.get(); a.palette = p.palette.get(); a.npal = p.npal; a.shape_words = p.shape_words;
        a.brp = A->brp; a.rvb = A->rvb;
        a.rows = A->rows; a.nbr = A->nbr; a.cols = A->cols; a.cap_blk = p.cap_blk; a.cap_val = p.cap_val; a.cap_lines = p.cap_lines;
        const int rt = p.tile_rows;
        a.so = tile_smem(rt, a.cap_blk, a.cap_val, a.cap_lines, sizeof(T), sizeof(X));
        const size_t smem = a.so.total;
        const int grid = ntiles < 0 ? (int)ceil_div(A->nbr, rt) : ntiles;
        if (grid <= 0) return BMSP_OK;
        if (p.kernel == 0) {
            // streaming kernel (tile_rows == STREAM_RT, plan_tiles).  A launch over all tiles takes one of the matrix's scheduler
            // slots in turn (launches on different streams may overlap: they must not share a counter); launches over a tile range
            // (the host-buffer pipeline's chunks) keep static shares.
            int32_t* sched = ntiles < 0 ? p.sched.get() + 2 * (p.sched_next++ % SCHED_SLOTS) : nullptr;
            if (p.shapes) return launch_stream_kernel<T, X, H, true, true>(a, x, y, hd, grid, st, sched);
            if (p.npal > 0) return launch_stream_kernel<T, X, H, true, false>(a, x, y, hd, grid, st, sched);
            return launch_stream_kernel<T, X, H, false, false>(a, x, y, hd, grid, st, sched);
        }
        if (rt == 32) return launch_tile_kernel<T, X, 32, 24, H>(a, x, y, hd, grid, smem, st);
        if (rt == 16) return launch_tile_kernel<T, X, 16, 32, H>(a, x, y, hd, grid, smem, st);
        return launch_tile_kernel<T, X, 64, 12, H>(a, x, y, hd, grid, smem, st);
    }
    const unsigned grid1 = (unsigned)ceil_div(p.n_work, 8), grid2 = (unsigned)ceil_div((int64_t)p.n_split_rows * 32, 256);
    spmv_blockpar_kernel<T, X><<<grid1, 256, 0, st>>>(A->bmps, A->bcol, A->offsets, (const T*)A->values, p.work.get(), p.n_work,
                                                    A->rows, x, y, p.split_partial.get(), A->brp);
    BMSP_KERNEL_CHECK();
    if (p.n_split_rows > 0) {
        spmv_fixup_kernel<<<grid2, 256, 0, st>>>((const int32_t*)p.item_ofs.get(), p.split_partial.get(), p.split_list.get(),
                                                 p.n_split_rows, A->rows, y);
        BMSP_KERNEL_CHECK();
    }
    return BMSP_OK;
}

// chunks of the host-buffer pipeline.  P4096 on PCIe 5 x16: 8 chunks 1.67 ms, 16: 1.68, 32: 1.84 (per-chunk dependencies cost
// more than the shorter fill saves)
constexpr int HOST_CHUNKS = 8;

// A's pipeline, built on the first call and published in the plan only when complete
static int host_pipe_get(const bmsp_matrix_s* A, SpmvPlan& p, cudaStream_t st) {
    if (p.host) return BMSP_OK;
    std::unique_ptr<HostPipe> hp(new HostPipe());
    BMSP_TRY(new_stream(hp->s_in));
    BMSP_TRY(new_stream(hp->s_out));
    BMSP_TRY(new_event(hp->ev_start));
    BMSP_TRY(new_event(hp->ev_done));
    BMSP_TRY(hp->x_dev.alloc((size_t)A->cols * 4 + 256, st));
    BMSP_TRY(hp->y_dev.alloc((size_t)A->rows + 64, st));
    BMSP_TRY(new_stream(hp->s_cap));
    if (p.path == SpmvPlan::ROW_TILED && (int64_t)A->rows * 4 >= (1 << 20)) {
        const int rt = p.tile_rows, ntiles = (int)ceil_div(A->nbr, rt);
        std::vector<TileDesc> desc((size_t)ntiles);
        BMSP_CUDA(cudaMemcpyAsync(desc.data(), p.desc.get(), sizeof(TileDesc) * (size_t)ntiles, cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
        const int nch = std::min(HOST_CHUNKS, ntiles), per = (int)ceil_div(ntiles, nch);
        int64_t need = 0;
        for (int t0 = 0; t0 < ntiles; t0 += per) {
            const int t1 = std::min(ntiles, t0 + per);
            for (int t = t0; t < t1; t++)
                if (desc[t].nb > 0) need = std::max(need, std::min<int64_t>(A->cols, ((int64_t)desc[t].lmax + 1) * 32));
            hp->tile_lo.push_back(t0);
            hp->x_need.push_back(need);
        }
        hp->tile_lo.push_back(ntiles);
    } else {
        // one chunk: all tiles of a row-tiled matrix (ADVICE r1: {0, 0} launched nothing and left y_host untouched); the
        // block-parallel path ignores tile_lo
        hp->tile_lo = {0, p.path == SpmvPlan::ROW_TILED ? (int)ceil_div(A->nbr, p.tile_rows) : 0};
        hp->x_need = {(int64_t)A->cols};
    }
    hp->ev_x.resize(hp->x_need.size()); hp->ev_k.resize(hp->x_need.size());
    for (auto& e : hp->ev_x) BMSP_TRY(new_event(e));
    for (auto& e : hp->ev_k) BMSP_TRY(new_event(e));
    p.host = std::move(hp);
    return BMSP_OK;
}

// y can leave without a copy engine: when y_host is pinned (and therefore mapped into the device's address space) the
// row-range launches store their float4 results straight into it over PCIe (posted writes), so the pipeline is
// H2D slices of x on s_in against kernels that write host memory -- no D2H copies, no events per chunk on the way out.
static float* mapped_host_ptr(float* y_host) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, y_host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer || ((uintptr_t)at.devicePointer & 15)) return nullptr;
    return (float*)at.devicePointer;
}

template <typename T>
static int spmv_host_run(const bmsp_matrix_s* A, SpmvPlan& p, const void* x_host, int32_t x_dtype, float* y_host, cudaStream_t st) {
    HostPipe* hp = p.host.get();
    const size_t xs = dtype_bytes(x_dtype);
    float* y_map = p.path == SpmvPlan::ROW_TILED ? mapped_host_ptr(y_host) : nullptr;     // row-tiled kernel only: it stores 512 contiguous bytes per warp
    float* y_out = y_map ? y_map : hp->y_dev.get();
    BMSP_CUDA(cudaEventRecord(hp->ev_start.get(), st));         // earlier work on st (and the previous call) is done with x_dev / y_dev
    BMSP_CUDA(cudaStreamWaitEvent(hp->s_in.get(), hp->ev_start.get(), 0));
    BMSP_CUDA(cudaStreamWaitEvent(hp->s_out.get(), hp->ev_start.get(), 0));
    int64_t sent = 0;
    const int64_t rows_per_tile = (int64_t)p.tile_rows * 8;
    for (int c = 0; c < (int)hp->x_need.size(); c++) {
        const int64_t need = hp->x_need[c];
        if (need > sent) {
            BMSP_CUDA(cudaMemcpyAsync(hp->x_dev.get() + sent * xs, (const char*)x_host + sent * xs, (size_t)(need - sent) * xs,
                                      cudaMemcpyHostToDevice, hp->s_in.get()));
            BMSP_CUDA(cudaEventRecord(hp->ev_x[c].get(), hp->s_in.get()));
            BMSP_CUDA(cudaStreamWaitEvent(st, hp->ev_x[c].get(), 0));
            sent = need;
        }
        int64_t row0 = 0, row1 = A->rows;
        int t0 = 0, nt = -1;                               // block-parallel path: the whole matrix
        if (p.path == SpmvPlan::ROW_TILED) {
            const int t1 = hp->tile_lo[c + 1];
            t0 = hp->tile_lo[c]; nt = t1 - t0;
            row0 = std::min<int64_t>(A->rows, t0 * rows_per_tile); row1 = std::min<int64_t>(A->rows, t1 * rows_per_tile);
        }
        BMSP_TRY(with_value_type(x_dtype, [&](auto x) {
            using X = decltype(x);
            return launch_spmv<T, X>(A, p, (const X*)hp->x_dev.get(), y_out, st, t0, nt);
        }));
        if (row1 > row0 && !y_map) {
            BMSP_CUDA(cudaEventRecord(hp->ev_k[c].get(), st));
            BMSP_CUDA(cudaStreamWaitEvent(hp->s_out.get(), hp->ev_k[c].get(), 0));
            BMSP_CUDA(cudaMemcpyAsync(y_host + row0, hp->y_dev.get() + row0, (size_t)(row1 - row0) * 4, cudaMemcpyDeviceToHost, hp->s_out.get()));
        }
    }
    BMSP_CUDA(cudaEventRecord(hp->ev_done.get(), hp->s_out.get()));
    BMSP_CUDA(cudaStreamWaitEvent(st, hp->ev_done.get(), 0));   // the caller synchronises `st` as for bmsp_spmv
    return BMSP_OK;
}

// Second call with the same pinned buffers: capture the pipeline once (origin stream s_cap, forks into s_in / s_out, all
// joined before the capture ends) and replay it with one cudaGraphLaunch on the caller's stream from then on.
template <typename T>
static int spmv_host_graph(const bmsp_matrix_s* A, SpmvPlan& p, const void* x_host, int32_t x_dtype, float* y_host, cudaStream_t st, bool* used) {
    HostPipe* hp = p.host.get();
    *used = false;
    if (!(hp->gexec && hp->g_x == x_host && hp->g_y == y_host && hp->g_xdt == x_dtype)) {
        const bool again = hp->seen_x == x_host && hp->seen_y == y_host && hp->seen_xdt == x_dtype;
        hp->seen_x = x_host; hp->seen_y = y_host; hp->seen_xdt = x_dtype;
        if (!again) return BMSP_OK;                        // first sight of these buffers: run eagerly
        cudaPointerAttributes ax, ay;
        if (cudaPointerGetAttributes(&ax, x_host) != cudaSuccess || cudaPointerGetAttributes(&ay, y_host) != cudaSuccess ||
            ax.type != cudaMemoryTypeHost || ay.type != cudaMemoryTypeHost) { cudaGetLastError(); return BMSP_OK; }   // pageable: eager only
        hp->gexec.reset();
        cudaGraph_t graph = nullptr;
        BMSP_CUDA(cudaStreamBeginCapture(hp->s_cap.get(), cudaStreamCaptureModeThreadLocal));
        const int rc = spmv_host_run<T>(A, p, x_host, x_dtype, y_host, hp->s_cap.get());
        const cudaError_t ce = cudaStreamEndCapture(hp->s_cap.get(), &graph);
        if (rc != BMSP_OK || ce != cudaSuccess || !graph) { cudaGetLastError(); if (graph) cudaGraphDestroy(graph); return BMSP_OK; }
        cudaGraphExec_t ge = nullptr;
        const cudaError_t ie = cudaGraphInstantiate(&ge, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); return BMSP_OK; }
        hp->gexec.reset(ge);
        hp->g_x = x_host; hp->g_y = y_host; hp->g_xdt = x_dtype;
    }
    BMSP_CUDA(cudaGraphLaunch(hp->gexec.get(), st));
    *used = true;
    return BMSP_OK;
}

}  // namespace bmsp

using namespace bmsp;

extern "C" int bmsp_spmv_host(bmsp_matrix_t A, const void* x_host, int32_t x_dtype, float* y_host, void* stream) {
    if (!A || !x_host || !y_host || (x_dtype != BMSP_F16 && x_dtype != BMSP_F32)) { set_error("bmsp_spmv_host: invalid argument"); return BMSP_ERR_INVALID; }
    if (A->transposed) { set_error("bmsp_spmv_host: matrix is in transposed-operand form"); return BMSP_ERR_UNSUPPORTED; }
    if (A->rows == 0) return BMSP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    BMSP_TRY(plan_spmv(A, st));
    SpmvPlan& p = *A->spmv;
    BMSP_TRY(host_pipe_get(A, p, st));
    return with_value_type(A->dtype, [&](auto t) -> int {
        using T = decltype(t);
        bool replayed = false;
        BMSP_TRY(spmv_host_graph<T>(A, p, x_host, x_dtype, y_host, st, &replayed));
        return replayed ? BMSP_OK : spmv_host_run<T>(A, p, x_host, x_dtype, y_host, st);
    });
}

namespace bmsp {

// ---- multi-GPU product with the halo exchange over peer memory ---------------------------------------------------
static int halo_to_dev(const bmsp_halo_desc* d, int rows, HaloDev* h) {
    if (!d || d->n_push < 0 || d->n_push > HALO_MAX || d->n_peer < 0 || d->n_peer > HALO_MAX || (d->n_peer > 0 && !d->scratch)) {
        set_error("halo descriptor: bad counts or missing scratch"); return BMSP_ERR_INVALID;
    }
    // n_peer is the union of both directions: a rank that pushes rows has at least the peers it pushes to.  Without this check
    // such a descriptor would silently push nothing (bmsp_spmv_halo takes the plain product, bmsp_halo_push returns at once).
    if (d->n_push > 0 && d->n_peer == 0) { set_error("halo descriptor: push ranges without peers"); return BMSP_ERR_INVALID; }
    memset(h, 0, sizeof(*h));
    h->n_push = 0; h->n_peer = d->n_peer; h->scratch = (uint32_t*)d->scratch; h->solo_tile = -1;
    h->own_c0 = d->own_col_lo; h->own_c1 = d->own_col_hi;
    for (int i = 0; i < d->n_push; i++) {
        if (d->push_lo[i] < 0 || d->push_hi[i] > rows || d->push_lo[i] > d->push_hi[i] || (d->push_lo[i] & 3) || ((uintptr_t)d->push_dst[i] & 15)) {
            set_error("halo descriptor: push range %d [%d,%d) invalid or misaligned", i, d->push_lo[i], d->push_hi[i]); return BMSP_ERR_INVALID;
        }
        if (d->push_lo[i] == d->push_hi[i]) continue;      // an empty range pushes nothing and must not count as a signalling tile
        const int k = h->n_push++;
        h->lo[k] = d->push_lo[i]; h->hi[k] = d->push_hi[i]; h->dst[k] = (float*)d->push_dst[i];
    }
    for (int i = 0; i < d->n_peer; i++) { h->peer_flag[i] = (uint32_t*)d->peer_flag[i]; h->my_flag[i] = (const uint32_t*)d->my_flag[i]; }
    return BMSP_OK;
}

}  // namespace bmsp
using namespace bmsp;

extern "C" int bmsp_halo_push(const float* y_own, int32_t rows, const bmsp_halo_desc* halo, uint32_t signal_epoch, void* stream) {
    if (!y_own && rows > 0) { set_error("bmsp_halo_push: null vector"); return BMSP_ERR_INVALID; }
    HaloDev h;
    BMSP_TRY(halo_to_dev(halo, rows, &h));
    if (h.n_peer == 0) return BMSP_OK;
    int lo_all = 0x7FFFFFFF, hi_all = 0;
    for (int i = 0; i < h.n_push; i++) { lo_all = std::min(lo_all, h.lo[i]); hi_all = std::max(hi_all, h.hi[i]); }
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div((int64_t)std::max(0, hi_all - lo_all), 1024), 592));
    h.signal_epoch = signal_epoch; h.n_sig = (uint32_t)grid;
    halo_push_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(y_own, rows, h);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

extern "C" int bmsp_halo_status(const bmsp_halo_desc* halo, void* stream, int32_t* timed_out) {
    if (!halo || !timed_out) { set_error("bmsp_halo_status: null argument"); return BMSP_ERR_INVALID; }
    uint32_t v[2] = {0, 0};
    if (halo->scratch) {
        BMSP_CUDA(cudaMemcpyAsync(v, halo->scratch, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        BMSP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    }
    *timed_out = (int32_t)v[1];
    return BMSP_OK;
}

extern "C" int bmsp_spmv_halo(bmsp_matrix_t A, const float* x_ext, float* y_own, const bmsp_halo_desc* halo, uint32_t wait_epoch,
                              uint32_t signal_epoch, void* stream) {
    // a rank that owns no rows (an empty shard) reads and writes no vector: its x and y may be empty tensors (null pointers)
    if (!A || (A->rows > 0 && (!x_ext || !y_own))) { set_error("bmsp_spmv_halo: null argument"); return BMSP_ERR_INVALID; }
    if (A->transposed) { set_error("bmsp_spmv_halo: matrix is in transposed-operand form"); return BMSP_ERR_UNSUPPORTED; }
    if (((uintptr_t)x_ext & 15) || ((uintptr_t)y_own & 15)) { set_error("bmsp_spmv_halo: x and y must be 16-byte aligned"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    HaloDev h;
    BMSP_TRY(halo_to_dev(halo, A->rows, &h));
    h.wait_epoch = wait_epoch; h.signal_epoch = signal_epoch;
    // no rows: nothing to wait for or push, but the peers wait for this rank's epoch
    if (A->rows == 0) return h.n_peer == 0 ? BMSP_OK : bmsp_halo_push(y_own, 0, halo, signal_epoch, stream);
    if (h.n_peer == 0) return bmsp_spmv(A, x_ext, BMSP_F32, y_own, stream);
    BMSP_TRY(plan_spmv(A, st));
    SpmvPlan& p = *A->spmv;
    if (p.path == SpmvPlan::ROW_TILED) {
        // One launch of the halo variant over all tiles.  Running the tiles that wait or push in a launch of their own ahead of the
        // plain kernel over the rest was slower on P4096 (one GPU as its own peer): 85.7 us on the same stream (the small launch is
        // all latency) and 79.5 us on a side stream, against 69.7 us.
        // tiles that own pushed rows (union of the ranges' tile intervals); they count down to the signal
        const int64_t rpt = (int64_t)p.tile_rows * 8;
        std::vector<std::pair<int64_t, int64_t>> iv;
        for (int i = 0; i < h.n_push; i++) if (h.hi[i] > h.lo[i]) iv.push_back({h.lo[i] / rpt, (h.hi[i] - 1) / rpt});
        std::sort(iv.begin(), iv.end());
        int64_t n = 0, reach = -1;
        h.n_iv = 0;
        for (auto& p : iv) {
            const int64_t a0 = std::max(p.first, reach + 1);
            if (p.second >= a0) { n += p.second - a0 + 1; reach = p.second; h.iv_lo[h.n_iv] = (int32_t)a0; h.iv_hi[h.n_iv] = (int32_t)p.second; h.n_iv++; }
        }
        if (n == 0) { h.solo_tile = 0; n = 1; }
        h.n_sig = (uint32_t)n;
        h.rot = (int)(ceil_div(A->nbr, p.tile_rows) / 2);
        return with_value_type(A->dtype, [&](auto t) { return launch_spmv<decltype(t), float, HaloDev>(A, p, x_ext, y_own, st, 0, -1, h); });
    }
    // block-parallel path: wait kernel, product, push kernel
    halo_wait_kernel<<<1, 32, 0, st>>>(h);
    BMSP_KERNEL_CHECK();
    BMSP_TRY(bmsp_spmv(A, x_ext, BMSP_F32, y_own, stream));
    return bmsp_halo_push(y_own, A->rows, halo, signal_epoch, stream);
}

// ---- peer-mapped device memory for the halo buffers (one process per GPU: CUDA IPC handles travel through the caller) ----
extern "C" int bmsp_peer_alloc(int64_t bytes, void** ptr, void* handle64) {
    if (!ptr || !handle64 || bytes <= 0) { set_error("bmsp_peer_alloc: invalid argument"); return BMSP_ERR_INVALID; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    *ptr = nullptr;
    BMSP_CUDA(cudaMalloc(ptr, (size_t)bytes));          // IPC needs a plain allocation, not the stream-ordered pool
    BMSP_CUDA(cudaMemset(*ptr, 0, (size_t)bytes));
    cudaIpcMemHandle_t hd;
    BMSP_CUDA(cudaIpcGetMemHandle(&hd, *ptr));
    memcpy(handle64, &hd, 64);
    return BMSP_OK;
}
extern "C" int bmsp_peer_open(const void* handle64, void** ptr) {
    if (!ptr || !handle64) { set_error("bmsp_peer_open: invalid argument"); return BMSP_ERR_INVALID; }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle64, 64);
    *ptr = nullptr;
    BMSP_CUDA(cudaIpcOpenMemHandle(ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    return BMSP_OK;
}
extern "C" int bmsp_peer_close(void* ptr) { if (ptr) BMSP_CUDA(cudaIpcCloseMemHandle(ptr)); return BMSP_OK; }
extern "C" int bmsp_peer_free(void* ptr) { if (ptr) BMSP_CUDA(cudaFree(ptr)); return BMSP_OK; }

extern "C" int bmsp_spmv(bmsp_matrix_t A, const void* x, int32_t x_dtype, float* y, void* stream) {
    if (!A || !x || !y || (x_dtype != BMSP_F16 && x_dtype != BMSP_F32)) { set_error("bmsp_spmv: invalid argument"); return BMSP_ERR_INVALID; }
    if (A->transposed) { set_error("bmsp_spmv: matrix is in transposed-operand form"); return BMSP_ERR_UNSUPPORTED; }
    if (A->rows == 0) return BMSP_OK;
    if (((uintptr_t)x & 15) || ((uintptr_t)y & 15)) { set_error("bmsp_spmv: x and y must be 16-byte aligned"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    BMSP_TRY(plan_spmv(A, st));
    return with_value_type(A->dtype, [&](auto t) { return with_value_type(x_dtype, [&](auto xt) {
        using X = decltype(xt);
        return launch_spmv<decltype(t), X>(A, *A->spmv, (const X*)x, y, st);
    }); });
}

// SURVEY.md section 8(d): nblk*(4+8) + nbr*(4+4) + nnz*sizeof(value) + ncols*sizeof(x) + nrows*4
extern "C" int bmsp_spmv_bytes(bmsp_matrix_t A, int32_t x_dtype, int64_t* bytes) {
    if (!A || !bytes) { set_error("bmsp_spmv_bytes: null argument"); return BMSP_ERR_INVALID; }
    *bytes = A->nblk * 12 + (int64_t)A->nbr * 8 + A->nnz * (int64_t)dtype_bytes(A->dtype) + (int64_t)A->cols * (int64_t)dtype_bytes(x_dtype) +
             (int64_t)A->rows * 4;
    return BMSP_OK;
}

extern "C" int bmsp_debug_spmv_plan(bmsp_matrix_t A, bmsp_spmv_plan_info* out, void* stream) {
    if (!A || !out) { set_error("bmsp_debug_spmv_plan: null argument"); return BMSP_ERR_INVALID; }
    if (A->transposed || A->rows == 0) { set_error("bmsp_debug_spmv_plan: the matrix is transposed or empty"); return BMSP_ERR_UNSUPPORTED; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    BMSP_TRY(plan_spmv(A, st));
    const SpmvPlan& p = *A->spmv;
    memset(out, 0, sizeof(*out));
    if (p.path == SpmvPlan::BLOCK_PARALLEL) {
        out->path = 1;
        out->n_work = p.n_work; out->n_split_rows = p.n_split_rows;
        std::vector<int4> work((size_t)p.n_work);
        if (p.n_work > 0) BMSP_CUDA(cudaMemcpyAsync(work.data(), p.work.get(), sizeof(int4) * work.size(), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
        for (const int4& w : work) out->n_bundles += w.w == 2;
        return BMSP_OK;
    }
    out->kernel = p.kernel; out->tile_rows = p.tile_rows; out->npal = p.npal;
    out->cap_blk = p.cap_blk; out->cap_val = p.cap_val; out->cap_lines = p.cap_lines;
    const int ntiles = out->ntiles = (int)ceil_div(A->nbr, p.tile_rows);
    std::vector<TileDesc> desc((size_t)ntiles);
    BMSP_CUDA(cudaMemcpyAsync(desc.data(), p.desc.get(), sizeof(TileDesc) * desc.size(), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    for (const TileDesc& d : desc) {
        out->empty_tiles += d.nb == 0;
        out->tail_line_tiles += (d.flags & 2) != 0;
        if (!(d.flags & 1)) {
            out->unplanned_tiles++;
            if (d.nb > PLAN_MAXB) out->unplanned_blocks++;
            else if (d.nl > XL_MAX) out->unplanned_lines++;
            continue;
        }
        out->over_cap_tiles += d.nb > p.cap_blk || d.nv > p.cap_val || d.nl > p.cap_lines;
        if (d.nb > 0) out->runs[d.nruns]++;
    }
    return BMSP_OK;
}

extern "C" int bmsp_debug_spmv_shapes(bmsp_matrix_t A, int32_t* nshapes, int32_t* nwords, void* stream) {
    if (!A || !nshapes || !nwords) { set_error("bmsp_debug_spmv_shapes: null argument"); return BMSP_ERR_INVALID; }
    if (A->transposed || A->rows == 0) { set_error("bmsp_debug_spmv_shapes: the matrix is transposed or empty"); return BMSP_ERR_UNSUPPORTED; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(A, st);
    BMSP_TRY(plan_spmv(A, st));
    const SpmvPlan& p = *A->spmv;
    *nshapes = p.shapes ? p.nshapes : -1;
    *nwords = p.shapes ? p.shape_words : -1;
    return BMSP_OK;
}
