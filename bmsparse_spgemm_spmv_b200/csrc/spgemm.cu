// spgemm.cu -- C = A * B on the bmSparse form (A plain fp16, B in transposed-operand form fp16, C plain fp32).
//
// Replaces bmSparse_mult (src/bmSparse_SPGEMM.cu:827-1223).  The reference materialises every candidate
// (A-block, B-block) pair as a 16-byte task (T_3), filters them with 64 AND-tests each (T_4), sorts the
// survivors by C key with an indirect comparator or bb_segsort (T_5), and runs ~20 thrust passes over
// the task list before its numeric kernel.  Here nothing is materialised and nothing is sorted:
//
//   row-wise (Gustavson) over A's block rows, one CTA per block row (dynamic queue), three passes
//     COUNT   candidates are tested four at a time (one 32-bit load of B's inner-dimension masks against the
//             replicated mask of the A block); survivors set a bit in a per-row bit set over C's block
//             columns                                   -> C blocks and survivors per block row  (T_1..T_4)
//     FILL    same walk; survivors are also appended to a global pair list (8 B each -- the only thing that
//             is materialised, after the filter, never sorted).  The bit set is ranked by a popc prefix: the
//             rank of column j IS its sorted position, so C.keys come out ascending without a sort
//             (replaces T_5/T_6 and bb_segsort); the boolean 8x8 product of the operand bitmaps is OR-ed
//             into the block's bitmap; value offsets are scanned per row                              (T_9)
//     NUMERIC bit set rebuilt from C.keys; the pair list is multiplied (scalar lanes for sparse blocks,
//             mma.sync m16n8k8 fp16->fp32 for dense blocks, two B blocks per MMA) and accumulated in
//             shared memory, then stored coalesced                                                    (T_7)
//   block rows whose bit set / block list / value list exceed the shared-memory caps run the same
//   code on global scratch.
#include "common.cuh"
#include <vector>
#include <algorithm>

namespace bmsp {

// the passes; as the template argument of apply_pair, drain and enumerate_row: what is done with a surviving pair
enum { PASS_COUNT = 0, PASS_FILL = 1, PASS_NUMERIC = 2, PASS_NUMERIC_MMA = 3 };
constexpr int QSLOTS = 192;   // per-warp queue: 64 pairs (uint2) + 32 staged PairMeta (32 B each) for the MMA drain

// Counters and maxima the kernels reduce into: one device allocation per product, zeroed first, read back by field.
struct Counters {
    int32_t max_words;              // rowinfo_kernel: the widest bit set of a block row, in 32-bit words
    int32_t max_c_item;             // COUNT: the most C blocks of a work item (sizes FILL's shared C block stage)
    int32_t max_nnz_item;           // FILL: the most C values of a work item
    int32_t max_c_row;              // COUNT: the most C blocks of a block row (the MMA pass runs row by row)
    int32_t queue[2];               // work-queue heads: the main launch, the heavy-row launch
    unsigned long long surviving;   // COUNT: surviving pairs
    unsigned long long sum_words;   // rowinfo_kernel: bit-set words over all block rows
    unsigned long long max_cand;    // rowinfo_kernel: the most candidate pairs of a block row
    unsigned long long sum_cand;    // rowinfo_kernel: candidate pairs
};

struct GemmArgs {
    const int32_t* a_brp; const int32_t* a_bcol; const uint64_t* a_bmps; const uint8_t* a_kmask; const uint64_t* a_off; const __half* a_val;
    const int32_t* b_brp; const int32_t* b_bcol; const uint64_t* b_bmps; const uint8_t* b_kmask; const uint64_t* b_off; const __half* b_val;
    const uint4* b_pm;         // packed per-B-block records, two uint4 each: {bitmap lo, bitmap hi, block column, value offset}, {first 8 values}
    // fine index of B (sparse-block operands; null: candidate scan): bucket (k, t) = the blocks of B's block row k whose kmask has
    // bit t, i.e. that have something in row 8k + (inner index of bit t).  An A block with kmask `am` meets exactly the blocks of
    // the buckets (bcol(a), t), t in am -- read as contiguous runs instead of found by testing every block of the B block row.
    const uint32_t* f_ptr; const uint32_t* f_bcol; const uint8_t* f_kmask; const uint4* f_rec;
    const int2* rowinfo;       // per A block row: x = first C block column of the bit set (multiple of 32), y = words
    int32_t row_begin, row_end;
    int32_t G;                 // lanes cooperating on one A block (power of two <= 32)
    int32_t cap_words, cap_c, cap_nnz;
    uint32_t* g_bitset; uint32_t* g_wrank; int32_t max_words;   // per-CTA global scratch for over-cap rows
    int32_t* work_counter;
    const int32_t* row_list;   // when set: the rows to process, in this order (heavy-row / light-row launches); else row_begin + i
    int32_t n_list;
    int32_t batch;             // work items a CTA takes from the queue per atomic (tiny rows: the queue head would serialise the launch)
    int32_t sort_max;          // FILL: leave a work item's segment of the pair list sorted by pair class (see pair_class) when it has at
                               // most this many pairs (0: never; SORT_K x the smallest CTA of the pass: a thread keeps its pairs in registers)
    int32_t split8;            // NUMERIC: 8 lanes per surviving pair, one per row of the A block (blocks with >= 4 values: a lane
                               // that multiplies a whole pair alone walks up to 64 x 8 dependent loads)
    int32_t group;             // consecutive block rows per work item (1..32): tiny rows are processed a group at a time -- one bit set, one
                               // pair-list segment, one set of accumulators for the group -- so that a CTA has hundreds of pairs in flight
    uint32_t* row_count;       // COUNT out: C blocks per row (indexed row - row_begin)
    uint32_t* row_surv;        // COUNT out: surviving pairs per row; FILL/NUMERIC in: exclusive scan of it
    uint2* surv_list;          // FILL out / NUMERIC in: (A block, B block) of every surviving pair, row-segmented
    Counters* ctr;
    const int32_t* c_brp;      // FILL/NUMERIC in: C block-row pointers (indexed row - row_begin)
    uint64_t* c_keys; uint64_t* c_bmps; int32_t* c_bcol; uint8_t* c_kmask;
    uint64_t* c_off;           // FILL out: value offsets relative to the row; NUMERIC: rebased to absolute
    uint64_t* row_nnz;         // FILL out: values per row; NUMERIC in: exclusive scan of it (row value base)
    float* c_val;
};

// boolean 8x8 product of an A bitmap (row-major) and a B bitmap in transposed-operand form:
// bit (i,j) = (row i of A) & (byte j of Bt) != 0   -- bmp_calculator, SPGEMM.cu:787-810
// Two evaluations: blocks with few cells (uniform-random and R-MAT inputs average ~1.1 per block) walk A's set bits --
// cell (i,k) contributes column k of B, i.e. bit k of every byte of bt, gathered into one byte by a multiply -- about 8
// instructions per cell; denser blocks take the row-wise SWAR form (8 rows x ~14 instructions whatever the fill).
__device__ __forceinline__ uint64_t pair_bitmap_dense(uint64_t a, uint64_t bt);
__device__ __forceinline__ uint64_t pair_bitmap(uint64_t a, uint64_t bt) {
    if (__popcll(a) > 8) return pair_bitmap_dense(a, bt);
    uint64_t res = 0;
    while (a) {
        const int p = __clzll((long long)a);
        a &= ~(0x8000000000000000ull >> p);
        const int i = p >> 3, k = p & 7;
        const uint64_t col = (bt >> (7 - k)) & 0x0101010101010101ull;           // B(k, j) in bit 0 of byte j (from the MSB)
        res |= ((col * 0x0102040810204080ull) >> 56) << (56 - 8 * i);           // gathered: j = 0 lands in the byte's MSB
    }
    return res;
}
__device__ __forceinline__ uint64_t pair_bitmap_dense(uint64_t a, uint64_t bt) {
    const uint32_t bh = (uint32_t)(bt >> 32), bl = (uint32_t)bt;
    uint64_t res = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t ai = (uint32_t)(a >> (56 - 8 * i)) & 0xFFu;
        const uint32_t rep = ai * 0x01010101u;
        const uint32_t th = rep & bh, tl = rep & bl;
        // 1 in the low bit of every non-zero byte
        const uint32_t nh = ((((th & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | th) & 0x80808080u) >> 7;
        const uint32_t nl = ((((tl & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | tl) & 0x80808080u) >> 7;
        // gather bits 24,16,8,0 into a nibble (bit 24 -> 3 ... bit 0 -> 0): partial products never collide
        const uint32_t byte = ((((nh * 0x01020408u) >> 24) & 0xFu) << 4) | (((nl * 0x01020408u) >> 24) & 0xFu);
        res |= (uint64_t)byte << (56 - 8 * i);
    }
    return res;
}

__device__ __forceinline__ int rank64(uint64_t bmp, int p) { return p == 0 ? 0 : __popcll(bmp >> (64 - p)); }

__global__ void pair_bitmap_test_kernel(const uint64_t* a, const uint64_t* bt, uint64_t* out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = pair_bitmap(a[i], bt[i]);
}

// One 32-byte record (= one DRAM sector) per B block: {bitmap lo, bitmap hi, block column, value offset} + its first eight values.
// A surviving pair of a sparse-block product (uniform random, R-MAT: ~1 value per block) then costs ONE random sector for
// everything it needs from B -- column, bitmap and values -- instead of three (b_bcol, the packed metadata, b_val).
__global__ void pack_meta_kernel(const uint64_t* __restrict__ bmps, const int32_t* __restrict__ bcol, const uint64_t* __restrict__ off,
                                 const __half* __restrict__ val, int64_t nnz, uint4* __restrict__ pm, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t b = bmps[i], o = off[i];
    pm[2 * i] = make_uint4((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)bcol[i], (uint32_t)o);
    unsigned short h[8];
    const int cnt = __popcll(b);
#pragma unroll
    for (int k = 0; k < 8; k++) h[k] = (k < cnt && (int64_t)o + k < nnz) ? __half_as_ushort(val[o + k]) : (unsigned short)0;
    pm[2 * i + 1] = make_uint4(h[0] | ((uint32_t)h[1] << 16), h[2] | ((uint32_t)h[3] << 16), h[4] | ((uint32_t)h[5] << 16), h[6] | ((uint32_t)h[7] << 16));
}

// P0: warp per A block row (grid-stride): candidate pairs, and the span [jmin, jmax] of C block columns.  The statistics are
// reduced per warp and per CTA before they touch global memory: with one global atomic -- or even one volatile load -- per row,
// the 2.1 M rows of P4096 serialise on three L2 addresses (3.7 ms for a kernel that otherwise takes 0.3 ms).
__global__ void __launch_bounds__(256) rowinfo_kernel(const int32_t* __restrict__ a_brp, const int32_t* __restrict__ a_bcol,
                                                      const int32_t* __restrict__ b_brp, const int32_t* __restrict__ b_bcol,
                                                      int row_begin, int row_end, int2* __restrict__ rowinfo,
                                                      unsigned long long* __restrict__ cand, Counters* __restrict__ ctr) {
    __shared__ unsigned long long s_words, s_maxc, s_cand;
    __shared__ int s_maxw;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { s_words = 0; s_maxc = 0; s_maxw = 0; s_cand = 0; }
    __syncthreads();
    unsigned long long w_sum = 0, w_maxc = 0, w_cand = 0;
    int w_maxw = 0;
    for (int row = row_begin + blockIdx.x * 8 + (threadIdx.x >> 5); row < row_end; row += gridDim.x * 8) {
        int jmin = 0x7FFFFFFF, jmax = -1;
        unsigned long long c = 0;
        for (int a = a_brp[row] + lane; a < a_brp[row + 1]; a += 32) {
            const int k = a_bcol[a];
            const int b0 = b_brp[k], b1 = b_brp[k + 1];
            if (b1 > b0) {
                c += (unsigned long long)(b1 - b0);
                jmin = min(jmin, b_bcol[b0]);
                jmax = max(jmax, b_bcol[b1 - 1]);
            }
        }
        c = warp_sum(c); jmin = warp_min(jmin); jmax = warp_max(jmax);
        if (lane == 0) {
            int jbase = 0, words = 0;
            if (jmax >= 0) { jbase = jmin & ~31; words = ((jmax - jbase) >> 5) + 1; }
            rowinfo[row - row_begin] = make_int2(jbase, words);
            cand[row - row_begin] = c;
            w_maxw = max(w_maxw, words); w_sum += (unsigned long long)words; w_maxc = max(w_maxc, c); w_cand += c;
        }
    }
    if (lane == 0) { atomicMax(&s_maxw, w_maxw); atomicAdd(&s_words, w_sum); atomicMax(&s_maxc, w_maxc); atomicAdd(&s_cand, w_cand); }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_maxw) atomicMax(&ctr->max_words, s_maxw);
        if (s_words) atomicAdd(&ctr->sum_words, s_words);
        if (s_maxc) atomicMax(&ctr->max_cand, s_maxc);
        if (s_cand) atomicAdd(&ctr->sum_cand, s_cand);
    }
}

__device__ __forceinline__ uint32_t popc(uint32_t w) { return __popc(w); }
__device__ __forceinline__ uint32_t popc(uint64_t w) { return __popcll(w); }

// CTA-wide exclusive scan of popc(words[i]), i < n: the prefix goes to out[i] (out may be null: the total only); returns the total
// to every thread.  Ranks the bit set's words (32-bit) and scans the C blocks' value counts (64-bit bitmaps).
template <typename W, typename O>
__device__ __forceinline__ uint32_t scan_popc(const W* words, O* out, int n, uint32_t* s_tmp) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int per = (n + T - 1) / T;
    const int w0 = min(tid * per, n), w1 = min(w0 + per, n);
    uint32_t s = 0;
    for (int w = w0; w < w1; w++) s += popc(words[w]);
    uint32_t inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_tmp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t v = lane < (T >> 5) ? s_tmp[lane] : 0, vi = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, vi, o);
            if (lane >= o) vi += t;
        }
        s_tmp[lane] = vi - v;
        if (lane == 31) s_tmp[32] = vi;
    }
    __syncthreads();
    uint32_t run = s_tmp[wid] + inc - s;
    if (out) for (int w = w0; w < w1; w++) { out[w] = run; run += popc(words[w]); }
    const uint32_t total = s_tmp[32];
    __syncthreads();
    return total;
}

// Per-row state shared by the enumeration modes.
struct RowCtx {
    int row, nr;         // first block row of the work item and the number of rows in it
    int a0, a1, jbase, c0;
    const int* abr;      // [nr+1] a_brp of the rows                        (shared)
    const int* jb;       // [nr]   first C block column of each row's bit set
    const int* wo;       // [nr+1] word offset of each row's bit set inside the work item's
    uint32_t* rsurv;     // [nr]   COUNT: surviving pairs per row
    uint32_t* bitset; uint32_t* wrank;
    uint64_t* cbmp;      // FILL: staging (shared or global C.bmps+c0); NUMERIC: shared copy or null
    uint32_t* coff;      // NUMERIC: value offsets relative to the row, or null (global mode)
    float* acc;          // NUMERIC: shared accumulators or null (global atomics)
    float* dense;        // NUMERIC_MMA: [ccount][64] fp32, two slots per lane (cell (r,c) at (c*4 + r/2) + 32*(r&1))
};

// index of the row of a work item that owns v, given the rows' ascending start offsets (A blocks, bit-set words or C blocks)
// (nr <= 32.  Five fixed halving steps: the linear scan this replaces was 15 % of the NUMERIC pass's instructions on P4096 -- every
// lane of every surviving pair walks the 16 rows of its group, and the lanes of a warp stop at different rows.)
__device__ __forceinline__ int local_row(const int* bounds, int nr, int v) {
    int rl = 0;
    if (nr > 1) {
#pragma unroll
        for (int s = 16; s; s >>= 1) {
            const int t = rl + s;
            if (t < nr && v >= bounds[t]) rl = t;
        }
    }
    return rl;
}

// the global loads a surviving pair starts with, kept apart from the work on them so that the scalar NUMERIC pass can have two
// pairs' loads in flight per thread before it touches the first result (A/B on one box: U1M numeric 10.65 -> 9.55 ms, R-MAT-18
// 146 -> 109 ms; the same batching in FILL and in the 8-lanes-per-pair walk cost more in registers than it hid in latency)
struct PairIn { uint4 pm; uint4 bv8; uint64_t abmp; uint32_t aoff; };
template <int PASS>
__device__ __forceinline__ PairIn load_pair(const GemmArgs& g, int a, int b) {
    PairIn in;
    in.pm = __ldg(g.b_pm + 2 * (int64_t)b);
    in.bv8 = PASS == PASS_FILL ? make_uint4(0, 0, 0, 0) : __ldg(g.b_pm + 2 * (int64_t)b + 1);     // same sector
    in.abmp = g.a_bmps[a];
    in.aoff = PASS == PASS_FILL ? 0u : (uint32_t)g.a_off[a];
    return in;
}
// value k (< 8) of a B block out of its record's inline copy
__device__ __forceinline__ float inline_val(const uint4& v, int k) {
    const uint32_t w = (k & 4) ? ((k & 2) ? v.w : v.z) : ((k & 2) ? v.y : v.x);
    return __half2float(__ushort_as_half((unsigned short)((k & 1) ? (w >> 16) : (w & 0xFFFFu))));
}

template <int PASS>
__device__ __forceinline__ void apply_pair(const GemmArgs& g, const RowCtx& r, int a, const PairIn& in, int arow = -1) {
    const uint4 pm = in.pm;
    const uint64_t abmp = in.abmp, bbmp = ((uint64_t)pm.y << 32) | pm.x;
    const int rl = local_row(r.abr, r.nr, a);
    const int j = (int)pm.z - r.jb[rl];
    const int wi = r.wo[rl] + (j >> 5);
    const uint32_t word = r.bitset[wi];
    const int c = (int)r.wrank[wi] + __popc(word & ((1u << (j & 31)) - 1u));
    if (PASS == PASS_FILL) {
        const uint64_t pb = pair_bitmap(abmp, bbmp);
        unsigned int* w = reinterpret_cast<unsigned int*>(&r.cbmp[c]);      // native 32-bit ATOMS.OR, not a 64-bit CAS loop
        if ((uint32_t)pb) atomicOr(w, (unsigned int)pb);
        if ((uint32_t)(pb >> 32)) atomicOr(w + 1, (unsigned int)(pb >> 32));
    } else {
        const __half* av = g.a_val + in.aoff;
        const __half* bv = g.b_val + pm.w;
        const bool b_inline = __popcll(bbmp) <= 8;               // the record carries the block's values
        uint64_t cb; float* dst;
        if (r.acc) { cb = r.cbmp[c]; dst = r.acc + r.coff[c]; }
        else { cb = g.c_bmps[r.c0 + c]; dst = g.c_val + g.c_off[r.c0 + c]; }
        uint64_t rem = abmp;
        int ka = 0;
        if (arow >= 0) {                                    // this lane's row of the A block only
            rem = abmp & (0xFF00000000000000ull >> (8 * arow));
            ka = arow ? __popcll(abmp >> (64 - 8 * arow)) : 0;
            if (!rem) return;
        }
        while (rem) {
            const int p = __clzll((long long)rem);
            rem &= ~(0x8000000000000000ull >> p);
            const int rr = p >> 3, k = p & 7;
            const float aval = __half2float(av[ka++]);
            uint64_t hits = bbmp & (0x8080808080808080ull >> k);    // B(k, c) for c = 0..7 (Bt cell = c*8+k)
            while (hits) {
                const int q = __clzll((long long)hits);
                hits &= ~(0x8000000000000000ull >> q);
                const int kb = rank64(bbmp, q);
                const float bval = b_inline ? inline_val(in.bv8, kb) : __half2float(bv[kb]);
                atomicAdd(dst + rank64(cb, rr * 8 + (q >> 3)), aval * bval);
            }
        }
    }
}

// ---- pair classes (scalar NUMERIC pass with several lanes per pair) ---------------------------------------------------------------
// The lanes of a warp walk their pairs in lockstep, so a warp takes as long as its slowest lane: on a stencil product the four pairs
// of a warp mix tridiagonal x tridiagonal blocks (9 products per lane) with diagonal x diagonal ones (1) and single-value A blocks
// (7 of 8 lanes idle) -- ncu showed ~4 active threads per instruction in the product loops.  FILL, which touches every pair's two
// bitmaps anyway, therefore leaves a work item's segment of the pair list sorted by class: classes 0..8 = A blocks with more than two
// values, ordered by (values per row of A) x (values per row of B) descending; classes 9..11 = A blocks with one or two values (top bit
// of the entry's A index set): NUMERIC gives those ONE lane per pair instead of eight.
constexpr int PAIR_CLASSES = 12, PAIR_LIGHT = 9, SORT_K = 4;
constexpr uint32_t PAIR_LIGHT_FLAG = 0x80000000u;
__device__ __forceinline__ int pair_class(uint64_t abmp, uint64_t bbmp) {
    const int pa = __popcll(abmp), pb = __popcll(bbmp);
    const int cb = min(3, (pb + 7) >> 3);                       // 1..3
    if (pa <= 2) return PAIR_LIGHT + (3 - cb);
    const int ca = min(3, (pa + 7) >> 3);
    return 8 - ((ca - 1) * 3 + (cb - 1));
}

// ---- tensor-core path (dense blocks) -----------------------------------------------------------------
// Two halves of an 8x8 fp16 operand row for mma.m16n8k8: the cells p0 = g*8 + 2t and p0+1 of a block, packed
// as .f16x2 (absent cells are 0).  Works for the A block (cell = row*8 + k) and for the transposed-operand B
// block (cell = col*8 + k) alike -- which is exactly why the reference stores B transposed (SPGEMM.cu:309-312).
__device__ __forceinline__ uint32_t frag_pair(uint64_t bmp, const __half* __restrict__ vals, int p0) {
    const uint32_t two = (uint32_t)(bmp >> (62 - p0)) & 3u;        // bit1 = cell p0, bit0 = cell p0+1
    if (!two) return 0u;
    const int r = rank64(bmp, p0);
    const unsigned short lo = (two & 2u) ? __half_as_ushort(vals[r]) : (unsigned short)0;
    const unsigned short hi = (two & 1u) ? __half_as_ushort(vals[r + (int)(two >> 1)]) : (unsigned short)0;
    return (uint32_t)lo | ((uint32_t)hi << 16);
}

// Drain n (<= 32) queued (A block, B block) pairs with the whole warp.  Stage 1: lane l fetches the metadata of
// pair l (bitmaps, value offsets, dense C slot) -- one round of global latency for the whole batch -- into a per-warp
// shared staging area.  Stage 2: walk the batch; consecutive pairs that share the A block are multiplied two at a
// time by one mma.sync.m16n8k8 (A-operand = the two B^t blocks stacked, B-operand = the A block, D = the two 8x8
// fp32 products transposed); the fragments of the next step are loaded before the current MMA is issued.  Each
// lane owns two fixed slots of every dense C block, so the accumulation needs no warp syncs.
struct PairMeta { uint64_t abmp, bbmp; uint32_t aoff, boff; int32_t cidx; uint32_t a; };   // 32 bytes

__device__ __forceinline__ void drain_mma(const GemmArgs& g, const RowCtx& r, const uint2* q, int n, PairMeta* sm) {
    const int lane = threadIdx.x & 31;
    const int p0 = (lane >> 2) * 8 + (lane & 3) * 2;
    if (lane < n) {
        const uint2 e = q[lane];
        PairMeta m;
        m.a = e.x;
        m.abmp = g.a_bmps[e.x]; m.aoff = (uint32_t)g.a_off[e.x];
        m.bbmp = g.b_bmps[e.y]; m.boff = (uint32_t)g.b_off[e.y];
        const int j = g.b_bcol[e.y] - r.jbase;
        m.cidx = (int)r.wrank[j >> 5] + __popc(r.bitset[j >> 5] & ((1u << (j & 31)) - 1u));
        sm[lane] = m;
    }
    __syncwarp();
    uint32_t fb = 0, fa0 = 0, fa1 = 0, cur_a = 0xFFFFFFFFu;
    int c0 = 0, c1 = 0;
    bool two = false;
    auto load = [&](int i, uint32_t& fb_, uint32_t& fa0_, uint32_t& fa1_, int& c0_, int& c1_, bool& two_, uint32_t& a_) {
        const PairMeta m0 = sm[i];
        two_ = (i + 1 < n) && (sm[i + 1].a == m0.a);
        if (m0.a != a_) { fb_ = frag_pair(m0.abmp, g.a_val + m0.aoff, p0); a_ = m0.a; }
        fa0_ = frag_pair(m0.bbmp, g.b_val + m0.boff, p0);
        c0_ = m0.cidx;
        if (two_) { const PairMeta m1 = sm[i + 1]; fa1_ = frag_pair(m1.bbmp, g.b_val + m1.boff, p0); c1_ = m1.cidx; }
        else fa1_ = 0u;
    };
    int i = 0;
    if (n > 0) load(0, fb, fa0, fa1, c0, c1, two, cur_a);
    while (i < n) {
        const int nxt = i + (two ? 2 : 1);
        uint32_t nfb = fb, nfa0 = 0, nfa1 = 0, na = cur_a; int nc0 = 0, nc1 = 0; bool ntwo = false;
        if (nxt < n) load(nxt, nfb, nfa0, nfa1, nc0, nc1, ntwo, na);
        float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                     : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3) : "r"(fa0), "r"(fa1), "r"(fb));
        // several warps of the CTA work on different A blocks of the row and may meet in a C block: shared-memory float atomics
        // (one instruction each)
        float* a0 = r.dense + c0 * 64 + lane;
        atomicAdd(a0, d0); atomicAdd(a0 + 32, d1);
        if (two) { float* a1 = r.dense + c1 * 64 + lane; atomicAdd(a1, d2); atomicAdd(a1 + 32, d3); }
        i = nxt; fb = nfb; fa0 = nfa0; fa1 = nfa1; c0 = nc0; c1 = nc1; two = ntwo; cur_a = na;
    }
    __syncwarp();
}

template <int PASS>
__device__ __forceinline__ void drain(const GemmArgs& g, const RowCtx& r, const uint2* q, int n) {
    if constexpr (PASS == PASS_NUMERIC_MMA) {
        drain_mma(g, r, q, n, reinterpret_cast<PairMeta*>(const_cast<uint2*>(q) + 64));
    } else {
        const int lane = threadIdx.x & 31;
        if (lane < n) { const uint2 e = q[lane]; apply_pair<PASS>(g, r, (int)e.x, load_pair<PASS>(g, (int)e.x, (int)e.y)); }
    }
}

// Candidate walk, four B blocks per lane and step: `slots` A blocks at a time, G lanes per A block, each lane
// tests one aligned 32-bit word of B's inner-dimension masks (kmask) against the replicated mask of its A block.
// COUNT (!LIST): survivors set their C block column in the row's bit set and are counted per row.  FILL (LIST): they
// are appended to the row's segment of the global pair list (one shared cursor bump per warp and step).
template <bool LIST>
__device__ __forceinline__ void enumerate_vec(const GemmArgs& g, const RowCtx& r, uint2* list, uint32_t* s_cursor, uint32_t& n_surv) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    const int Gs = g.G, slots = T / Gs, slot = tid / Gs, gl = tid % Gs;
    const int niter = (r.a1 - r.a0 + slots - 1) / slots;
    for (int itA = 0; itA < niter; itA++) {
        const int a = r.a0 + itA * slots + slot;
        int b0 = 0, b1 = 0, rl = 0, jb = 0, wb = 0; uint32_t am4 = 0;
        if (a < r.a1) {
            const int k = g.a_bcol[a];
            b0 = g.b_brp[k]; b1 = g.b_brp[k + 1];
            am4 = (uint32_t)g.a_kmask[a] * 0x01010101u;
            rl = local_row(r.abr, r.nr, a); jb = r.jb[rl]; wb = r.wo[rl];
        }
        const int bs = b0 & ~3;
        int ngrp = (b1 - bs + 3) >> 2;           // 4-block groups of this lane's B row (0 when the row is empty)
        if (b1 <= b0) ngrp = 0;
        int maxgrp = ngrp;
#pragma unroll
        for (int o = 16; o; o >>= 1) maxgrp = max(maxgrp, __shfl_xor_sync(0xffffffffu, maxgrp, o));
        for (int grp0 = 0; grp0 < maxgrp; grp0 += Gs) {
            const int grp = grp0 + gl;
            const int bb = bs + 4 * grp;
            uint32_t nz = 0;
            if (grp < ngrp) {
                const uint32_t km4 = *reinterpret_cast<const uint32_t*>(g.b_kmask + bb);
                const int lo = max(b0 - bb, 0), hi = min(b1 - bb, 4);          // valid bytes [lo, hi)
                const uint32_t vm = (0xFFFFFFFFu << (8 * lo)) & (hi >= 4 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu << (8 * hi)));
                nz = __vcmpne4(km4 & am4, 0u) & vm;                              // 0xFF in every surviving byte
            }
            if (LIST) {
                // recompute per-byte positions without packing tricks (at most 4 survivors per lane)
                uint32_t total = 0, base = 0;
                uint32_t p4[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const bool s = (nz >> (8 * i)) & 1u;
                    const uint32_t m = __ballot_sync(0xffffffffu, s);
                    p4[i] = total + __popc(m & ((1u << lane) - 1u));
                    total += __popc(m);
                }
                if (total) {
                    if (lane == 0) base = atomicAdd(s_cursor, total);
                    base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if ((nz >> (8 * i)) & 1u) list[base + p4[i]] = make_uint2((uint32_t)a, (uint32_t)(bb + i));
                }
            } else {
                const int cnt = __popc(nz) >> 3;
                n_surv += cnt;
                if (r.nr > 1 && cnt) atomicAdd(&r.rsurv[rl], (uint32_t)cnt);      // single row: reduced by the caller
                for (uint32_t rem = nz; rem;) {
                    const int i = (__ffs(rem) - 1) >> 3;
                    rem &= ~(0xFFu << (8 * i));
                    const int j = g.b_bcol[bb + i] - jb;
                    atomicOr(&r.bitset[wb + (j >> 5)], 1u << (j & 31));
                }
            }
        }
    }
}

// ---- fine index of B ---------------------------------------------------------------------------------------------
// Uniform-random and R-MAT operands have about one value per 8x8 block.  The candidate scan then tests every block of B's block
// row bcol(a) against the A block (U1M: 128 tests for 16 survivors) and fetches each survivor's record with a random access: one
// 64-byte DRAM burst per pair and pass (ncu, U1M: 31 GB read by FILL, 31 GB by NUMERIC, for 12 GB of algorithmic bytes).  With
// B's blocks bucketed by inner index the survivors of an A block are the contiguous bucket(s) of its own inner index(es).
__global__ void fine_max_kernel(const uint32_t* __restrict__ cnt, int64_t n, uint32_t* __restrict__ mx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t v = warp_max(i < n ? cnt[i] : 0u);
    if ((threadIdx.x & 31) == 0 && v) atomicMax(mx, v);
}
__global__ void fine_count_kernel(const uint64_t* __restrict__ keys, const uint8_t* __restrict__ kmask, int64_t nblk, uint32_t* __restrict__ cnt) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint32_t br = (uint32_t)(keys[b] >> 32);
    uint32_t m = kmask[b];
    while (m) { const int t = __ffs(m) - 1; m &= m - 1; atomicAdd(cnt + (size_t)br * 8 + t, 1u); }
}
// one thread per bucket walks its block row in order: entries of a bucket keep the block order (deterministic)
__global__ void fine_fill_kernel(const int32_t* __restrict__ brp, const uint8_t* __restrict__ kmask, const uint4* __restrict__ pm, int32_t nbr,
                                 const uint32_t* __restrict__ fptr, uint32_t* __restrict__ f_bcol, uint8_t* __restrict__ f_kmask, uint4* __restrict__ f_rec) {
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= (int64_t)nbr * 8) return;
    const int br = (int)(u >> 3), t = (int)(u & 7);
    uint32_t w = fptr[u];
    for (int b = brp[br]; b < brp[br + 1]; b++) {
        const uint32_t km = kmask[b];
        if (!((km >> t) & 1u)) continue;
        const uint4 r0 = pm[2 * (int64_t)b], r1 = pm[2 * (int64_t)b + 1];
        f_bcol[w] = r0.z; f_kmask[w] = (uint8_t)km; f_rec[2 * (int64_t)w] = r0; f_rec[2 * (int64_t)w + 1] = r1;
        w++;
    }
}

// Walk the row's candidate pairs (MMA pass, one block row per work item): `slots` A blocks at a time, G lanes per A block striding
// over the B block row; survivors are compacted through a per-warp queue so that all 32 lanes work on surviving pairs.
template <int PASS>
__device__ __forceinline__ void enumerate_row(const GemmArgs& g, const RowCtx& r, uint2* q) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    const int Gs = g.G, slots = T / Gs, slot = tid / Gs, gl = tid % Gs;
    int qn = 0;
    const int niter = (r.a1 - r.a0 + slots - 1) / slots;
    for (int itA = 0; itA < niter; itA++) {
        const int a = r.a0 + itA * slots + slot;
        int b0 = 0, b1 = 0; uint32_t am = 0;
        if (a < r.a1) {
            const int k = g.a_bcol[a];
            b0 = g.b_brp[k]; b1 = g.b_brp[k + 1];
            am = g.a_kmask[a];
        }
        int maxlen = b1 - b0;    // warp-uniform trip count (ballot below)
#pragma unroll
        for (int o = 16; o; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
        for (int off = 0; off < maxlen; off += Gs) {
            const int b = b0 + off + gl;
            const bool valid = b < b1;
            const bool surv = valid && (am & g.b_kmask[b]) != 0;
            const uint32_t m = __ballot_sync(0xffffffffu, surv);
            if (surv) q[qn + __popc(m & ((1u << lane) - 1u))] = make_uint2((uint32_t)a, (uint32_t)b);
            qn += __popc(m);
            __syncwarp();
            if (qn >= 32) {
                drain<PASS>(g, r, q, 32);
                __syncwarp();
                uint2 t = make_uint2(0, 0);
                const bool mv = lane + 32 < qn;
                if (mv) t = q[32 + lane];
                __syncwarp();
                if (mv) q[lane] = t;
                qn -= 32;
                __syncwarp();
            }
        }
    }
    drain<PASS>(g, r, q, qn);
    __syncwarp();
}

// Walk the surviving pairs of a work item through B's fine index: 8 lanes per A block, one bucket per bit of its kmask, the
// lanes striding over the bucket, two entries in flight per lane.  A B block that shares several inner indices with the A block
// sits in several of those buckets; it is taken from the lowest one.  Buckets longer than FINE_LONG entries (the hub rows of a
// power-law B) are left to a second walk with a whole warp per bucket -- eight lanes on a 10^4-entry bucket would be the tail of
// the row.
//   FMODE 0: set the C block column's bit (f_bcol / f_kmask only: 5 bytes per pair), count survivors when STATS
//   FMODE 1: OR the pair's boolean block product into the C block's bitmap          (32-byte record)
//   FMODE 2: multiply                                                                 (32-byte record, values inline)
// CTA-wide: every thread of the CTA must call it (it synchronises).
constexpr int FINE_LONG = 256;
template <int FMODE, bool STATS>
__device__ __forceinline__ void fine_entry(const GemmArgs& g, const RowCtx& r, int a, int rl, int jb, int wb, uint64_t abmp, uint32_t aoff, uint32_t f,
                                           uint32_t& cnt) {
    if (FMODE == 0) {
        const int j = (int)g.f_bcol[f] - jb;
        atomicOr(&r.bitset[wb + (j >> 5)], 1u << (j & 31));
        cnt++;
    } else {
        PairIn in;
        in.pm = __ldg(g.f_rec + 2 * (int64_t)f);
        in.bv8 = FMODE == 2 ? __ldg(g.f_rec + 2 * (int64_t)f + 1) : make_uint4(0, 0, 0, 0);
        in.abmp = abmp; in.aoff = aoff;
        apply_pair<FMODE == 1 ? PASS_FILL : PASS_NUMERIC>(g, r, a, in);
    }
}
template <int FMODE, bool STATS>
__device__ __forceinline__ void fine_bucket(const GemmArgs& g, const RowCtx& r, int a, int rl, uint32_t am, uint32_t below, uint64_t abmp, uint32_t aoff,
                                            uint32_t f0, uint32_t f1, uint32_t first, uint32_t step, uint32_t& cnt) {
    const int jb = r.jb[rl], wb = r.wo[rl];
    uint32_t f = f0 + first;
    if constexpr (FMODE == 0) {
        for (; f < f1; f += step) {
            if (below && (g.f_kmask[f] & below)) continue;                 // already met in a lower bucket
            fine_entry<FMODE, STATS>(g, r, a, rl, jb, wb, abmp, aoff, f, cnt);
        }
    } else {
    // two records in flight per lane: the loads of entries f and f + step are issued before either is used
    for (; f + step < f1; f += 2 * step) {
        const bool s0 = !(below && (g.f_kmask[f] & below)), s1 = !(below && (g.f_kmask[f + step] & below));
        PairIn i0, i1;
        i0.abmp = i1.abmp = abmp; i0.aoff = i1.aoff = aoff;
        i0.pm = i1.pm = make_uint4(0, 0, 0, 0); i0.bv8 = i1.bv8 = make_uint4(0, 0, 0, 0);
        if (s0) { i0.pm = __ldg(g.f_rec + 2 * (int64_t)f); if (FMODE == 2) i0.bv8 = __ldg(g.f_rec + 2 * (int64_t)f + 1); }
        if (s1) { i1.pm = __ldg(g.f_rec + 2 * (int64_t)(f + step)); if (FMODE == 2) i1.bv8 = __ldg(g.f_rec + 2 * (int64_t)(f + step) + 1); }
        if (s0) apply_pair<FMODE == 1 ? PASS_FILL : PASS_NUMERIC>(g, r, a, i0);
        if (s1) apply_pair<FMODE == 1 ? PASS_FILL : PASS_NUMERIC>(g, r, a, i1);
    }
    if (f < f1 && !(below && (g.f_kmask[f] & below))) fine_entry<FMODE, STATS>(g, r, a, rl, jb, wb, abmp, aoff, f, cnt);
    }
}
template <int FMODE, bool STATS>
__device__ __forceinline__ void enumerate_fine(const GemmArgs& g, const RowCtx& r, uint32_t& n_surv) {
    constexpr int GL = 8;
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarps = T >> 5;
    const int slots = T / GL, slot = tid / GL, gl = tid % GL;
    bool any_long = false;
    for (int a = r.a0 + slot; a < r.a1; a += slots) {
        const int k = g.a_bcol[a];
        const uint32_t am = g.a_kmask[a];
        const int rl = local_row(r.abr, r.nr, a);
        uint64_t abmp = 0; uint32_t aoff = 0;
        if (FMODE >= 1) abmp = g.a_bmps[a];
        if (FMODE == 2) aoff = (uint32_t)g.a_off[a];
        uint32_t m = am, cnt = 0;
        while (m) {
            const int t = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t f0 = g.f_ptr[(size_t)k * 8 + t], f1 = g.f_ptr[(size_t)k * 8 + t + 1];
            if (f1 - f0 > FINE_LONG) { any_long = true; continue; }       // second walk below
            fine_bucket<FMODE, STATS>(g, r, a, rl, am, am & ((1u << t) - 1u), abmp, aoff, f0, f1, gl, GL, cnt);
        }
        if (STATS && cnt) { n_surv += cnt; if (r.nr > 1) atomicAdd(&r.rsurv[rl], cnt); }
    }
    // long buckets: warp w takes the A blocks a0 + w, a0 + w + nwarps, ...; its 32 lanes stride over the bucket.  The walk is
    // warp-uniform (every lane sees the same A block and bit), so nothing has to be handed over between lanes.
    if (!__syncthreads_or(any_long)) return;
    for (int a = r.a0 + wid; a < r.a1; a += nwarps) {
        const int k = g.a_bcol[a];
        const uint32_t am = g.a_kmask[a];
        uint32_t m = am, cnt = 0;
        int rl = -1; uint64_t abmp = 0; uint32_t aoff = 0;
        while (m) {
            const int t = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t f0 = g.f_ptr[(size_t)k * 8 + t], f1 = g.f_ptr[(size_t)k * 8 + t + 1];
            if (f1 - f0 <= FINE_LONG) continue;
            if (rl < 0) {
                rl = local_row(r.abr, r.nr, a);
                if (FMODE >= 1) abmp = g.a_bmps[a];
                if (FMODE == 2) aoff = (uint32_t)g.a_off[a];
            }
            fine_bucket<FMODE, STATS>(g, r, a, rl, am, am & ((1u << t) - 1u), abmp, aoff, f0, f1, (uint32_t)lane, 32u, cnt);
        }
        if (STATS && cnt) { n_surv += cnt; if (r.nr > 1) atomicAdd(&r.rsurv[rl], cnt); }
    }
}

// REUSE (NUMERIC passes of a kept plan, bmsp_spgemm_numeric): C's value offsets are absolute already -- the first NUMERIC pass made
// them so in place -- and are read, never written.
template <int PASS, int MAXT, bool REUSE = false>
__global__ void __launch_bounds__(MAXT) spgemm_pass_kernel(GemmArgs g) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarps = T >> 5;
    // shared-memory carve-up (sizes mirrored by pass_smem_bytes on the host)
    constexpr bool HAS_CBMP = PASS == PASS_FILL || PASS == PASS_NUMERIC;
    constexpr bool HAS_QUEUE = PASS == PASS_NUMERIC_MMA;
    uint64_t* s_cbmp = reinterpret_cast<uint64_t*>(smem);                                        // [cap_c]     FILL, NUMERIC
    uint2* s_queue = reinterpret_cast<uint2*>(s_cbmp + (HAS_CBMP ? g.cap_c : 0));                 // [nwarps*QSLOTS] NUMERIC_MMA
    uint32_t* s_bitset = reinterpret_cast<uint32_t*>(s_queue + (HAS_QUEUE ? nwarps * QSLOTS : 0)); // [cap_words]
    uint32_t* s_wrank = s_bitset + g.cap_words;                                                   // [cap_words] (COUNT: only for row groups)
    uint32_t* s_coff = s_wrank + ((PASS == PASS_COUNT && g.group == 1) ? 0 : g.cap_words);        // [cap_c]     NUMERIC
    float* s_acc = reinterpret_cast<float*>(s_coff + (PASS == PASS_NUMERIC ? g.cap_c : 0));       // [cap_nnz]   NUMERIC
    float* s_dense = s_acc + (PASS == PASS_NUMERIC ? g.cap_nnz : 0);                              // [cap_c*64]  NUMERIC_MMA
    uint32_t* s_tmp = reinterpret_cast<uint32_t*>(s_dense + (PASS == PASS_NUMERIC_MMA ? g.cap_c * 64 : 0)); // [34]
    int* s_row = reinterpret_cast<int*>(s_tmp + 34);
    uint32_t* s_cursor = reinterpret_cast<uint32_t*>(s_row + 1);
    int* s_batch = s_row + 2;                          // [0] next queue index of this CTA's batch, [1] its end
    // per-row tables of the work item (<= 32 rows): A block offsets, bit-set origin and word offsets, C block offsets, surviving
    // pairs, value offsets
    int* s_abr = s_row + 4;                            // [33]
    int* s_jb = s_abr + 33;                            // [32]
    int* s_wo = s_jb + 32;                             // [33]
    int* s_cbr = s_wo + 33;                            // [33]
    uint32_t* s_rsurv = reinterpret_cast<uint32_t*>(s_cbr + 33);   // [32]
    uint32_t* s_rowoff = s_rsurv + 32;                 // [33]
    if (tid == 0) { s_batch[0] = 0; s_batch[1] = 0; }
    __shared__ uint32_t s_cls[PAIR_CLASSES];           // FILL: pairs per class of the work item (zero between work items)
    if (tid < PAIR_CLASSES) s_cls[tid] = 0;

    unsigned long long n_surv_total = 0;
    int my_max1 = 0, my_max2 = 0, my_max3 = 0;         // per-thread maxima, published once when the CTA retires
    uint2* q = s_queue + wid * QSLOTS;
    const int R = g.row_list ? 1 : g.group;
    const int n_items = g.row_list ? g.n_list : (g.row_end - g.row_begin + R - 1) / R;

    while (true) {
        if (tid == 0) {
            if (s_batch[0] == s_batch[1]) { s_batch[0] = atomicAdd(g.work_counter, g.batch); s_batch[1] = s_batch[0] + g.batch; }
            const int i = s_batch[0]++;
            *s_row = i < n_items ? (g.row_list ? g.row_list[i] : g.row_begin + i * R) : g.row_end;
            *s_cursor = 0;
        }
        __syncthreads();
        RowCtx r;
        r.row = *s_row;
        __syncthreads();
        if (r.row >= g.row_end) break;
        r.nr = min(R, g.row_end - r.row);
        const int nr = r.nr;
        const int lrow = r.row - g.row_begin;
        // ---- the rows of this work item
        if (tid < 32) {
            int nw = 0;
            if (tid < nr) { const int2 ri = g.rowinfo[lrow + tid]; s_jb[tid] = ri.x; nw = ri.y; s_rsurv[tid] = 0; }
            int inc = nw;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            if (tid < nr) s_wo[tid + 1] = inc;
            if (tid == 0) s_wo[0] = 0;
            if (tid <= nr) {
                s_abr[tid] = g.a_brp[r.row + tid];
                if (PASS != PASS_COUNT) s_cbr[tid] = g.c_brp[lrow + tid];
                if (PASS == PASS_NUMERIC || PASS == PASS_NUMERIC_MMA) s_rowoff[tid] = (uint32_t)(g.row_nnz[lrow + tid] - g.row_nnz[lrow]);
            }
        }
        __syncthreads();
        const int nwords = s_wo[nr];
        r.a0 = s_abr[0]; r.a1 = s_abr[nr]; r.jbase = s_jb[0];
        r.abr = s_abr; r.jb = s_jb; r.wo = s_wo; r.rsurv = s_rsurv;
        if (nwords == 0) {
            if (PASS == PASS_COUNT && tid < nr) { g.row_count[lrow + tid] = 0; g.row_surv[lrow + tid] = 0; }
            if (PASS == PASS_FILL && tid < nr) g.row_nnz[lrow + tid] = 0;
            continue;
        }
        const bool wfit = nwords <= g.cap_words;
        r.bitset = wfit ? s_bitset : g.g_bitset + (size_t)blockIdx.x * g.max_words;
        r.wrank = wfit ? s_wrank : g.g_wrank + (size_t)blockIdx.x * g.max_words;
        r.cbmp = nullptr; r.coff = nullptr; r.acc = nullptr; r.dense = nullptr; r.c0 = 0;
        for (int w = tid; w < nwords; w += T) r.bitset[w] = 0;
        int ccount = 0;
        uint32_t s0 = 0, nsurv = 0;
        if (PASS != PASS_COUNT) {
            r.c0 = s_cbr[0]; ccount = s_cbr[nr] - r.c0;
            s0 = g.row_surv[lrow]; nsurv = g.row_surv[lrow + nr] - s0;
        }
        if (PASS != PASS_COUNT && ccount == 0) {
            if (PASS == PASS_FILL && tid < nr) g.row_nnz[lrow + tid] = 0;
            __syncthreads();
            continue;
        }
        uint2* list = g.surv_list + s0;
        const int c0 = r.c0;                           // s_cbr holds absolute C block offsets; c - c0 is the index inside the work item

        if (PASS == PASS_COUNT) {
            __syncthreads();
            uint32_t ns = 0;
            if (g.f_ptr) enumerate_fine<0, true>(g, r, ns);
            else enumerate_vec<false>(g, r, nullptr, nullptr, ns);      // bits; survivors per row into s_rsurv
            if (nr == 1) {
#pragma unroll
                for (int o = 16; o; o >>= 1) ns += __shfl_xor_sync(0xffffffffu, ns, o);
                if (lane == 0 && ns) atomicAdd(&s_rsurv[0], ns);
            }
            __syncthreads();
            const uint32_t total = scan_popc(r.bitset, nr > 1 ? r.wrank : nullptr, nwords, s_tmp);
            if (tid < nr) {
                uint32_t cnt = total;
                if (nr > 1) {
                    const int w0 = s_wo[tid], w1 = s_wo[tid + 1];
                    cnt = (w1 < nwords ? r.wrank[w1] : total) - (w0 < nwords ? r.wrank[w0] : total);
                }
                g.row_count[lrow + tid] = cnt; g.row_surv[lrow + tid] = s_rsurv[tid]; n_surv_total += s_rsurv[tid];
                my_max3 = max(my_max3, (int)cnt);                                // largest single row (dense-block NUMERIC runs row by row)
            }
            if (tid == 0) my_max1 = max(my_max1, (int)total);
        }
        if (PASS == PASS_FILL) {
            const bool cfit = ccount <= g.cap_c;
            r.cbmp = cfit ? s_cbmp : g.c_bmps + c0;            // global C.bmps is pre-zeroed
            if (cfit) for (int c = tid; c < ccount; c += T) r.cbmp[c] = 0;
            __syncthreads();
            uint32_t ns = 0;
            if (g.f_ptr) {
                // fine index: no pair list at all -- bits from the 5-byte bucket entries, then the records once
                enumerate_fine<0, false>(g, r, ns);
                __syncthreads();
                scan_popc(r.bitset, r.wrank, nwords, s_tmp);
                enumerate_fine<1, false>(g, r, ns);
            } else {
            // pair list only: a survivor's C block column comes with its packed B record (one sector, fetched here for the first time
            // and again -- from L2 -- by the pair pass below) instead of a separate random read of b_bcol per survivor
            enumerate_vec<true>(g, r, list, s_cursor, ns);
            __syncthreads();
            for (uint32_t e = tid; e < nsurv; e += T) {
                const uint2 pr = list[e];
                const int rl = local_row(r.abr, r.nr, (int)pr.x);
                const int j = (int)__ldg(&g.b_pm[2 * (int64_t)pr.y].z) - r.jb[rl];
                atomicOr(&r.bitset[r.wo[rl] + (j >> 5)], 1u << (j & 31));
            }
            __syncthreads();
            scan_popc(r.bitset, r.wrank, nwords, s_tmp);
            if (nsurv <= (uint32_t)g.sort_max) {
                // apply the pairs and leave the segment sorted by class for NUMERIC (counting sort through shared counters; a thread
                // keeps its <= SORT_K pairs in registers between reading and rewriting the segment)
                uint2 mine[SORT_K]; uint32_t slot[SORT_K];
#pragma unroll
                for (int k = 0; k < SORT_K; k++) {
                    const uint32_t e = tid + (uint32_t)k * T;
                    slot[k] = 0xFFFFFFFFu;
                    if (e < nsurv) {
                        const uint2 pr = list[e];
                        const PairIn in = load_pair<PASS_FILL>(g, (int)pr.x, (int)pr.y);
                        apply_pair<PASS_FILL>(g, r, (int)pr.x, in);
                        const int cls = pair_class(in.abmp, ((uint64_t)in.pm.y << 32) | in.pm.x);
                        mine[k] = pr;
                        slot[k] = ((uint32_t)cls << 24) | atomicAdd(&s_cls[cls], 1u);
                    }
                }
                __syncthreads();
                if (tid == 0) {
                    uint32_t run = 0;
                    for (int c = 0; c < PAIR_CLASSES; c++) { const uint32_t t = s_cls[c]; s_cls[c] = run; run += t; }
                }
                __syncthreads();
#pragma unroll
                for (int k = 0; k < SORT_K; k++) {
                    if (slot[k] != 0xFFFFFFFFu) {
                        const uint32_t cls = slot[k] >> 24;
                        uint2 pr = mine[k];
                        if (cls >= (uint32_t)PAIR_LIGHT) pr.x |= PAIR_LIGHT_FLAG;
                        list[s_cls[cls] + (slot[k] & 0xFFFFFFu)] = pr;
                    }
                }
                __syncthreads();
                if (tid < PAIR_CLASSES) s_cls[tid] = 0;
            } else {
                for (uint32_t e = tid; e < nsurv; e += T) { const uint2 pr = list[e]; apply_pair<PASS_FILL>(g, r, (int)pr.x, load_pair<PASS_FILL>(g, (int)pr.x, (int)pr.y)); }
            }
            }
            __syncthreads();
            // keys, bitmaps and the derived per-block arrays out: ascending (row, bit index) = ascending key
            for (int w = tid; w < nwords; w += T) {
                uint32_t word = r.bitset[w];
                if (!word) continue;
                int c = (int)r.wrank[w];
                const int rl = local_row(s_wo, nr, w);
                const int jw = s_jb[rl] + (w - s_wo[rl]) * 32;
                while (word) {
                    const int bit = __ffs(word) - 1;
                    word &= word - 1;
                    const int j = jw + bit;
                    const uint64_t bm = r.cbmp[c];
                    g.c_keys[c0 + c] = ((uint64_t)(uint32_t)(r.row + rl) << 32) | (uint32_t)j;
                    g.c_bcol[c0 + c] = j;
                    g.c_kmask[c0 + c] = (uint8_t)kmask_of(bm);
                    if (cfit) g.c_bmps[c0 + c] = bm;
                    c++;
                }
            }
            __syncthreads();
            // value offsets: scanned over the work item, then made relative to each block's own row (NUMERIC rebases them once the
            // row totals are scanned)
            const uint32_t rn = scan_popc(r.cbmp, g.c_off + c0, ccount, s_tmp);
            if (tid <= nr) { const int cs = s_cbr[tid] - c0; s_rowoff[tid] = cs < ccount ? (uint32_t)g.c_off[c0 + cs] : rn; }
            __syncthreads();
            if (nr > 1)
                for (int c = tid; c < ccount; c += T) g.c_off[c0 + c] -= s_rowoff[local_row(s_cbr, nr, c0 + c)];
            if (tid < nr) g.row_nnz[lrow + tid] = s_rowoff[tid + 1] - s_rowoff[tid];
            if (tid == 0) my_max2 = max(my_max2, (int)min(rn, 0x7FFFFFFFu));
        }
        if (PASS == PASS_NUMERIC || PASS == PASS_NUMERIC_MMA) {
            const uint64_t vbase = g.row_nnz[lrow];
            const int64_t rownnz = (int64_t)(g.row_nnz[lrow + nr] - vbase);
            const bool fit = PASS == PASS_NUMERIC ? (ccount <= g.cap_c && rownnz <= g.cap_nnz) : (ccount <= g.cap_c);
            for (int c = tid; c < ccount; c += T) {
                const int rl = local_row(s_cbr, nr, c0 + c);
                // relative to the work item's first value
                const uint64_t local = REUSE ? g.c_off[c0 + c] - vbase : s_rowoff[rl] + g.c_off[c0 + c];
                if (PASS == PASS_NUMERIC && fit) { s_cbmp[c] = g.c_bmps[c0 + c]; s_coff[c] = (uint32_t)local; }
                if (!REUSE) g.c_off[c0 + c] = vbase + local;                 // absolute from here on
                const int j = g.c_bcol[c0 + c] - s_jb[rl];                   // bit set from C's own block columns
                atomicOr(&r.bitset[s_wo[rl] + (j >> 5)], 1u << (j & 31));
            }
            if (PASS == PASS_NUMERIC && fit) {
                r.cbmp = s_cbmp; r.coff = s_coff; r.acc = s_acc;
                for (int v = tid; v < rownnz; v += T) s_acc[v] = 0.f;
            }
            if (PASS == PASS_NUMERIC_MMA && fit) {
                r.dense = s_dense;
                for (int v = tid; v < ccount * 64; v += T) s_dense[v] = 0.f;
            }
            __syncthreads();
            scan_popc(r.bitset, r.wrank, nwords, s_tmp);
            if (PASS == PASS_NUMERIC && g.f_ptr) {
                uint32_t ns = 0;
                enumerate_fine<2, false>(g, r, ns);
            } else if (PASS == PASS_NUMERIC) {
                if (g.split8) {
                    // the segment is sorted by class (FILL): h pairs with eight lanes each -- one per row of the A block --, then the
                    // pairs whose A block has one or two values, one lane each.  An unsorted segment (too many pairs for FILL's
                    // registers) carries no flags: h = nsurv.
                    uint32_t h = nsurv;
                    if (nsurv <= (uint32_t)g.sort_max) {
                        h = 0;
                        for (uint32_t e0 = 0; e0 < nsurv; e0 += T) h += (uint32_t)__syncthreads_count(e0 + tid < nsurv && !(list[e0 + tid].x & PAIR_LIGHT_FLAG));
                    }
                    for (uint64_t e = tid; e < (uint64_t)h * 8u; e += T) {
                        const uint2 pr = list[e >> 3]; const int a = (int)(pr.x & ~PAIR_LIGHT_FLAG);
                        apply_pair<PASS_NUMERIC>(g, r, a, load_pair<PASS_NUMERIC>(g, a, (int)pr.y), (int)(e & 7u));
                    }
                    for (uint32_t e = h + tid; e < nsurv; e += T) {
                        const uint2 pr = list[e]; const int a = (int)(pr.x & ~PAIR_LIGHT_FLAG);
                        apply_pair<PASS_NUMERIC>(g, r, a, load_pair<PASS_NUMERIC>(g, a, (int)pr.y));
                    }
                } else if (MAXT == 1024) {            // 32 registers per thread: one pair at a time
                    for (uint32_t e = tid; e < nsurv; e += T) { const uint2 pr = list[e]; apply_pair<PASS_NUMERIC>(g, r, (int)pr.x, load_pair<PASS_NUMERIC>(g, (int)pr.x, (int)pr.y)); }
                } else {
                    for (uint32_t e = tid; e < nsurv; e += 2 * T) {       // two pairs' loads in flight
                        const bool two = e + T < nsurv;
                        const uint2 p0 = list[e], p1 = two ? list[e + T] : make_uint2(0, 0);
                        const PairIn i0 = load_pair<PASS_NUMERIC>(g, (int)p0.x, (int)p0.y);
                        PairIn i1 = i0;
                        if (two) i1 = load_pair<PASS_NUMERIC>(g, (int)p1.x, (int)p1.y);
                        apply_pair<PASS_NUMERIC>(g, r, (int)p0.x, i0);
                        if (two) apply_pair<PASS_NUMERIC>(g, r, (int)p1.x, i1);
                    }
                }
            } else if (!fit) {
                // too many C blocks for the dense accumulators: scalar products into global memory.  The row's pairs are enumerated
                // again rather than read from the pair list: FILL may have written the list a group of rows at a time
                enumerate_row<PASS_NUMERIC>(g, r, q);
            } else {
                // every warp enumerates its own A blocks, so the pairs of an A block stay adjacent in its queue (two B blocks per MMA);
                // walking FILL's pair list instead of enumerating a third time measured no faster (BC4M 19.2 vs 18.6 ms)
                enumerate_row<PASS_NUMERIC_MMA>(g, r, q);
            }
            __syncthreads();
            if (PASS == PASS_NUMERIC && fit) for (int v = tid; v < rownnz; v += T) g.c_val[vbase + v] = s_acc[v];
            if (PASS == PASS_NUMERIC_MMA && fit) {
                // compact the dense accumulators through C's bitmaps: slot L <-> cell (r = 2t, c = g), slot L+32 <-> (2t+1, g)
                const int P0 = (lane & 3) * 16 + (lane >> 2);
                for (int c = wid; c < ccount; c += nwarps) {
                    const uint64_t bmp = g.c_bmps[c0 + c];
                    float* dst = g.c_val + g.c_off[c0 + c];
                    if ((bmp >> (63 - P0)) & 1ull) dst[rank64(bmp, P0)] = s_dense[c * 64 + lane];
                    if ((bmp >> (55 - P0)) & 1ull) dst[rank64(bmp, P0 + 8)] = s_dense[c * 64 + 32 + lane];
                }
            }
        }
        __syncthreads();
    }
    if (my_max1) atomicMax(&g.ctr->max_c_item, my_max1);
    if (my_max2) atomicMax(&g.ctr->max_nnz_item, my_max2);
    if (my_max3) atomicMax(&g.ctr->max_c_row, my_max3);
    if (PASS == PASS_COUNT) {
#pragma unroll
        for (int o = 16; o; o >>= 1) n_surv_total += __shfl_xor_sync(0xffffffffu, n_surv_total, o);
        if (lane == 0) atomicAdd(&g.ctr->surviving, n_surv_total);
    }
}

// ---- dense-block numeric pass, narrow rows (block-clustered / banded operands) -------------------------------------------------
// The generic mma.sync pass above fetches every fragment element with its own rank + 2-byte global load (two dependent latencies
// per fragment, 32 scattered loads) and keeps 12 two-warp CTAs per SM busy at 19 % warps active (ncu, round 1: BC4M 18.5 ms).
// Here one warp owns a block row.  A block's compact values are read ONCE, coalesced (lane l takes values l and l + 32 of the
// block, packed in one register); a fragment element is then a rank (shift + popc) and a warp shuffle -- no dependent load.  Two
// B^t blocks are stacked as the 16x8 A-operand of mma.m16n8k8, the A block is the B-operand, D = the two 8x8 products transposed;
// each lane owns two fixed slots of every dense C block in shared memory, so the accumulation needs no atomics.  The loads of the
// next pair of B blocks are issued before the current MMA.  C block index of a pair: a per-row table over the row's column span.

// values l and l + 32 of a block (cnt values from vals + off) in one register: low half = value l, high half = value l + 32
__device__ __forceinline__ uint32_t load_block_vals(const __half* __restrict__ vals, uint32_t off, int cnt, int lane) {
    const unsigned short lo = lane < cnt ? __half_as_ushort(__ldg(vals + off + lane)) : (unsigned short)0;
    const unsigned short hi = lane + 32 < cnt ? __half_as_ushort(__ldg(vals + off + 32 + lane)) : (unsigned short)0;
    return (uint32_t)lo | ((uint32_t)hi << 16);
}
// fragment register for cells p0, p0 + 1 of a block whose values sit in the warp as packed by load_block_vals
__device__ __forceinline__ uint32_t frag_shfl(uint64_t bmp, uint32_t packed, int p0) {
    const uint32_t two = (uint32_t)(bmp >> (62 - p0)) & 3u;        // bit1 = cell p0, bit0 = cell p0+1
    const int r0 = rank64(bmp, p0), r1 = r0 + (int)(two >> 1);
    const uint32_t w0 = __shfl_sync(0xffffffffu, packed, r0 & 31), w1 = __shfl_sync(0xffffffffu, packed, r1 & 31);
    const uint32_t v0 = (r0 & 32) ? (w0 >> 16) : (w0 & 0xFFFFu), v1 = (r1 & 32) ? (w1 >> 16) : (w1 & 0xFFFFu);
    return ((two & 2u) ? v0 : 0u) | (((two & 1u) ? v1 : 0u) << 16);
}

// One warp per block row; the row's C block columns are covered in windows of DENSE_WCOLS columns so that a warp's dense
// accumulators stay small (16 columns: 4 KB per warp, 48 warps per SM; BC4M NUMERIC 17.7 -> 10.1 ms against the generic MMA pass;
// with all of a 63-column row resident the SM held 12 warps and the pass waited on its own loads: 23.7 ms).  Per A block the lanes
// test the B block row in parallel (block column inside the window, inner-dimension masks overlap) and the survivors are taken two
// at a time off the ballot.
constexpr int DENSE_WARPS = 4, DENSE_WCOLS = 16;
template <bool REUSE = false>      // as spgemm_pass_kernel's
__global__ void __launch_bounds__(DENSE_WARPS * 32) spgemm_dense_kernel(GemmArgs g) {
    __shared__ float s_dense_all[DENSE_WARPS * DENSE_WCOLS * 64];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    float* s_dense = s_dense_all + wid * DENSE_WCOLS * 64;
    const int p0 = (lane >> 2) * 8 + (lane & 3) * 2;
    const int P0 = (lane & 3) * 16 + (lane >> 2);          // slot L <-> cell (r = 2t, c = g), slot L + 32 <-> (2t + 1, g)
    const int nrows = g.row_end - g.row_begin;
    for (;;) {
        int lrow = 0;
        if (lane == 0) lrow = atomicAdd(g.work_counter, 1);
        lrow = __shfl_sync(0xffffffffu, lrow, 0);
        if (lrow >= nrows) break;
        const int row = g.row_begin + lrow;
        const int c0 = g.c_brp[lrow], ccount = g.c_brp[lrow + 1] - c0;
        if (ccount == 0) continue;
        if (!REUSE) {
            const uint64_t vbase = g.row_nnz[lrow];
            for (int c = lane; c < ccount; c += 32) g.c_off[c0 + c] += vbase;   // FILL left row-relative offsets: absolute from here on
        }
        const int jfirst = g.c_bcol[c0], jlast = g.c_bcol[c0 + ccount - 1];
        const int a0 = g.a_brp[row], a1 = g.a_brp[row + 1];
        int cdone = 0;                                                           // C blocks of the windows already stored
        for (int jw = jfirst; jw <= jlast; jw += DENSE_WCOLS) {
            for (int v = lane; v < DENSE_WCOLS * 64; v += 32) s_dense[v] = 0.f;
            __syncwarp();
            for (int a = a0; a < a1; a++) {
                const int k = g.a_bcol[a];
                const uint32_t am = g.a_kmask[a];
                const int b0 = g.b_brp[k], b1 = g.b_brp[k + 1];
                uint32_t fb = 0; bool have_fb = false;
                for (int bb = b0; bb < b1; bb += 32) {
                    const int b = bb + lane;
                    bool in = false;
                    if (b < b1) { const int j = g.b_bcol[b] - jw; in = j >= 0 && j < DENSE_WCOLS && (am & g.b_kmask[b]) != 0; }
                    uint32_t mask = __ballot_sync(0xffffffffu, in);
                    if (!mask) continue;
                    if (!have_fb) {
                        const uint64_t abmp = g.a_bmps[a];
                        fb = frag_shfl(abmp, load_block_vals(g.a_val, (uint32_t)g.a_off[a], __popcll(abmp), lane), p0);
                        have_fb = true;
                    }
                    // survivors two at a time; the record and the values of the next pair are loaded before this pair's MMA
                    auto take = [&](uint4& rec, uint32_t& pk) {
                        const int l = __ffs(mask) - 1;
                        mask &= mask - 1;
                        rec = __ldg(g.b_pm + 2 * (int64_t)(bb + l));
                        pk = load_block_vals(g.b_val, rec.w, __popc(rec.x) + __popc(rec.y), lane);
                    };
                    uint4 r0 = make_uint4(0, 0, 0, 0), r1 = r0, n0 = r0, n1 = r0; uint32_t k0 = 0, k1 = 0, m0 = 0, m1 = 0;
                    bool two = false, ntwo = false, more;
                    take(r0, k0);
                    if (mask) { take(r1, k1); two = true; }
                    for (;;) {
                        more = mask != 0;
                        if (more) { take(n0, m0); ntwo = mask != 0; if (ntwo) take(n1, m1); }
                        const uint32_t fa0 = frag_shfl(((uint64_t)r0.y << 32) | r0.x, k0, p0);
                        const uint32_t fa1 = two ? frag_shfl(((uint64_t)r1.y << 32) | r1.x, k1, p0) : 0u;
                        float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
                        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                                     : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3) : "r"(fa0), "r"(fa1), "r"(fb));
                        float* q0 = s_dense + ((int)r0.z - jw) * 64 + lane;
                        q0[0] += d0; q0[32] += d1;
                        if (two) { float* q1 = s_dense + ((int)r1.z - jw) * 64 + lane; q1[0] += d2; q1[32] += d3; }
                        if (!more) break;
                        r0 = n0; k0 = m0; r1 = n1; k1 = m1; two = ntwo;
                    }
                }
            }
            __syncwarp();
            // the window's C blocks out: compact the dense accumulators through C's bitmaps
            while (cdone < ccount) {
                const int j = g.c_bcol[c0 + cdone] - jw;
                if (j >= DENSE_WCOLS) break;
                const uint64_t bmp = g.c_bmps[c0 + cdone];
                float* dst = g.c_val + g.c_off[c0 + cdone];
                if ((bmp >> (63 - P0)) & 1ull) dst[rank64(bmp, P0)] = s_dense[j * 64 + lane];
                if ((bmp >> (55 - P0)) & 1ull) dst[rank64(bmp, P0 + 8)] = s_dense[j * 64 + 32 + lane];
                cdone++;
            }
            __syncwarp();
        }
    }
}

static size_t pass_smem_bytes(int pass, int T, int cap_words, int cap_c, int cap_nnz, int group) {
    size_t s = 0;
    if (pass == PASS_FILL || pass == PASS_NUMERIC) s += (size_t)cap_c * 8;
    if (pass == PASS_NUMERIC_MMA) s += (size_t)(T / 32) * QSLOTS * 8;
    s += (size_t)cap_words * ((pass == PASS_COUNT && group == 1) ? 4 : 8);
    if (pass == PASS_NUMERIC) s += (size_t)cap_c * 4 + (size_t)cap_nnz * 4;
    if (pass == PASS_NUMERIC_MMA) s += (size_t)cap_c * 64 * 4;
    s += (38 + 33 + 32 + 33 + 33 + 32 + 33) * 4 + 16;      // s_tmp, row / cursor / batch words, the per-row tables
    return s;
}

// C's derived row arrays: block-row pointers and value bases for every block row of the full matrix
// (rows outside [rb, re) are empty in a sharded product).
__global__ void finish_rows_kernel(const uint32_t* __restrict__ c_brp_local, const uint64_t* __restrict__ row_vbase, int rb, int re,
                                   int nbr, int32_t* __restrict__ brp, uint32_t* __restrict__ rvb, uint64_t* __restrict__ c_off,
                                   int64_t c_size, uint64_t c_nnz) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) c_off[c_size] = c_nnz;
    if (r > nbr) return;
    if (r < rb) { brp[r] = 0; rvb[r] = 0; }
    else if (r >= re) { brp[r] = (int32_t)c_size; rvb[r] = (uint32_t)c_nnz; }
    else { brp[r] = (int32_t)c_brp_local[r - rb]; rvb[r] = (uint32_t)row_vbase[r - rb]; }
}

}  // namespace bmsp

using namespace bmsp;

extern "C" int bmsp_debug_pair_bitmap(int64_t n, const uint64_t* a_host, const uint64_t* bt_host, uint64_t* out_host) {
    DevBuf<uint64_t> a, b, o;
    cudaStream_t st = 0;
    BMSP_TRY(a.alloc((size_t)n, st)); BMSP_TRY(b.alloc((size_t)n, st)); BMSP_TRY(o.alloc((size_t)n, st));
    BMSP_CUDA(cudaMemcpyAsync(a.get(), a_host, 8 * n, cudaMemcpyHostToDevice, st));
    BMSP_CUDA(cudaMemcpyAsync(b.get(), bt_host, 8 * n, cudaMemcpyHostToDevice, st));
    pair_bitmap_test_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(a.get(), b.get(), o.get(), n);
    BMSP_KERNEL_CHECK();
    BMSP_CUDA(cudaMemcpyAsync(out_host, o.get(), 8 * n, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    return BMSP_OK;
}

template <int PASS, int MAXT, bool REUSE = false>
static int launch_pass_t(const GemmArgs& g, int T, int sms, int nrows, cudaStream_t st) {
    const size_t smem = pass_smem_bytes(PASS, T, g.cap_words, g.cap_c, g.cap_nnz, g.row_list ? 1 : g.group);
    auto kern = spgemm_pass_kernel<PASS, MAXT, REUSE>;
    BMSP_TRY(kernel_smem((const void*)kern, smem, false));
    int occ = 0;
    BMSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, T, smem));
    if (occ < 1) { set_error("spgemm pass %d does not fit: smem %zu", PASS, smem); return BMSP_ERR_CUDA; }
    int grid = (int)std::min<int64_t>((int64_t)sms * occ, (int64_t)nrows);
    grid = std::max(grid, 1);
    BMSP_CUDA(cudaMemsetAsync(g.work_counter, 0, sizeof(int32_t), st));
    kern<<<grid, T, smem, st>>>(g);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

// Heavy block rows (hub rows of power-law inputs: 10^6..10^8 candidate pairs each) are taken out of the row queue and run
// first, heaviest first, by 1024-thread CTAs on a second stream, while the 256-thread CTAs of the main launch work through the
// light rows: one CTA per row stays the unit of work, but a hub row gets four times the threads and no longer ends up as the
// tail of the launch.
struct RowSplit {
    bool active = false;
    DevBuf<int32_t> list;          // heavy rows (descending weight) then light rows (ascending index)
    int n_heavy = 0, n_light = 0;
    Stream side;
    Event fork, join;
    size_t heavy_scratch_off = 0;  // words: the heavy launch's slice of g_bitset / g_wrank
};

template <int PASS, bool REUSE = false>
static int launch_pass(GemmArgs& g, int T, int sms, cudaStream_t st, const RowSplit& sp) {
    if (!sp.active) {
        if (T > 256) return launch_pass_t<PASS, 1024, REUSE>(g, T, sms, (int)ceil_div(g.row_end - g.row_begin, g.group), st);
        return launch_pass_t<PASS, 256, REUSE>(g, T, sms, (int)ceil_div(g.row_end - g.row_begin, g.group), st);
    }
    GemmArgs gh = g, gl = g;
    gh.group = gl.group = 1;
    gh.row_list = sp.list.get(); gh.n_list = sp.n_heavy; gh.work_counter = g.work_counter + 1; gh.G = 32; gh.batch = 1;
    if (g.g_bitset) { gh.g_bitset = g.g_bitset + sp.heavy_scratch_off; gh.g_wrank = g.g_wrank + sp.heavy_scratch_off; }
    gl.row_list = sp.list.get() + sp.n_heavy; gl.n_list = sp.n_light;
    BMSP_CUDA(cudaEventRecord(sp.fork.get(), st));
    BMSP_CUDA(cudaStreamWaitEvent(sp.side.get(), sp.fork.get(), 0));
    BMSP_TRY((launch_pass_t<PASS, 1024, REUSE>(gh, 1024, sms, sp.n_heavy, sp.side.get())));
    if (sp.n_light > 0) BMSP_TRY((launch_pass_t<PASS, 256, REUSE>(gl, T, sms, sp.n_light, st)));
    BMSP_CUDA(cudaEventRecord(sp.join.get(), sp.side.get()));
    BMSP_CUDA(cudaStreamWaitEvent(st, sp.join.get(), 0));
    return BMSP_OK;
}

static double block_density(const bmsp_matrix_s* m) { return m->nblk ? (double)m->nnz / m->nblk : 0.0; }
static int clampi(double v, int lo, int hi) { return (int)std::min<double>(hi, std::max<double>(lo, v)); }

// Row statistics and the heavy-row split.  rowinfo_kernel writes every block row's bit-set span and candidate pairs and reduces
// the maxima and sums into ctr; they are read back into h.  Rows with at least BMSP_SPGEMM_HEAVY candidate pairs (default 2^20;
// 0 disables the split) are heavy when the heaviest row has four times that.  The variable is a test hook:
// tests/test_gpu_spgemm.py::test_heavy_row_split lowers it so that small inputs run the split.
static int plan_rows(const bmsp_matrix_s* A, const bmsp_matrix_s* Bt, int rb, int re, int sms, int2* rowinfo, unsigned long long* cand,
                     Counters* ctr, Counters& h, RowSplit& sp, cudaStream_t st) {
    const int nrows = re - rb;
    if (nrows > 0) {
        rowinfo_kernel<<<(unsigned)std::min<int64_t>(ceil_div(nrows, 8), (int64_t)sms * 8), 256, 0, st>>>(A->brp, A->bcol, Bt->brp, Bt->bcol, rb, re,
                                                                                                        rowinfo, cand, ctr);
        BMSP_KERNEL_CHECK();
    }
    BMSP_CUDA(cudaMemcpyAsync(&h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    const char* e = getenv("BMSP_SPGEMM_HEAVY");
    const long long heavy_min = e ? atoll(e) : (1ll << 20);
    if (heavy_min <= 0 || nrows <= 1 || h.max_cand < 4ull * (unsigned long long)heavy_min) return BMSP_OK;
    std::vector<unsigned long long> hc((size_t)nrows);
    BMSP_CUDA(cudaMemcpyAsync(hc.data(), cand, sizeof(unsigned long long) * (size_t)nrows, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> heavy, order;
    for (int i = 0; i < nrows; i++) if (hc[i] >= (unsigned long long)heavy_min) heavy.push_back(rb + i);
    std::sort(heavy.begin(), heavy.end(), [&](int32_t x, int32_t y) { return hc[x - rb] != hc[y - rb] ? hc[x - rb] > hc[y - rb] : x < y; });
    order = heavy;
    for (int i = 0; i < nrows; i++) if (hc[i] < (unsigned long long)heavy_min) order.push_back(rb + i);
    sp.n_heavy = (int)heavy.size(); sp.n_light = nrows - sp.n_heavy;
    BMSP_TRY(sp.list.alloc((size_t)nrows + 1, st));
    BMSP_CUDA(cudaMemcpyAsync(sp.list.get(), order.data(), sizeof(int32_t) * (size_t)nrows, cudaMemcpyHostToDevice, st));
    BMSP_CUDA(cudaStreamSynchronize(st));       // `order` dies with this scope
    BMSP_TRY(new_stream(sp.side));
    BMSP_TRY(new_event(sp.fork));
    BMSP_TRY(new_event(sp.join));
    sp.active = sp.n_heavy > 0;
    return BMSP_OK;
}

// What products build for a matrix used as their B operand, once, and reuse (bmsp_matrix_s::bidx; created by ensure_pmeta)
struct bmsp::BIndex {
    DevBuf<uint4> pmeta;         // [nblk] 32-byte records {bitmap lo, hi, block column, value offset}, {first 8 values} (none if nblk == 0)
    // sparse-block operands: B's blocks bucketed by inner index (block row k, bit t of kmask), the "fine index"
    enum { UNEXAMINED, BUILT, NOT_WORTH_IT } fine_state = UNEXAMINED;   // not worth it: dense blocks, the buckets would replicate every block ~8 times
    DevBuf<uint32_t> fine_ptr;   // [nbr * 8 + 1] bucket offsets
    DevBuf<uint32_t> fine_bcol;  // [entries] block column of the bucket entry
    DevBuf<uint8_t> fine_kmask;  // [entries] kmask of the bucket entry's block (de-duplicates blocks that sit in several buckets)
    DevBuf<uint4> fine_rec;      // [entries] 32-byte records as in pmeta
};

// the index's buffers free on the stream they were built on, in the same order as bmsp_destroy's frees (as for spmv_release)
void bmsp::bindex_release(bmsp_matrix_s* m) { delete m->bidx; m->bidx = nullptr; }

// the two copies of a B operand's values that products keep, (re)written in place: the packed block records and the fine index's
// (the destinations are arguments: a first build writes them before they are published in Bt)
static int pack_meta(const bmsp_matrix_s* Bt, uint4* pmeta, cudaStream_t st) {
    pack_meta_kernel<<<(unsigned)ceil_div(Bt->nblk, 256), 256, 0, st>>>(Bt->bmps, Bt->bcol, Bt->offsets, (const __half*)Bt->values, Bt->nnz,
                                                                      pmeta, Bt->nblk);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}
static int fine_fill(const bmsp_matrix_s* Bt, const uint32_t* fptr, uint32_t* fbcol, uint8_t* fkmask, uint4* frec, cudaStream_t st) {
    fine_fill_kernel<<<(unsigned)ceil_div((int64_t)Bt->nbr * 8, 128), 128, 0, st>>>(Bt->brp, Bt->kmask, Bt->bidx->pmeta.get(), Bt->nbr, fptr,
                                                                                   fbcol, fkmask, frec);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

int bmsp::refresh_value_copies(bmsp_matrix_s* m, cudaStream_t st) {
    const BIndex* bi = m->bidx;
    if (bi && bi->pmeta.get()) BMSP_TRY(pack_meta(m, bi->pmeta.get(), st));
    if (bi && bi->fine_state == BIndex::BUILT) BMSP_TRY(fine_fill(m, bi->fine_ptr.get(), bi->fine_bcol.get(), bi->fine_kmask.get(), bi->fine_rec.get(), st));
    return BMSP_OK;
}

// B's packed block records: built once per B operand, reused by later products
static int ensure_pmeta(bmsp_matrix_s* Bt, cudaStream_t st) {
    if (Bt->bidx) return BMSP_OK;
    std::unique_ptr<BIndex> bi(new BIndex());
    if (Bt->nblk > 0) {
        BMSP_TRY(bi->pmeta.alloc(2 * (size_t)Bt->nblk, st));
        BMSP_TRY(pack_meta(Bt, bi->pmeta.get(), st));
    }
    Bt->bidx = bi.release();
    return BMSP_OK;
}

// Fine index of B for sparse-block operands (about one value per block: uniform random, R-MAT): examined once per B operand, by
// the rule below only (U1M A*A: 30.8 ms by the candidate scan, 18.9 ms through the buckets).
static int ensure_fine_index(bmsp_matrix_s* Bt, const bmsp_matrix_s* A, cudaStream_t st) {
    BIndex& bi = *Bt->bidx;
    if (bi.fine_state != BIndex::UNEXAMINED || Bt->nblk == 0 || (int64_t)Bt->nbr * 8 + 1 >= 0x7FFFFFFFll) return BMSP_OK;
    if (!(block_density(Bt) <= 2.0 && block_density(A) <= 4.0)) return BMSP_OK;
    const size_t nb = (size_t)Bt->nbr * 8;
    DevBuf<uint32_t> fp;
    BMSP_TRY(fp.alloc(nb + 2, st));
    BMSP_CUDA(cudaMemsetAsync(fp.get(), 0, sizeof(uint32_t) * (nb + 2), st));
    fine_count_kernel<<<(unsigned)ceil_div(Bt->nblk, 256), 256, 0, st>>>(Bt->keys, Bt->kmask, Bt->nblk, fp.get());
    BMSP_KERNEL_CHECK();
    // the longest bucket: slot nb + 1 of the zeroed array
    fine_max_kernel<<<(unsigned)ceil_div((int64_t)nb, 256), 256, 0, st>>>(fp.get(), (int64_t)nb, fp.get() + nb + 1);
    BMSP_KERNEL_CHECK();
    uint32_t longest = 0, total = 0;
    BMSP_CUDA(cudaMemcpyAsync(&longest, fp.get() + nb + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    BMSP_TRY(exclusive_scan_u32(fp.get(), fp.get(), (int64_t)nb, st));
    BMSP_CUDA(cudaMemcpyAsync(&total, fp.get() + nb, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    // worth it while the buckets replicate little (a block with m inner indices sits in m buckets) and are of similar length:
    // a power-law B (R-MAT) has hub buckets of 10^4 entries next to a mean of 2, and the candidate scan, which spreads a B block
    // row over up to 32 lanes, handles those better (R-MAT-18 A*A: 164 ms by scan, 181 ms through the buckets)
    const double mean_bucket = (double)total / std::max<double>(1.0, (double)nb);
    const bool even = (double)longest <= 32.0 * std::max(mean_bucket, 1.0) || longest <= 512;
    if (!((double)total <= 1.5 * (double)Bt->nblk && even)) { bi.fine_state = BIndex::NOT_WORTH_IT; return BMSP_OK; }
    DevBuf<uint32_t> fbcol; DevBuf<uint8_t> fkmask; DevBuf<uint4> frec;
    BMSP_TRY(fbcol.alloc((size_t)total + 4, st));
    BMSP_TRY(fkmask.alloc((size_t)total + 16, st));
    BMSP_TRY(frec.alloc(2 * ((size_t)total + 1), st));
    BMSP_TRY(fine_fill(Bt, fp.get(), fbcol.get(), fkmask.get(), frec.get(), st));
    bi.fine_ptr = std::move(fp); bi.fine_bcol = std::move(fbcol); bi.fine_kmask = std::move(fkmask); bi.fine_rec = std::move(frec);
    bi.fine_state = BIndex::BUILT;
    return BMSP_OK;
}

// The numeric path: the requested one, else by about dA * dB / 8 products per surviving pair (dA, dB: values per block) -- scalar
// lanes for sparse blocks, mma.sync from 40 on
static int numeric_path(const bmsp_matrix_s* A, const bmsp_matrix_s* Bt, const bmsp_spgemm_opts* opts) {
    const int path = opts ? opts->numeric_path : -1;
    return path >= 0 ? path : (block_density(A) * block_density(Bt) / 8.0 >= 40.0 ? 1 : 0);
}

struct Plan {
    int T;           // threads per CTA of COUNT, FILL and the scalar NUMERIC pass
    int mma_batch;   // work items per queue atomic of the generic MMA pass
};

// Launch shape of the passes from the operands' averages and the row statistics: fills g's shape fields.
static Plan plan_launch(GemmArgs& g, const bmsp_matrix_s* A, const bmsp_matrix_s* Bt, int nrows, const Counters& h, bool split,
                        bool fine, int path) {
    const double avgB = Bt->nbr ? (double)Bt->nblk / Bt->nbr : 0.0;
    const double avgA = A->nbr ? (double)A->nblk / A->nbr : 0.0;
    const double avg_cand = avgA * avgB;
    // G lanes share one A block, each lane tests 4 B blocks per step
    int G = 1;
    while (G < 32 && G * 4 < avgB) G <<= 1;
    // Tiny rows (stencils: 25 candidate pairs per block row) are processed 16 rows at a time by 128-thread CTAs: one warp per row
    // leaves the SM at 32 one-warp CTAs, each waiting on its own chain of dependent loads (P4096 A*A: 21.7 ms, cuSPARSE 13.0 ms;
    // 8 rows per work item: 12.7 ms, 16: 12.3 ms).  P4096 has 2.1 M block rows: one atomic on the queue head per row and pass cost
    // more than the rows
    const int group = (avg_cand <= 96 && !split && (int64_t)16 * h.max_words <= 8192) ? 16 : 1;
    int T = group > 1 ? 128 : (avg_cand <= 96 ? 32 : (avg_cand <= 2048 ? 128 : 256));
    // Walking B's fine index a row's passes wait on record loads and are held to 3-4 CTAs per SM by the row's bit set in shared
    // memory: more threads per CTA are more loads in flight for the same shared memory (512 threads; no measurement of 256 / 512 /
    // 1024 is recorded)
    if (fine && T == 256 && !split) T = 512;
    g.G = G;
    g.group = group;
    // (four / two lanes per pair with two / four rows each were measured on P4096: NUMERIC 8.35 / 8.97 ms against 7.45 ms with eight)
    g.split8 = block_density(A) >= 4.0;
    // FILL sorts its pair-list segments by class only for the pass that reads them, the scalar NUMERIC pass with 8 lanes per pair
    // (P4096 A*A: 11.5 ms unsorted, 8.0 ms sorted)
    g.sort_max = (g.split8 && path == 0) ? SORT_K * T : 0;
    g.batch = group > 1 ? 2 : (avg_cand <= 96 ? 32 : (avg_cand <= 2048 ? 4 : 1));
    // Shared-memory capacities decide how many CTAs an SM holds, and these passes are latency-bound: size them for the rows
    // that can use them.  When every row fits, take the maxima; when the typical row would not fit anyway (R-MAT: C rows of
    // 10^4..10^5 blocks spanning every block column), keep the CTAs small -- those rows run from global scratch / global
    // atomics either way and need the occupancy (R-MAT-17 NUMERIC: 102 KB per CTA = 2 CTAs per SM, 14 % issue utilisation).
    const double avg_words = nrows ? (double)h.sum_words / nrows : 0.0;
    g.cap_words = (int64_t)group * h.max_words <= 8192 ? std::max(1, group * h.max_words) : (avg_words > 4096.0 ? 256 : 8192);
    g.max_words = group * h.max_words;
    return Plan{T, avg_cand <= 96 ? 32 : 1};
}

// NUMERIC: the dense-block kernel for narrow rows of dense blocks, the generic mma.sync pass for the other dense-block products,
// the scalar pass for sparse blocks.  REUSE: a kept plan's rerun (C's offsets are absolute).  Every launch zeroes its own queue heads,
// and C's values are zeroed here whenever rows accumulate with global atomics, so a rerun needs nothing else reset.
template <bool REUSE = false>
static int run_numeric(GemmArgs& g, const bmsp_matrix_s* C, const Counters& h, const Plan& plan, int path, const RowSplit& sp, int nrows,
                       int sms, cudaStream_t st) {
    if (path == 1 && !sp.active && (int64_t)h.max_words * 32 <= 1024) {
        // narrow rows: one warp per block row, dense accumulators for a window of C columns in shared memory
        int occ = 0;
        BMSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, spgemm_dense_kernel<REUSE>, DENSE_WARPS * 32, 0));
        if (occ < 1) { set_error("spgemm dense pass does not fit"); return BMSP_ERR_CUDA; }
        BMSP_CUDA(cudaMemsetAsync(g.work_counter, 0, sizeof(int32_t), st));
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)sms * occ, ceil_div(nrows, DENSE_WARPS)));
        spgemm_dense_kernel<REUSE><<<grid, DENSE_WARPS * 32, 0, st>>>(g);
        BMSP_KERNEL_CHECK();
        return BMSP_OK;
    }
    if (path == 1) {
        const int max_c_row = std::max(1, h.max_c_row);
        GemmArgs gm = g;
        gm.cap_c = std::min(max_c_row, 192);
        if (max_c_row > gm.cap_c) BMSP_CUDA(cudaMemsetAsync(C->values, 0, (size_t)C->nnz * 4, st));
        gm.group = 1; gm.batch = plan.mma_batch;          // one block row per work item: pairs of an A block stay adjacent
        // two warps per block row, sharing the row's accumulators (BC4M numeric, one box: 32 threads 19.5 ms, 64: 17.7 ms, 128:
        // 20.2 ms -- a row has ~10 A blocks x 4 lanes to hand out)
        return launch_pass_t<PASS_NUMERIC_MMA, 256, REUSE>(gm, 64, sms, nrows, st);
    }
    const int max_c = h.max_c_item, max_rownnz = h.max_nnz_item;
    const double avg_c = nrows ? (double)C->nblk / nrows : 0.0, avg_nnz = nrows ? (double)C->nnz / nrows : 0.0;
    if (max_c <= 4096 && max_rownnz <= 12288) { g.cap_c = std::max(1, max_c); g.cap_nnz = std::max(1, max_rownnz); }
    else if (avg_c <= 512.0 && avg_nnz <= 1536.0) { g.cap_c = clampi(4.0 * avg_c, 256, 2048); g.cap_nnz = clampi(4.0 * avg_nnz, 1024, 8192); }
    else { g.cap_c = 64; g.cap_nnz = 256; }
    if (max_c > g.cap_c || max_rownnz > g.cap_nnz) BMSP_CUDA(cudaMemsetAsync(C->values, 0, (size_t)C->nnz * 4, st));
    return launch_pass<PASS_NUMERIC, REUSE>(g, plan.T, sms, st, sp);
}

// What a product allocates, and the launch state of its NUMERIC pass.  bmsp_spgemm frees all of it after the product; a plan keeps
// what its NUMERIC launch reads (bmsp_spgemm_plan_create).  Members are destroyed in reverse order: `sp` drains its side stream
// before the scratch and C, which the side stream's launches use, are freed.
struct ProductState {
    HandlePtr C;                        // until spgemm_run hands it out
    DevBuf<int2> rowinfo; DevBuf<unsigned long long> cand; DevBuf<Counters> ctr;
    DevBuf<uint32_t> row_count, row_surv; DevBuf<uint64_t> row_nnz; DevBuf<uint2> surv_list;
    DevBuf<uint32_t> g_bitset, g_wrank;
    size_t surv_n = 0, scratch_n = 0;   // entries of surv_list and of each of g_bitset / g_wrank
    RowSplit sp;
    GemmArgs g;
    Counters h{};
    Plan plan{};
    int path = 0, nrows = 0, sms = 0;
    bool use_fine = false;
};

// C = A * Bt: COUNT, FILL, NUMERIC.  On success the scratch stays in `s` (the caller frees or keeps it with s); on failure C is
// destroyed with s.
static int spgemm_run(bmsp_matrix_t A, bmsp_matrix_t Bt, const bmsp_spgemm_opts* opts, cudaStream_t st, ProductState& s, bmsp_matrix_t* Cout,
                      bmsp_spgemm_info* info) {
    if (!A || !Bt || !Cout) { set_error("bmsp_spgemm: null argument"); return BMSP_ERR_INVALID; }
    if (A->transposed || !Bt->transposed) { set_error("bmsp_spgemm: A must be plain and B in transposed-operand form (SPGEMM.cu:1261-1262)"); return BMSP_ERR_INVALID; }
    if (A->dtype != BMSP_F16 || Bt->dtype != BMSP_F16) { set_error("bmsp_spgemm: operands must be fp16 (bmSparse_mult<half,float>)"); return BMSP_ERR_UNSUPPORTED; }
    if (A->cols != Bt->rows) { set_error("bmsp_spgemm: inner dimensions differ (%d vs %d)", A->cols, Bt->rows); return BMSP_ERR_INVALID; }
    touch(A, st); touch(Bt, st);
    int rb = 0, re = A->nbr;
    // brow_range_set: the range is taken literally ([r, r) multiplies nothing: a shard that owns no rows); without it the legacy
    // rule applies -- [0, 0) means all rows
    if (opts && (opts->brow_range_set || opts->brow_begin != 0 || opts->brow_end != 0)) { rb = opts->brow_begin; re = opts->brow_end; }
    if (rb < 0 || re > A->nbr || rb > re) { set_error("bmsp_spgemm: bad block-row range [%d,%d)", rb, re); return BMSP_ERR_INVALID; }
    const int nrows = re - rb;
    const bool verbose = opts && opts->verbose;

    const DeviceInfo* dev = nullptr;
    BMSP_TRY(current_device(&dev));
    const int sms = s.sms = dev->sms;

    Event ev[4];                 // start, after FILL, end, after COUNT
    if (verbose) for (Event& e : ev) BMSP_TRY(new_event(e, true));
    if (verbose) BMSP_CUDA(cudaEventRecord(ev[0].get(), st));

    // ---- scratch
    s.nrows = nrows;
    BMSP_TRY(s.rowinfo.alloc((size_t)nrows + 1, st));
    BMSP_TRY(s.cand.alloc((size_t)nrows + 1, st));
    BMSP_TRY(s.ctr.alloc(1, st));
    BMSP_TRY(s.row_count.alloc((size_t)nrows + 2, st));
    BMSP_TRY(s.row_surv.alloc((size_t)nrows + 2, st));
    BMSP_TRY(s.row_nnz.alloc((size_t)nrows + 2, st));
    Counters* ctr = s.ctr.get();
    uint32_t *row_count = s.row_count.get(), *row_surv = s.row_surv.get();
    uint64_t* row_nnz = s.row_nnz.get();
    BMSP_CUDA(cudaMemsetAsync(ctr, 0, sizeof(Counters), st));

    Counters& h = s.h;
    RowSplit& sp = s.sp;
    BMSP_TRY(plan_rows(A, Bt, rb, re, sms, s.rowinfo.get(), s.cand.get(), ctr, h, sp, st));
    BMSP_TRY(ensure_pmeta(Bt, st));
    BMSP_TRY(ensure_fine_index(Bt, A, st));
    const BIndex& bi = *Bt->bidx;
    const bool use_fine = s.use_fine = bi.fine_state == BIndex::BUILT;
    const int path = s.path = numeric_path(A, Bt, opts);

    GemmArgs& g = s.g;
    memset(&g, 0, sizeof(g));
    if (use_fine) { g.f_ptr = bi.fine_ptr.get(); g.f_bcol = bi.fine_bcol.get(); g.f_kmask = bi.fine_kmask.get(); g.f_rec = bi.fine_rec.get(); }
    g.b_pm = bi.pmeta.get();
    g.a_brp = A->brp; g.a_bcol = A->bcol; g.a_bmps = A->bmps; g.a_kmask = A->kmask; g.a_off = A->offsets; g.a_val = (const __half*)A->values;
    g.b_brp = Bt->brp; g.b_bcol = Bt->bcol; g.b_bmps = Bt->bmps; g.b_kmask = Bt->kmask; g.b_off = Bt->offsets; g.b_val = (const __half*)Bt->values;
    g.rowinfo = s.rowinfo.get(); g.row_begin = rb; g.row_end = re;
    g.work_counter = &ctr->queue[0]; g.ctr = ctr; g.row_count = row_count; g.row_surv = row_surv; g.row_nnz = row_nnz;
    const Plan plan = s.plan = plan_launch(g, A, Bt, nrows, h, sp.active, use_fine, path);

    if (g.max_words > g.cap_words) {
        // over-cap rows use per-CTA global scratch; size it for the largest persistent grid (32 CTAs/SM)
        sp.heavy_scratch_off = (size_t)sms * 32 * g.max_words;                // + 2 heavy CTAs per SM
        const size_t n = s.scratch_n = sp.heavy_scratch_off + (size_t)sms * 2 * g.max_words;
        BMSP_TRY(s.g_bitset.alloc(n, st));
        BMSP_TRY(s.g_wrank.alloc(n, st));
        g.g_bitset = s.g_bitset.get(); g.g_wrank = s.g_wrank.get();
    }

    // ---- COUNT: C blocks and surviving pairs per block row
    int64_t c_size = 0, n_surv = 0;
    if (nrows > 0) {
        BMSP_TRY(launch_pass<PASS_COUNT>(g, plan.T, sms, st, sp));
        BMSP_TRY(exclusive_scan_u32(row_count, row_count, nrows, st));
        BMSP_TRY(exclusive_scan_u32(row_surv, row_surv, nrows, st));
        uint32_t tot[2] = {0, 0};
        BMSP_CUDA(cudaMemcpyAsync(&tot[0], row_count + nrows, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaMemcpyAsync(&tot[1], row_surv + nrows, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaMemcpyAsync(&h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaStreamSynchronize(st));
        c_size = tot[0]; n_surv = tot[1];
    }
    if (verbose) BMSP_CUDA(cudaEventRecord(ev[3].get(), st));
    if (c_size > 0x7FFFFFFFll || h.surviving > 0xFFFFFFFFull) {
        set_error("product too large for one call: %lld C blocks, %llu surviving pairs (shard A's block rows with brow_begin/brow_end)",
                  (long long)c_size, h.surviving);
        return BMSP_ERR_TOO_LARGE;
    }
    const int max_c = h.max_c_item;

    BMSP_TRY(new_handle(A->rows, Bt->cols, c_size, -1, BMSP_F32, 0, st, s.C));      // values: once FILL has counted them
    bmsp_matrix_s* C = s.C.get();
    C->offsets_len = c_size + 1;
    C->nbr = (int32_t)ceil_div(C->rows, 8);
    BMSP_TRY(dev_alloc_t(&C->bcol, (size_t)c_size + 8, st));
    BMSP_TRY(dev_alloc_t(&C->kmask, (size_t)c_size + 16, st));
    BMSP_TRY(dev_alloc_t(&C->brp, (size_t)C->nbr + 1 + 8, st));
    BMSP_TRY(dev_alloc_t(&C->rvb, (size_t)C->nbr + 1 + 8, st));
    s.surv_n = use_fine ? (size_t)1 : (size_t)n_surv + 1;
    BMSP_TRY(s.surv_list.alloc(s.surv_n, st));
    g.c_brp = (const int32_t*)row_count; g.c_keys = C->keys; g.c_bmps = C->bmps; g.c_bcol = C->bcol; g.c_kmask = C->kmask;
    g.c_off = C->offsets; g.surv_list = s.surv_list.get();

    // ---- FILL: pair list, keys, bitmaps, row-relative value offsets
    const double avg_c = nrows ? (double)c_size / nrows : 0.0;
    g.cap_c = max_c <= 4096 ? std::max(1, max_c) : (avg_c <= 512.0 ? clampi(4.0 * avg_c, 256, 2048) : 64);
    if (c_size > 0) {
        if (max_c > g.cap_c) BMSP_CUDA(cudaMemsetAsync(C->bmps, 0, sizeof(uint64_t) * c_size, st));
        BMSP_TRY(launch_pass<PASS_FILL>(g, plan.T, sms, st, sp));
    } else if (nrows > 0) {
        BMSP_CUDA(cudaMemsetAsync(row_nnz, 0, sizeof(uint64_t) * ((size_t)nrows + 1), st));
    }
    BMSP_TRY(exclusive_scan_u64(row_nnz, row_nnz, nrows, st));
    uint64_t c_nnz = 0;
    BMSP_CUDA(cudaMemcpyAsync(&c_nnz, row_nnz + nrows, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(&h, ctr, sizeof(h), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    if (c_nnz > 0xFFFFFFFFull) { set_error("C has %llu values (> 2^32-1)", (unsigned long long)c_nnz); return BMSP_ERR_TOO_LARGE; }
    C->nnz = (int64_t)c_nnz;
    BMSP_TRY(dev_alloc(&C->values, (size_t)c_nnz * 4 + 16, st));
    if (verbose) BMSP_CUDA(cudaEventRecord(ev[1].get(), st));

    g.c_val = (float*)C->values;
    if (c_nnz > 0) BMSP_TRY(run_numeric(g, C, h, plan, path, sp, nrows, sms, st));
    finish_rows_kernel<<<(unsigned)ceil_div(C->nbr + 1, 256), 256, 0, st>>>(row_count, row_nnz, rb, re, C->nbr, C->brp, C->rvb, C->offsets, c_size, c_nnz);
    BMSP_KERNEL_CHECK();
    if (verbose) BMSP_CUDA(cudaEventRecord(ev[2].get(), st));

    if (info) {
        memset(info, 0, sizeof(*info));
        info->candidate_pairs = (int64_t)h.sum_cand; info->surviving_pairs = (int64_t)h.surviving;
        info->c_blocks = c_size; info->c_nnz = (int64_t)c_nnz; info->numeric_path = path;
        if (verbose) {
            BMSP_CUDA(cudaEventSynchronize(ev[2].get()));
            cudaEventElapsedTime(&info->symbolic_ms, ev[0].get(), ev[1].get());
            cudaEventElapsedTime(&info->numeric_ms, ev[1].get(), ev[2].get());
            cudaEventElapsedTime(&info->count_ms, ev[0].get(), ev[3].get());
            cudaEventElapsedTime(&info->fill_ms, ev[3].get(), ev[1].get());
            info->total_ms = info->symbolic_ms + info->numeric_ms;
        }
    }
    *Cout = s.C.release();
    return BMSP_OK;
}

extern "C" int bmsp_spgemm(bmsp_matrix_t A, bmsp_matrix_t Bt, const bmsp_spgemm_opts* opts, void* stream, bmsp_matrix_t* Cout,
                           bmsp_spgemm_info* info) {
    ProductState s;
    return spgemm_run(A, Bt, opts, (cudaStream_t)stream, s, Cout, info);
}

// ---- plans: C's structure kept, its values recomputed from the operands' current values ---------------------------------------
// A plan keeps what the chosen NUMERIC launch reads: the row tables (bit-set spans, C's block-row pointers, surviving-pair bases,
// value bases), the counters block (queue heads), the over-cap bit-set scratch, the heavy-row split (row list, side stream, events)
// and, for the scalar pass over the candidate scan only, FILL's pair list -- left sorted by pair class, which depends on bitmaps
// alone.  The fine-index walk, the dense-block kernel and the generic MMA pass enumerate their pairs and keep no list.
struct bmsp_spgemm_plan_s {
    bmsp_matrix_s *A = nullptr, *Bt = nullptr, *C = nullptr;
    ProductState s;
    int64_t bytes = 0;
    cudaStream_t last_stream = nullptr;   // stream ordering of the plan's scratch, as bmsp_matrix_s::last_stream (touch)
    bool multi_stream = false, touched = false;
};

static int64_t alloc_bytes(size_t n) { return n ? (int64_t)(n + BMSP_PAD_BYTES) : 0; }

extern "C" int bmsp_spgemm_plan_create(bmsp_matrix_t A, bmsp_matrix_t Bt, const bmsp_spgemm_opts* opts, void* stream,
                                       bmsp_spgemm_plan_t* plan, bmsp_matrix_t* Cout, bmsp_spgemm_info* info) {
    if (!plan) { set_error("bmsp_spgemm_plan_create: null argument"); return BMSP_ERR_INVALID; }
    *plan = nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    std::unique_ptr<bmsp_spgemm_plan_s> p(new bmsp_spgemm_plan_s());
    ProductState& s = p->s;
    BMSP_TRY(spgemm_run(A, Bt, opts, st, s, Cout, info));
    s.cand.reset();
    if (s.path == 1 || s.use_fine) { s.surv_list.reset(); s.g.surv_list = nullptr; s.surv_n = 0; }
    p->A = A; p->Bt = Bt; p->C = *Cout;
    touch(p.get(), st);
    const size_t nr = (size_t)s.nrows;
    p->bytes = alloc_bytes((nr + 1) * sizeof(int2)) + alloc_bytes(sizeof(Counters)) + 2 * alloc_bytes((nr + 2) * sizeof(uint32_t)) +
               alloc_bytes((nr + 2) * sizeof(uint64_t)) + alloc_bytes(s.surv_n * sizeof(uint2)) + 2 * alloc_bytes(s.scratch_n * sizeof(uint32_t)) +
               (s.sp.list.get() ? alloc_bytes((nr + 1) * sizeof(int32_t)) : 0);
    *plan = p.release();
    return BMSP_OK;
}

extern "C" int bmsp_spgemm_numeric(bmsp_spgemm_plan_t p, void* stream) {
    if (!p) { set_error("bmsp_spgemm_numeric: null plan"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(p->A, st); touch(p->Bt, st); touch(p->C, st); touch(p, st);
    if (p->C->nnz > 0) BMSP_TRY(run_numeric<true>(p->s.g, p->C, p->s.h, p->s.plan, p->s.path, p->s.sp, p->s.nrows, p->s.sms, st));
    return refresh_value_copies(p->C, st);
}

extern "C" int bmsp_spgemm_plan_bytes(bmsp_spgemm_plan_t p, int64_t* bytes) {
    if (!p || !bytes) { set_error("bmsp_spgemm_plan_bytes: null argument"); return BMSP_ERR_INVALID; }
    *bytes = p->bytes;
    return BMSP_OK;
}

extern "C" int bmsp_spgemm_plan_destroy(bmsp_spgemm_plan_t p) {
    if (!p) return BMSP_OK;
    if (p->multi_stream) cudaDeviceSynchronize();     // else the scratch is freed on the one stream the plan used
    delete p;
    return BMSP_OK;
}
