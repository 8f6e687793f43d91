// common.cuh -- shared internals of libbmsparse_b200 (handle layout, error plumbing, device helpers).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <cstdio>
#include <cstdarg>
#include <memory>
#include <utility>
#include <vector>
#include <algorithm>
#include "../../include/bmsparse_b200.h"

#define BMSP_PAD_BYTES 256   // every array is over-allocated so 16-byte bulk copies may overrun the tail

namespace bmsp { struct SpmvPlan; struct BIndex; }   // spmv.cu, spgemm.cu

// Device-resident matrix.  keys/bmps/offsets/values are the interchange surface of the reference (include/bmSpMatrix.h:28-31),
// bit-identical; brp/bcol/rvb/kmask are derived once; spmv / bidx are built by the first operation that needs them.
struct bmsp_matrix_s {
    int32_t rows = 0, cols = 0;
    int64_t nnz = 0, nblk = 0, offsets_len = 0;
    int32_t nbr = 0;            // block rows = ceil(rows/8)
    int32_t dtype = BMSP_F16;
    int32_t transposed = 0;
    uint64_t* keys = nullptr;
    uint64_t* bmps = nullptr;
    uint64_t* offsets = nullptr;
    void* values = nullptr;
    int32_t* brp = nullptr;     // [nbr+1] block-row pointers
    int32_t* bcol = nullptr;    // [nblk]  block column of each block
    uint32_t* rvb = nullptr;    // [nbr+1] first value index of each block row
    uint8_t* kmask = nullptr;   // [nblk]  OR of the 8 bitmap bytes: inner-dimension (k) occupancy
    bmsp::SpmvPlan* spmv = nullptr;   // the SpMV plan, built by the first product (with bmsp_spmv_host's pipeline); freed by spmv_release
    bmsp::BIndex* bidx = nullptr;     // SpGEMM's index of the matrix as a B operand, built by the first such product; freed by bindex_release
    // Stream ordering of the handle's memory: every entry point that enqueues work on the arrays records its stream here
    // (bmsp::touch).  bmsp_destroy frees on that stream, so the frees are ordered behind the kernels that still read or write the
    // arrays; a handle that was used on more than one stream is drained with a device synchronisation first.  Streams passed to
    // calls on a matrix must outlive it.
    cudaStream_t last_stream = nullptr;
    bool multi_stream = false, touched = false;
};

namespace bmsp {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define BMSP_CUDA(call)                                                            \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) return bmsp::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

#define BMSP_TRY(call)                     \
    do {                                   \
        int s__ = (call);                  \
        if (s__ != BMSP_OK) return s__;    \
    } while (0)

#define BMSP_KERNEL_CHECK() BMSP_CUDA(cudaGetLastError())

// record that work on m's memory was enqueued on st (see bmsp_matrix_s::last_stream; SpGEMM plans follow the same rule)
template <typename M>
inline void touch(M* m, cudaStream_t st) {
    if (m->touched && m->last_stream != st) m->multi_stream = true;
    m->last_stream = st; m->touched = true;
}

// stream-ordered allocation (+padding).  Freed with dev_free on the same stream.
int dev_alloc(void** p, size_t bytes, cudaStream_t st);
void dev_free(void* p, cudaStream_t st);
template <typename T>
inline int dev_alloc_t(T** p, size_t n, cudaStream_t st) { return dev_alloc((void**)p, n * sizeof(T), st); }

// One device allocation of n T, freed on the stream it was allocated on when the buffer goes out of scope.
template <typename T>
class DevBuf {
public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), st_(o.st_) { o.p_ = nullptr; }
    DevBuf& operator=(DevBuf&& o) noexcept { std::swap(p_, o.p_); std::swap(st_, o.st_); return *this; }
    ~DevBuf() { reset(); }
    int alloc(size_t n, cudaStream_t st) { reset(); st_ = st; return dev_alloc_t(&p_, n, st); }
    T* get() const { return p_; }
    void reset() { dev_free(p_, st_); p_ = nullptr; }
private:
    T* p_ = nullptr;
    cudaStream_t st_ = nullptr;
};

// Owners of a stream, an event and a graph executable, next to DevBuf's ownership of memory.  A Stream synchronises before it is
// destroyed, so a struct that holds one declares it after the buffers its work uses: members are destroyed in reverse order, and
// the stream drains before they are freed.
struct StreamDrain { void operator()(cudaStream_t s) const { cudaStreamSynchronize(s); cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct GraphExecDestroy { void operator()(cudaGraphExec_t g) const { cudaGraphExecDestroy(g); } };
using Stream = std::unique_ptr<CUstream_st, StreamDrain>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;
using GraphExec = std::unique_ptr<CUgraphExec_st, GraphExecDestroy>;
inline int new_stream(Stream& s) {       // non-blocking: no implicit synchronisation with the legacy default stream
    cudaStream_t h = nullptr;
    BMSP_CUDA(cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking));
    s.reset(h);
    return BMSP_OK;
}
inline int new_event(Event& e, bool timing = false) {
    cudaEvent_t h = nullptr;
    BMSP_CUDA(cudaEventCreateWithFlags(&h, timing ? cudaEventDefault : cudaEventDisableTiming));
    e.reset(h);
    return BMSP_OK;
}

// Facts about the current device, looked up once per device (thread-safe; matrix.cu).  The first lookup on a device also makes its
// default memory pool keep freed blocks, so that repeated products reuse them without cudaMallocAsync going back to the driver.
struct DeviceInfo {
    int32_t sms = 0, cc_major = 0, cc_minor = 0;
    size_t smem_per_sm = 0;
    int64_t l2_bytes = 0, hbm_bytes = 0;
};
int current_device(const DeviceInfo** out);
// Lets kern launch with smem bytes of dynamic shared memory on the current device: raises its limit to max(smem, 48 KB), and with
// max_carveout prefers the largest shared-memory carveout, when the kernel is first configured on the device and whenever smem is
// above the limit it already has there.
int kernel_smem(const void* kern, size_t smem, bool max_carveout);

// A handle under construction: bmsp_destroy frees whatever it holds unless release() handed it to the caller.
struct HandleDeleter { void operator()(bmsp_matrix_s* m) const { bmsp_destroy(m); } };
using HandlePtr = std::unique_ptr<bmsp_matrix_s, HandleDeleter>;
// A new handle used on st, with its shape and the interchange arrays: keys / bmps / offsets for nblk blocks (+2 entries) and values
// for nnz values (+16 bytes).  nnz < 0 leaves the values to the caller (a product's C: FILL finds its value count).
int new_handle(int32_t rows, int32_t cols, int64_t nblk, int64_t nnz, int32_t dtype, int32_t transposed, cudaStream_t st, HandlePtr& out);

// out[0..n] = exclusive scan of in[0..n-1] (out has n+1 entries, out[n] = total).  in may be nullptr
// when a transform kernel filled out[0..n-1] in place (in == out allowed).
int exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, cudaStream_t st);
int exclusive_scan_u64(const uint64_t* in, uint64_t* out, int64_t n, cudaStream_t st);

// derive brp/bcol/rvb/kmask from keys/bmps/offsets (matrix.cu)
int derive_compact(bmsp_matrix_s* m, cudaStream_t st);
// free m->spmv (spmv.cu) and m->bidx (spgemm.cu); bmsp_destroy calls them once m's streams are done with the memory
void spmv_release(bmsp_matrix_s* m);
void bindex_release(bmsp_matrix_s* m);
// rebuild every copy of m's values that the library derived from them (SpGEMM's packed B records and fine index; spgemm.cu), on
// st: after m's values changed.  The SpMV plan holds no values and is kept.
int refresh_value_copies(bmsp_matrix_s* m, cudaStream_t st);

// SpMV's path rule (spmv.cu; dist.cu weighs block rows by it): under 2.5 values per block, or no blocks, runs block-parallel
inline bool spmv_block_parallel(const bmsp_matrix_s* m) { return m->nblk == 0 || (double)m->nnz / (double)m->nblk < 2.5; }

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------- interchange (data in and out of a matrix)
static inline size_t dtype_bytes(int32_t dtype) { return dtype == BMSP_F16 ? 2 : 4; }

// f(__half{}) for BMSP_F16, f(float{}) for BMSP_F32: the value type of a dtype code, for a generic lambda that launches the
// instantiation of that type.  Two nested calls dispatch an (input, output) pair.
template <typename F>
inline auto with_value_type(int32_t dtype, F&& f) { return dtype == BMSP_F16 ? f(__half{}) : f(float{}); }

// An array argument of an entry point that takes host or device input (mem): BMSP_DEVICE input is used where it is; any other input
// is copied into buf on st, and p is pointed at the copy.  buf is freed on st when it goes out of scope.  An entry point that staged
// host input synchronises st before it returns: its caller may free the host array then.
template <typename T>
int stage(DevBuf<char>& buf, const T*& p, size_t bytes, int32_t mem, cudaStream_t st) {
    if (mem == BMSP_DEVICE) return BMSP_OK;
    BMSP_TRY(buf.alloc(bytes, st));
    if (bytes) BMSP_CUDA(cudaMemcpyAsync(buf.get(), p, bytes, cudaMemcpyHostToDevice, st));
    p = (const T*)buf.get();
    return BMSP_OK;
}

// a host CSR's row_ptr starts at 0 and ends at nnz (the device input is checked by the kernels that read it)
bool host_row_ptr_spans(const int32_t* row_ptr, int32_t rows, int64_t nnz);

// Host COO -> CSR: a counting sort by row, then the columns of every row in ascending order; entries with the same (row, col) stay
// in input order.  Entries whose row is outside [0, rows) are left out; the return value is how many.
template <typename V>
int64_t coo_to_csr_host(int32_t rows, int64_t nnz, const int32_t* row_idx, const int32_t* col_idx, const V* vals,
                        std::vector<int32_t>& rp, std::vector<int32_t>& ci, std::vector<V>& v) {
    auto inside = [&](int64_t i) { return row_idx[i] >= 0 && row_idx[i] < rows; };
    rp.assign((size_t)rows + 1, 0);
    int64_t outside = 0;
    for (int64_t i = 0; i < nnz; i++) {
        if (inside(i)) rp[(size_t)row_idx[i] + 1]++;
        else outside++;
    }
    for (int32_t r = 0; r < rows; r++) rp[r + 1] += rp[r];
    std::vector<int64_t> perm((size_t)rp[rows]);
    {
        std::vector<int32_t> cur(rp.begin(), rp.end() - 1);
        for (int64_t i = 0; i < nnz; i++) if (inside(i)) perm[(size_t)cur[row_idx[i]]++] = i;
    }
    for (int32_t r = 0; r < rows; r++)
        std::stable_sort(perm.begin() + rp[r], perm.begin() + rp[r + 1], [&](int64_t a, int64_t b) { return col_idx[a] < col_idx[b]; });
    ci.resize(perm.size()); v.resize(perm.size());
    for (size_t i = 0; i < perm.size(); i++) { ci[i] = col_idx[perm[i]]; v[i] = vals[perm[i]]; }
    return outside;
}

// ---------------------------------------------------------------------------- device helpers
__device__ __forceinline__ uint32_t kmask_of(uint64_t bmp) {
    uint32_t w = (uint32_t)(bmp >> 32) | (uint32_t)bmp;
    w |= w >> 16;
    w |= w >> 8;
    return w & 0xFFu;
}

__device__ __forceinline__ float val_to_f32(const __half v) { return __half2float(v); }
__device__ __forceinline__ float val_to_f32(const float v) { return v; }

// value conversion on ingest (round to nearest)
template <typename Tin, typename Tout> __device__ __forceinline__ Tout conv(Tin v);
template <> __device__ __forceinline__ __half conv<float, __half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __half conv<__half, __half>(__half v) { return v; }
template <> __device__ __forceinline__ float conv<float, float>(float v) { return v; }
template <> __device__ __forceinline__ float conv<__half, float>(__half v) { return __half2float(v); }

// 8x8 bit-matrix transpose (three masked swaps); with MSB-first cell numbering the main diagonal is
// bits 63,54,...,0, so the classic delta-swap constants apply unchanged.
__device__ __forceinline__ uint64_t transpose8x8(uint64_t x) {
    uint64_t t;
    t = (x ^ (x >> 7)) & 0x00AA00AA00AA00AAull;  x = x ^ t ^ (t << 7);
    t = (x ^ (x >> 14)) & 0x0000CCCC0000CCCCull; x = x ^ t ^ (t << 14);
    t = (x ^ (x >> 28)) & 0x00000000F0F0F0F0ull; x = x ^ t ^ (t << 28);
    return x;
}

// ---- scans, reductions and searches of the set-up kernels (count per item, scan the counts, size the output, fill it).
// The warp functions need the full warp active.  The reductions use the xor butterfly: every lane gets the result.
template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// a flag counts 1: its warp sum and warp scan are a ballot and a popcount (uint32_t)
__device__ __forceinline__ uint32_t warp_inclusive_scan(bool p) {
    return __popc(__ballot_sync(0xffffffffu, p) & (0xffffffffu >> (31 - (threadIdx.x & 31))));
}
__device__ __forceinline__ uint32_t warp_sum(bool p) { return __popc(__ballot_sync(0xffffffffu, p)); }
template <typename T>
__device__ __forceinline__ T warp_min(T v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// The CTA functions take one value per thread from every thread of the CTA; blockDim.x is a multiple of 32, at most 1024.  Both
// end with a barrier, so a kernel may call them more than once.
// Exclusive scan in thread order; *total = the sum over the CTA.  Warp scans, then warp 0 scans the warp totals.  V is T, or bool
// with T uint32_t (flags).
template <typename V, typename T>
__device__ __forceinline__ T cta_exclusive_scan(V v, T* total) {
    __shared__ T s_warp[33];              // per warp: its total, then the sum of the earlier warps; [32]: the CTA's total
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const T incl = warp_inclusive_scan(v);
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    if (w == 0) {
        const T x = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : T(0);
        const T xi = warp_inclusive_scan(x);
        s_warp[lane] = xi - x;
        if (lane == 31) s_warp[32] = xi;
    }
    __syncthreads();
    const T ex = s_warp[w] + incl - v;
    *total = s_warp[32];
    __syncthreads();
    return ex;
}
// The sum over the CTA, returned to every thread (uint32_t for flags).  Warp sums, then warp 0 sums the warp totals.  The total
// is read after the last barrier: a next call writes it only after its first barrier, which every thread reaches after reading.
template <typename V>
__device__ __forceinline__ auto cta_sum(V v) {
    using T = decltype(warp_sum(v));
    __shared__ T s_warp[33];              // per warp: its sum; [32]: the CTA's
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const T ws = warp_sum(v);
    if (lane == 0) s_warp[w] = ws;
    __syncthreads();
    if (w == 0) {
        const T s = warp_sum(lane < (int)(blockDim.x >> 5) ? s_warp[lane] : T(0));
        if (lane == 0) s_warp[32] = s;
    }
    __syncthreads();
    return s_warp[32];
}

// Searches in a[lo, hi), ascending, in global or shared memory.  lower_bound: the first i with a[i] >= v; upper_bound: the first
// i with a[i] > v (hi when there is none).  The last i with a[i] <= v is upper_bound(...) - 1.
template <typename T, typename V, typename I>
__device__ __forceinline__ I lower_bound(const T* a, I lo, I hi, V v) {
    while (lo < hi) {
        const I mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
template <typename T, typename V, typename I>
__device__ __forceinline__ I upper_bound(const T* a, I lo, I hi, V v) {
    while (lo < hi) {
        const I mid = (lo + hi) >> 1;
        if (a[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// Merge path: how many of a's items are among the first diag items of the stable merge of the ascending a[0, na) and b[0, nb),
// ties to a (a's item of an equal pair comes first).
template <typename T, typename I>
__device__ __forceinline__ I merge_path(const T* a, I na, const T* b, I nb, I diag) {
    I lo = max((I)0, diag - nb), hi = min(diag, na);
    while (lo < hi) {
        const I mid = (lo + hi) >> 1;
        if (a[mid] <= b[diag - 1 - mid]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// streaming (read-once) loads: keep them out of L1 and mark evict-first in L2 so that x stays resident
__device__ __forceinline__ uint64_t ld_stream_u64(const uint64_t* p) {
    return (uint64_t)__ldcs(reinterpret_cast<const unsigned long long*>(p));   // ld.global.cs: evict-first
}
__device__ __forceinline__ int32_t ld_stream_s32(const int32_t* p) {
    return __ldcs(p);
}

// ---- mbarrier + bulk async copy (TMA 1-D; SASS: UBLKCP / SYNCS) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy; dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

}  // namespace bmsp
