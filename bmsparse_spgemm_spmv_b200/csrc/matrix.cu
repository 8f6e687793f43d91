// matrix.cu -- handle lifetime, derived compact arrays, scans, export/compare.
// Reference surface: include/bmSpMatrix.h:20-40, src/bmSpMatrix.cu:30-43 (adopting constructor),
// :320-363 (generate_coo), :381-432 (compare).
#include "common.cuh"
#include <vector>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <unordered_map>

namespace bmsp {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    return BMSP_ERR_CUDA;
}

// ------------------------------------------------------------------------------------ per-device state
// One entry per device index, filled by the first lookup on that device.  The limits of kernel_smem are attributes of the
// function in that device's context, so they are kept per device too.
namespace {
constexpr int MAX_DEVICES = 64;
struct DeviceEntry {
    std::once_flag once;
    cudaError_t err = cudaSuccess;             // of the first lookup: an invalid device or a dead context stays so
    DeviceInfo info;
    std::mutex mu;                             // guards smem_limit
    std::unordered_map<const void*, size_t> smem_limit;   // per configured kernel: its dynamic shared-memory limit
};
DeviceEntry g_devices[MAX_DEVICES];

cudaError_t init_device(int dev, DeviceInfo& d) {
    cudaDeviceProp p;
    cudaError_t e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) return e;
    d.sms = p.multiProcessorCount; d.cc_major = p.major; d.cc_minor = p.minor;
    d.smem_per_sm = p.sharedMemPerMultiprocessor;
    d.l2_bytes = p.l2CacheSize; d.hbm_bytes = (int64_t)p.totalGlobalMem;
    cudaMemPool_t pool;
    if ((e = cudaDeviceGetDefaultMemPool(&pool, dev)) != cudaSuccess) return e;
    uint64_t thr = UINT64_MAX;
    return cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
}

int device_entry(DeviceEntry** out) {
    int dev = 0;
    BMSP_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= MAX_DEVICES) { set_error("device %d: at most %d devices are supported", dev, MAX_DEVICES); return BMSP_ERR_UNSUPPORTED; }
    DeviceEntry& e = g_devices[dev];
    std::call_once(e.once, [&] { e.err = init_device(dev, e.info); });
    BMSP_CUDA(e.err);
    *out = &e;
    return BMSP_OK;
}
}  // namespace

int current_device(const DeviceInfo** out) {
    DeviceEntry* e = nullptr;
    BMSP_TRY(device_entry(&e));
    *out = &e->info;
    return BMSP_OK;
}

int kernel_smem(const void* kern, size_t smem, bool max_carveout) {
    DeviceEntry* e = nullptr;
    BMSP_TRY(device_entry(&e));
    std::lock_guard<std::mutex> lock(e->mu);
    const auto it = e->smem_limit.find(kern);
    if (it != e->smem_limit.end() && it->second >= smem) return BMSP_OK;
    const size_t limit = std::max<size_t>(smem, 48 * 1024);
    BMSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    if (max_carveout) BMSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    e->smem_limit[kern] = limit;
    return BMSP_OK;
}

int dev_alloc(void** p, size_t bytes, cudaStream_t st) {
    const DeviceInfo* d = nullptr;
    BMSP_TRY(current_device(&d));              // sets up the device's memory pool
    *p = nullptr;
    BMSP_CUDA(cudaMallocAsync(p, bytes + BMSP_PAD_BYTES, st));
    return BMSP_OK;
}
void dev_free(void* p, cudaStream_t st) {
    if (p) cudaFreeAsync(p, st);
}

// ------------------------------------------------------------------------------------ scans
// Three-kernel scan: per-tile sums -> (recursive) scan of sums -> per-tile scan with base.
template <typename T>
__global__ void scan_tile_sums(const T* __restrict__ in, T* __restrict__ sums, int64_t n) {
    constexpr int ITEMS = 8;
    int64_t base = (int64_t)blockIdx.x * (blockDim.x * ITEMS);
    T s = 0;
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        int64_t idx = base + (int64_t)i * blockDim.x + threadIdx.x;
        if (idx < n) s += in[idx];
    }
    s = cta_sum(s);
    if (threadIdx.x == 0) sums[blockIdx.x] = s;
}

template <typename T>
__global__ void scan_tiles(const T* in, T* out, const T* __restrict__ tile_base, int64_t n,
                           int write_total) {
    constexpr int ITEMS = 8;
    // blocked arrangement: thread t owns ITEMS consecutive elements
    int64_t base = (int64_t)blockIdx.x * (blockDim.x * ITEMS) + (int64_t)threadIdx.x * ITEMS;
    T v[ITEMS];
    T s = 0;
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        int64_t idx = base + i;
        v[i] = idx < n ? in[idx] : 0;
        s += v[i];
    }
    T total;
    T run = (tile_base ? tile_base[blockIdx.x] : 0) + cta_exclusive_scan(s, &total);
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        int64_t idx = base + i;
        if (idx < n) out[idx] = run;
        run += v[i];
        if (write_total && idx == n - 1) out[n] = run;
    }
}

template <typename T>
static int exclusive_scan_impl(const T* in, T* out, int64_t n, cudaStream_t st, int write_total) {
    constexpr int THREADS = 256, TILE = THREADS * 8;
    if (n <= 0) {
        if (write_total) BMSP_CUDA(cudaMemsetAsync(out, 0, sizeof(T), st));
        return BMSP_OK;
    }
    int64_t tiles = ceil_div(n, TILE);
    if (tiles == 1) {
        scan_tiles<T><<<1, THREADS, 0, st>>>(in, out, nullptr, n, write_total);
        BMSP_KERNEL_CHECK();
        return BMSP_OK;
    }
    DevBuf<T> sums;
    BMSP_TRY(sums.alloc((size_t)tiles + 1, st));
    scan_tile_sums<T><<<(unsigned)tiles, THREADS, 0, st>>>(in, sums.get(), n);
    BMSP_KERNEL_CHECK();
    BMSP_TRY(exclusive_scan_impl<T>(sums.get(), sums.get(), tiles, st, 0));
    scan_tiles<T><<<(unsigned)tiles, THREADS, 0, st>>>(in, out, sums.get(), n, write_total);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

int exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, cudaStream_t st) {
    return exclusive_scan_impl<uint32_t>(in, out, n, st, 1);
}
int exclusive_scan_u64(const uint64_t* in, uint64_t* out, int64_t n, cudaStream_t st) {
    return exclusive_scan_impl<uint64_t>(in, out, n, st, 1);
}

// ------------------------------------------------------------------------------------ derive
__global__ void derive_blocks_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ bmps,
                                     int32_t* __restrict__ bcol, uint8_t* __restrict__ kmask, int64_t nblk) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    bcol[b] = (int32_t)(keys[b] & 0xFFFFFFFFull);
    kmask[b] = (uint8_t)kmask_of(bmps[b]);
}

// brp[br] = first block whose block row >= br (lower bound on keys); rvb[br] = its value offset.
__global__ void derive_rows_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ offsets,
                                   int32_t* __restrict__ brp, uint32_t* __restrict__ rvb, int64_t nblk, int32_t nbr,
                                   uint64_t nnz) {
    int32_t br = blockIdx.x * blockDim.x + threadIdx.x;
    if (br > nbr) return;
    const int64_t lo = lower_bound(keys, (int64_t)0, nblk, (uint64_t)br << 32);
    brp[br] = (int32_t)lo;
    rvb[br] = (uint32_t)(lo < nblk ? offsets[lo] : nnz);
}

int derive_compact(bmsp_matrix_s* m, cudaStream_t st) {
    if (m->nblk > 0x7FFFFFFFll || m->nnz > 0xFFFFFFFFll) {
        set_error("matrix too large: %lld blocks, %lld values", (long long)m->nblk, (long long)m->nnz);
        return BMSP_ERR_TOO_LARGE;
    }
    m->nbr = (int32_t)ceil_div(m->rows, 8);
    BMSP_TRY(dev_alloc_t(&m->bcol, (size_t)m->nblk + 8, st));
    BMSP_TRY(dev_alloc_t(&m->kmask, (size_t)m->nblk + 16, st));
    BMSP_TRY(dev_alloc_t(&m->brp, (size_t)m->nbr + 1 + 8, st));
    BMSP_TRY(dev_alloc_t(&m->rvb, (size_t)m->nbr + 1 + 8, st));
    if (m->nblk > 0) {
        derive_blocks_kernel<<<(unsigned)ceil_div(m->nblk, 256), 256, 0, st>>>(m->keys, m->bmps, m->bcol, m->kmask, m->nblk);
        BMSP_KERNEL_CHECK();
    }
    derive_rows_kernel<<<(unsigned)ceil_div(m->nbr + 1, 256), 256, 0, st>>>(m->keys, m->offsets, m->brp, m->rvb, m->nblk,
                                                                          m->nbr, (uint64_t)m->nnz);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}

bool host_row_ptr_spans(const int32_t* row_ptr, int32_t rows, int64_t nnz) { return row_ptr[0] == 0 && (int64_t)row_ptr[rows] == nnz; }

int new_handle(int32_t rows, int32_t cols, int64_t nblk, int64_t nnz, int32_t dtype, int32_t transposed, cudaStream_t st, HandlePtr& out) {
    out.reset(new bmsp_matrix_s());
    bmsp_matrix_s* m = out.get();
    touch(m, st);
    m->rows = rows; m->cols = cols; m->nblk = nblk; m->nnz = std::max<int64_t>(nnz, 0); m->offsets_len = nblk;
    m->dtype = dtype; m->transposed = transposed;
    BMSP_TRY(dev_alloc_t(&m->keys, (size_t)nblk + 2, st));
    BMSP_TRY(dev_alloc_t(&m->bmps, (size_t)nblk + 2, st));
    BMSP_TRY(dev_alloc_t(&m->offsets, (size_t)nblk + 2, st));
    if (nnz >= 0) BMSP_TRY(dev_alloc(&m->values, (size_t)nnz * dtype_bytes(dtype) + 16, st));
    return BMSP_OK;
}

}  // namespace bmsp

using namespace bmsp;

extern "C" {

int bmsp_abi_version(void) { return BMSP_ABI_VERSION; }
const char* bmsp_last_error(void) { return g_err.c_str(); }

int bmsp_device_info(int32_t* sm_count, int64_t* l2_bytes, int64_t* hbm_bytes, int32_t* cc_major, int32_t* cc_minor) {
    const DeviceInfo* d = nullptr;
    BMSP_TRY(current_device(&d));
    if (sm_count) *sm_count = d->sms;
    if (l2_bytes) *l2_bytes = d->l2_bytes;
    if (hbm_bytes) *hbm_bytes = d->hbm_bytes;
    if (cc_major) *cc_major = d->cc_major;
    if (cc_minor) *cc_minor = d->cc_minor;
    return BMSP_OK;
}

int bmsp_create_from_arrays(int32_t rows, int32_t cols, int64_t block_num, int64_t nnz, const uint64_t* keys,
                            const uint64_t* bmps, const uint64_t* offsets, int64_t offsets_len, const void* values,
                            int32_t dtype, int32_t mem, int32_t transposed, void* stream, bmsp_matrix_t* out) {
    if (!out || rows < 0 || cols < 0 || block_num < 0 || nnz < 0 || (dtype != BMSP_F16 && dtype != BMSP_F32) ||
        (offsets_len != block_num && offsets_len != block_num + 1) ||
        (block_num > 0 && (!keys || !bmps || !offsets)) || (nnz > 0 && !values)) {
        set_error("bmsp_create_from_arrays: invalid argument");
        return BMSP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    HandlePtr m;
    BMSP_TRY(new_handle(rows, cols, block_num, nnz, dtype, transposed, st, m));
    m->offsets_len = offsets_len;
    cudaMemcpyKind kind = mem == BMSP_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    if (block_num > 0) {
        BMSP_CUDA(cudaMemcpyAsync(m->keys, keys, sizeof(uint64_t) * block_num, kind, st));
        BMSP_CUDA(cudaMemcpyAsync(m->bmps, bmps, sizeof(uint64_t) * block_num, kind, st));
        BMSP_CUDA(cudaMemcpyAsync(m->offsets, offsets, sizeof(uint64_t) * offsets_len, kind, st));
    }
    if (nnz > 0) BMSP_CUDA(cudaMemcpyAsync(m->values, values, (size_t)nnz * dtype_bytes(dtype), kind, st));
    BMSP_TRY(derive_compact(m.get(), st));
    if (mem == BMSP_HOST) BMSP_CUDA(cudaStreamSynchronize(st));   // host buffers may be freed by the caller
    *out = m.release();
    return BMSP_OK;
}

int bmsp_destroy(bmsp_matrix_t m) {
    if (!m) return BMSP_OK;
    // frees are ordered behind the last work enqueued on the arrays (ADVICE r1: stream 0 does not order after non-blocking streams)
    if (m->multi_stream) cudaDeviceSynchronize();
    cudaStream_t st = m->last_stream;
    spmv_release(m); bindex_release(m);
    dev_free(m->keys, st); dev_free(m->bmps, st); dev_free(m->offsets, st); dev_free(m->values, st);
    dev_free(m->brp, st); dev_free(m->bcol, st); dev_free(m->rvb, st); dev_free(m->kmask, st);
    delete m;
    return BMSP_OK;
}

int bmsp_get(bmsp_matrix_t m, bmsp_view* v) {
    if (!m || !v) { set_error("bmsp_get: null argument"); return BMSP_ERR_INVALID; }
    v->num_rows = m->rows; v->num_cols = m->cols; v->nnz = m->nnz; v->block_num = m->nblk;
    v->keys = m->keys; v->bmps = m->bmps; v->offsets = m->offsets; v->values = m->values;
    v->offsets_len = m->offsets_len; v->dtype = m->dtype; v->transposed = m->transposed;
    v->num_block_rows = m->nbr; v->block_row_ptr = m->brp; v->block_col = m->bcol; v->block_row_val = m->rvb;
    return BMSP_OK;
}

int bmsp_download(bmsp_matrix_t m, uint64_t* keys, uint64_t* bmps, uint64_t* offsets, void* values) {
    if (!m) { set_error("bmsp_download: null matrix"); return BMSP_ERR_INVALID; }
    BMSP_CUDA(cudaDeviceSynchronize());
    if (keys && m->nblk) BMSP_CUDA(cudaMemcpy(keys, m->keys, sizeof(uint64_t) * m->nblk, cudaMemcpyDeviceToHost));
    if (bmps && m->nblk) BMSP_CUDA(cudaMemcpy(bmps, m->bmps, sizeof(uint64_t) * m->nblk, cudaMemcpyDeviceToHost));
    if (offsets && m->offsets_len) BMSP_CUDA(cudaMemcpy(offsets, m->offsets, sizeof(uint64_t) * m->offsets_len, cudaMemcpyDeviceToHost));
    if (values && m->nnz) BMSP_CUDA(cudaMemcpy(values, m->values, (size_t)m->nnz * dtype_bytes(m->dtype), cudaMemcpyDeviceToHost));
    return BMSP_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------ to_coo / compare
// One thread per block walks its bits MSB-first (bmSpMatrix.cu:334-353) and writes (row, col, fp32 value)
// at offsets[b] + rank.
template <typename T>
__global__ void to_coo_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ bmps,
                              const uint64_t* __restrict__ offsets, const T* __restrict__ values, int transposed,
                              int32_t* __restrict__ rows, int32_t* __restrict__ cols, float* __restrict__ vals, int64_t nblk) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    uint64_t bmp = bmps[b], key = keys[b];
    int32_t br = (int32_t)(key >> 32), bc = (int32_t)(key & 0xFFFFFFFFull);
    uint64_t w = offsets[b];
    while (bmp) {
        int p = __clzll((long long)bmp);
        bmp &= ~(0x8000000000000000ull >> p);
        int hi = p >> 3, lo = p & 7;
        rows[w] = br * 8 + (transposed ? lo : hi);
        cols[w] = bc * 8 + (transposed ? hi : lo);
        vals[w] = val_to_f32(values[w]);
        w++;
    }
}

extern "C" int bmsp_to_coo(bmsp_matrix_t m, int32_t* rows, int32_t* cols, float* vals) {
    if (!m || !rows || !cols || !vals) { set_error("bmsp_to_coo: null argument"); return BMSP_ERR_INVALID; }
    if (m->nnz == 0) return BMSP_OK;
    if (m->multi_stream) BMSP_CUDA(cudaDeviceSynchronize());
    cudaStream_t st = m->last_stream;          // ordered behind whatever produced the arrays
    DevBuf<int32_t> dr, dc; DevBuf<float> dv;
    BMSP_TRY(dr.alloc((size_t)m->nnz, st));
    BMSP_TRY(dc.alloc((size_t)m->nnz, st));
    BMSP_TRY(dv.alloc((size_t)m->nnz, st));
    const unsigned grid = (unsigned)ceil_div(m->nblk, 128);
    BMSP_TRY(with_value_type(m->dtype, [&](auto t) -> int {
        using T = decltype(t);
        to_coo_kernel<T><<<grid, 128, 0, st>>>(m->keys, m->bmps, m->offsets, (const T*)m->values, m->transposed, dr.get(), dc.get(), dv.get(), m->nblk);
        BMSP_KERNEL_CHECK();
        return BMSP_OK;
    }));
    BMSP_CUDA(cudaMemcpyAsync(rows, dr.get(), sizeof(int32_t) * m->nnz, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(cols, dc.get(), sizeof(int32_t) * m->nnz, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaMemcpyAsync(vals, dv.get(), sizeof(float) * m->nnz, cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    return BMSP_OK;
}

// ------------------------------------------------------------------------------------ bmSparse <-> CSR on the device
// The blocks of a block row are already in ascending block column and a bitmap is row-major inside a block, so CSR order is an
// 8-way merge in reverse: entry (r, c) of block b goes to row_ptr[r] + (cells of row r in the earlier blocks of the block row) +
// (cells of row r left of c in this block).  Pass 1 counts the cells per matrix row (one thread per block), a scan gives row_ptr,
// pass 2 runs one warp per block row: lanes <-> blocks, 32 at a time; the eight per-row counts of a block travel as two 64-bit
// words of four 16-bit fields through one warp scan each.  The same walk run backwards scatters CSR values into the compact order
// (bmsp_set_values_csr).
__global__ void csr_count_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ bmps, int64_t nblk, int32_t rows,
                                 uint32_t* __restrict__ row_cnt) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk) return;
    const uint64_t bmp = bmps[b];
    const int64_t r0 = (int64_t)(keys[b] >> 32) * 8;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint32_t c = __popc((uint32_t)(bmp >> (56 - 8 * r)) & 0xFFu);
        if (c && r0 + r < rows) atomicAdd(row_cnt + r0 + r, c);
    }
}

// The cells of block row br in CSR order, one warp: cell(slot, r, col, k) for every cell -- slot its CSR position, r its row inside
// the block row, k its index in the compact values.  base[r]: the first slot of row r of the block row (warp-uniform); on return it
// is advanced past the row's cells.  TRANSPOSED: a transposed-operand matrix holds cell (r, c) at bit 63-(c*8+r); the CSR slot still
// comes from the row-major counts, the compact index is the cell's rank in the stored (column-major) bitmap.
template <bool TRANSPOSED, typename F>
__device__ __forceinline__ void csr_walk_block_row(const int32_t* __restrict__ brp, const int32_t* __restrict__ bcol, const uint64_t* __restrict__ bmps,
                                                   const uint64_t* __restrict__ offsets, int br, uint32_t (&base)[8], F&& cell) {
    const int lane = threadIdx.x & 31;
    for (int b0 = brp[br]; b0 < brp[br + 1]; b0 += 32) {
        const int b = b0 + lane;
        const bool valid = b < brp[br + 1];
        const uint64_t stored = valid ? bmps[b] : 0ull;
        const uint64_t bmp = TRANSPOSED ? transpose8x8(stored) : stored;     // row-major
        uint64_t lo = 0, hi = 0;          // per-row counts, 16-bit fields: rows 0-3 in lo, 4-7 in hi
#pragma unroll
        for (int r = 0; r < 4; r++) {
            lo |= (uint64_t)__popc((uint32_t)(bmp >> (56 - 8 * r)) & 0xFFu) << (16 * r);
            hi |= (uint64_t)__popc((uint32_t)(bmp >> (24 - 8 * r)) & 0xFFu) << (16 * r);
        }
        const uint64_t ilo = warp_inclusive_scan(lo), ihi = warp_inclusive_scan(hi);
        const uint64_t elo = ilo - lo, ehi = ihi - hi;             // exclusive: cells of each row in the earlier blocks of this chunk
        if (valid) {
            uint64_t k = offsets[b];
            const int32_t c0 = bcol[b] * 8;
            uint64_t rem = bmp;
            uint32_t in_row[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            while (rem) {
                const int p = __clzll((long long)rem);
                rem &= ~(0x8000000000000000ull >> p);
                const int r = p >> 3;
                const uint32_t ex = (uint32_t)(((r < 4 ? elo : ehi) >> (16 * (r & 3))) & 0xFFFFu);
                uint32_t slot = 0;
#pragma unroll
                for (int q = 0; q < 8; q++) if (q == r) slot = base[q] + ex + in_row[q]++;
                if (TRANSPOSED) {
                    const int t = (p & 7) * 8 + r;                      // the cell's bit in the stored bitmap
                    cell(slot, r, c0 + (p & 7), k + (t ? __popcll(stored >> (64 - t)) : 0));
                } else {
                    cell(slot, r, c0 + (p & 7), k++);
                }
            }
        }
        const uint64_t tlo = __shfl_sync(0xffffffffu, ilo, 31), thi = __shfl_sync(0xffffffffu, ihi, 31);
#pragma unroll
        for (int r = 0; r < 4; r++) { base[r] += (uint32_t)((tlo >> (16 * r)) & 0xFFFFu); base[4 + r] += (uint32_t)((thi >> (16 * r)) & 0xFFFFu); }
    }
}

template <typename T>
__global__ void __launch_bounds__(256) csr_fill_kernel(const int32_t* __restrict__ brp, const int32_t* __restrict__ bcol, const uint64_t* __restrict__ bmps,
                                                       const uint64_t* __restrict__ offsets, const T* __restrict__ values, int32_t nbr, int32_t rows,
                                                       const uint32_t* __restrict__ row_ptr, int32_t* __restrict__ col_idx, float* __restrict__ vals) {
    const int br = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (br >= nbr) return;
    uint32_t base[8];                     // next free slot of each of the block row's eight matrix rows (warp-uniform)
#pragma unroll
    for (int r = 0; r < 8; r++) base[r] = (int64_t)br * 8 + r < rows ? row_ptr[(int64_t)br * 8 + r] : 0u;
    csr_walk_block_row<false>(brp, bcol, bmps, offsets, br, base, [&](uint32_t slot, int, int32_t col, uint64_t k) {
        col_idx[slot] = col;
        vals[slot] = val_to_f32(values[k]);
    });
}

// CSR values -> the compact values of a matrix with the same pattern.  CHECK: writes nothing and raises *flag on any difference of
// pattern -- a row_ptr entry outside [0, nnz] or decreasing, a row whose length is not its cell count, an entry whose column is not
// its cell's.  col_idx is read inside the row's own [row_ptr[r], row_ptr[r+1]) only, so a malformed CSR is never read out of
// bounds.  !CHECK: the scatter, launched once the check has passed.
template <bool TRANSPOSED, bool CHECK, typename Tin, typename Tout>
__global__ void __launch_bounds__(256) csr_scatter_kernel(const int32_t* __restrict__ brp, const int32_t* __restrict__ bcol, const uint64_t* __restrict__ bmps,
                                                          const uint64_t* __restrict__ offsets, int32_t nbr, int32_t rows, int64_t nnz,
                                                          const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col_idx,
                                                          const Tin* __restrict__ vals, Tout* __restrict__ out, int32_t* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int br = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (br >= nbr) return;
    uint32_t base[8], end[8];
    bool bad = false;                     // warp-uniform until the walk
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int64_t R = (int64_t)br * 8 + r;
        int32_t lo = 0, hi = 0;
        if (R < rows) { lo = row_ptr[R]; hi = row_ptr[R + 1]; }
        bad |= lo < 0 || hi < lo || (int64_t)hi > nnz;
        base[r] = (uint32_t)lo; end[r] = (uint32_t)hi;
    }
    if (CHECK && bad) { if (lane == 0) atomicOr(flag, 1); return; }
    csr_walk_block_row<TRANSPOSED>(brp, bcol, bmps, offsets, br, base, [&](uint32_t slot, int r, int32_t col, uint64_t k) {
        if (CHECK) {
            uint32_t e = 0;
#pragma unroll
            for (int q = 0; q < 8; q++) if (q == r) e = end[q];
            if (slot >= e || col_idx[slot] != col) bad = true;
        } else {
            out[k] = conv<Tin, Tout>(vals[slot]);
        }
    });
    if (CHECK) {
#pragma unroll
        for (int r = 0; r < 8; r++) bad |= base[r] != end[r];          // base: the row's start + its cells
        if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flag, 1);
    }
}

// device CSR of m into caller-provided device arrays (row_ptr: rows + 1)
static int to_csr_device(bmsp_matrix_s* m, int32_t* d_rp, int32_t* d_ci, float* d_v, cudaStream_t st) {
    if (m->transposed) { set_error("bmsp_to_csr: matrix is in transposed-operand form (bmsp_block_transpose first)"); return BMSP_ERR_UNSUPPORTED; }
    BMSP_CUDA(cudaMemsetAsync(d_rp, 0, sizeof(int32_t) * ((size_t)m->rows + 1), st));
    if (m->nblk == 0) return BMSP_OK;
    csr_count_kernel<<<(unsigned)ceil_div(m->nblk, 256), 256, 0, st>>>(m->keys, m->bmps, m->nblk, m->rows, (uint32_t*)d_rp);
    BMSP_KERNEL_CHECK();
    BMSP_TRY(exclusive_scan_u32((const uint32_t*)d_rp, (uint32_t*)d_rp, m->rows, st));
    const unsigned grid = (unsigned)ceil_div(m->nbr, 8);
    return with_value_type(m->dtype, [&](auto t) -> int {
        using T = decltype(t);
        csr_fill_kernel<T><<<grid, 256, 0, st>>>(m->brp, m->bcol, m->bmps, m->offsets, (const T*)m->values, m->nbr, m->rows, (const uint32_t*)d_rp, d_ci, d_v);
        BMSP_KERNEL_CHECK();
        return BMSP_OK;
    });
}

extern "C" int bmsp_to_csr(bmsp_matrix_t m, int32_t* row_ptr, int32_t* col_idx, float* vals, int32_t mem, void* stream) {
    if (!m || !row_ptr || (m->nnz > 0 && (!col_idx || !vals))) { set_error("bmsp_to_csr: null argument"); return BMSP_ERR_INVALID; }
    if (m->nnz > 0x7FFFFFFFll) { set_error("bmsp_to_csr: %lld values exceed int32 row pointers", (long long)m->nnz); return BMSP_ERR_TOO_LARGE; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(m, st);
    if (mem == BMSP_DEVICE) return to_csr_device(m, row_ptr, col_idx, vals, st);
    DevBuf<int32_t> d_rp, d_ci; DevBuf<float> d_v;
    BMSP_TRY(d_rp.alloc((size_t)m->rows + 2, st));
    BMSP_TRY(d_ci.alloc((size_t)m->nnz + 1, st));
    BMSP_TRY(d_v.alloc((size_t)m->nnz + 1, st));
    BMSP_TRY(to_csr_device(m, d_rp.get(), d_ci.get(), d_v.get(), st));
    BMSP_CUDA(cudaMemcpyAsync(row_ptr, d_rp.get(), sizeof(int32_t) * ((size_t)m->rows + 1), cudaMemcpyDeviceToHost, st));
    if (m->nnz) {
        BMSP_CUDA(cudaMemcpyAsync(col_idx, d_ci.get(), sizeof(int32_t) * (size_t)m->nnz, cudaMemcpyDeviceToHost, st));
        BMSP_CUDA(cudaMemcpyAsync(vals, d_v.get(), sizeof(float) * (size_t)m->nnz, cudaMemcpyDeviceToHost, st));
    }
    BMSP_CUDA(cudaStreamSynchronize(st));
    return BMSP_OK;
}

// ------------------------------------------------------------------------------------ new values, same structure
template <typename Tin, typename Tout>
__global__ void convert_values_kernel(const Tin* __restrict__ in, Tout* __restrict__ out, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = conv<Tin, Tout>(in[i]);
}

// device values in m's compact order -> m->values, converted to m's dtype
static int values_from_device(bmsp_matrix_s* m, const void* v, int32_t dtype, cudaStream_t st) {
    const unsigned grid = (unsigned)ceil_div(m->nnz, 256);
    return with_value_type(dtype, [&](auto in) { return with_value_type(m->dtype, [&](auto out) -> int {
        using Tin = decltype(in); using Tout = decltype(out);
        if constexpr (std::is_same<Tin, Tout>::value) {
            BMSP_CUDA(cudaMemcpyAsync(m->values, v, (size_t)m->nnz * sizeof(Tin), cudaMemcpyDeviceToDevice, st));
        } else {
            convert_values_kernel<Tin, Tout><<<grid, 256, 0, st>>>((const Tin*)v, (Tout*)m->values, m->nnz);
            BMSP_KERNEL_CHECK();
        }
        return BMSP_OK;
    }); });
}

template <bool TRANSPOSED, bool CHECK, typename Tin, typename Tout>
static int launch_scatter(bmsp_matrix_s* m, const int32_t* rp, const int32_t* ci, const void* vals, int32_t* flag, cudaStream_t st) {
    csr_scatter_kernel<TRANSPOSED, CHECK, Tin, Tout><<<(unsigned)ceil_div(m->nbr, 8), 256, 0, st>>>(m->brp, m->bcol, m->bmps, m->offsets, m->nbr, m->rows,
                                                                                                  m->nnz, rp, ci, (const Tin*)vals, (Tout*)m->values, flag);
    BMSP_KERNEL_CHECK();
    return BMSP_OK;
}
template <bool TRANSPOSED>
static int scatter_values(bmsp_matrix_s* m, const int32_t* rp, const void* vals, int32_t vals_dtype, cudaStream_t st) {
    return with_value_type(vals_dtype, [&](auto in) { return with_value_type(m->dtype, [&](auto out) {
        return launch_scatter<TRANSPOSED, false, decltype(in), decltype(out)>(m, rp, nullptr, vals, nullptr, st);
    }); });
}

// device CSR with m's pattern -> m->values: the check pass, one read-back of its flag, then the scatter
static int set_values_csr_device(bmsp_matrix_s* m, const int32_t* rp, const int32_t* ci, const void* vals, int32_t vals_dtype, cudaStream_t st) {
    if (m->nbr == 0) return BMSP_OK;
    DevBuf<int32_t> flag;
    BMSP_TRY(flag.alloc(1, st));
    BMSP_CUDA(cudaMemsetAsync(flag.get(), 0, sizeof(int32_t), st));
    if (m->transposed) BMSP_TRY((launch_scatter<true, true, __half, __half>(m, rp, ci, nullptr, flag.get(), st)));
    else BMSP_TRY((launch_scatter<false, true, __half, __half>(m, rp, ci, nullptr, flag.get(), st)));
    int32_t h = 0;
    BMSP_CUDA(cudaMemcpyAsync(&h, flag.get(), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    if (h) { set_error("bmsp_set_values_csr: the CSR's pattern differs from the matrix's"); return BMSP_ERR_INVALID; }
    return m->transposed ? scatter_values<true>(m, rp, vals, vals_dtype, st) : scatter_values<false>(m, rp, vals, vals_dtype, st);
}

extern "C" int bmsp_set_values(bmsp_matrix_t m, const void* values, int32_t dtype, int32_t mem, void* stream) {
    if (!m || (values && dtype != BMSP_F16 && dtype != BMSP_F32)) { set_error("bmsp_set_values: invalid argument"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(m, st);
    if (values && m->nnz > 0) {
        const size_t bytes = (size_t)m->nnz * dtype_bytes(dtype);
        DevBuf<char> d;
        if (mem != BMSP_DEVICE && dtype == m->dtype) {
            BMSP_CUDA(cudaMemcpyAsync(m->values, values, bytes, cudaMemcpyHostToDevice, st));      // m's type already: no staging
        } else {
            BMSP_TRY(stage(d, values, bytes, mem, st));
            BMSP_TRY(values_from_device(m, values, dtype, st));
        }
    }
    BMSP_TRY(refresh_value_copies(m, st));
    if (values && mem == BMSP_HOST) BMSP_CUDA(cudaStreamSynchronize(st));      // host buffers may be freed by the caller
    return BMSP_OK;
}

extern "C" int bmsp_set_values_csr(bmsp_matrix_t m, const int32_t* row_ptr, const int32_t* col_idx, const void* vals, int32_t vals_dtype,
                                   int32_t mem, void* stream) {
    if (!m || !row_ptr || (m->nnz > 0 && (!col_idx || !vals)) || (vals_dtype != BMSP_F16 && vals_dtype != BMSP_F32)) {
        set_error("bmsp_set_values_csr: invalid argument");
        return BMSP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    touch(m, st);
    if (mem != BMSP_DEVICE && !host_row_ptr_spans(row_ptr, m->rows, m->nnz)) {
        set_error("bmsp_set_values_csr: row_ptr spans %lld entries, the matrix has %lld values", (long long)row_ptr[m->rows] - row_ptr[0], (long long)m->nnz);
        return BMSP_ERR_INVALID;
    }
    DevBuf<char> d_rp, d_ci, d_v;
    BMSP_TRY(stage(d_rp, row_ptr, sizeof(int32_t) * ((size_t)m->rows + 1), mem, st));
    BMSP_TRY(stage(d_ci, col_idx, sizeof(int32_t) * (size_t)m->nnz, mem, st));
    BMSP_TRY(stage(d_v, vals, (size_t)m->nnz * dtype_bytes(vals_dtype), mem, st));
    BMSP_TRY(set_values_csr_device(m, row_ptr, col_idx, vals, vals_dtype, st));
    BMSP_TRY(refresh_value_copies(m, st));
    if (mem != BMSP_DEVICE) BMSP_CUDA(cudaStreamSynchronize(st));      // host buffers may be freed by the caller
    return BMSP_OK;
}

// ------------------------------------------------------------------------------------ compare on the device
// Both sides as CSR (columns ascending in every row): one thread per matrix row merges the two column lists -- no sort.  Counts
// and error sums are reduced per CTA, then with one atomic per CTA (doubles: the mean is order-dependent only in the last bits).
__global__ void __launch_bounds__(256) compare_rows_kernel(int32_t rows, const int32_t* __restrict__ a_rp, const int32_t* __restrict__ a_ci,
                                                           const float* __restrict__ a_v, const int32_t* __restrict__ b_rp,
                                                           const int32_t* __restrict__ b_ci, const float* __restrict__ b_v,
                                                           unsigned long long* __restrict__ counts, double* __restrict__ sums) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long only_a = 0, only_b = 0, common = 0;
    double sum = 0.0, mx = 0.0;
    if (r < rows) {
        int i = a_rp[r], j = b_rp[r];
        const int ie = a_rp[r + 1], je = b_rp[r + 1];
        while (i < ie || j < je) {
            const int ca = i < ie ? a_ci[i] : 0x7FFFFFFF, cb = j < je ? b_ci[j] : 0x7FFFFFFF;
            if (ca < cb) { only_a++; i++; }
            else if (cb < ca) { only_b++; j++; }
            else {
                const double e = (double)b_v[j], g = (double)a_v[i];
                const double rel = fabs(e - g) / fmax(fabs(e), 1e-8);       // the reference's metric, bmSpMatrix.cu:418
                sum += rel; mx = fmax(mx, rel); common++;
                i++; j++;
            }
        }
    }
    __shared__ unsigned long long s_c[3];
    __shared__ double s_sum;
    __shared__ unsigned long long s_mx;
    if (threadIdx.x == 0) { s_c[0] = s_c[1] = s_c[2] = 0; s_sum = 0.0; s_mx = 0ull; }
    __syncthreads();
    only_a = warp_sum(only_a); only_b = warp_sum(only_b); common = warp_sum(common); sum = warp_sum(sum); mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_c[0], only_a); atomicAdd(&s_c[1], only_b); atomicAdd(&s_c[2], common); atomicAdd(&s_sum, sum);
        atomicMax(&s_mx, (unsigned long long)__double_as_longlong(mx));       // non-negative doubles order like their bit patterns
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_c[0]) atomicAdd(counts + 0, s_c[0]);
        if (s_c[1]) atomicAdd(counts + 1, s_c[1]);
        if (s_c[2]) atomicAdd(counts + 2, s_c[2]);
        if (s_sum != 0.0) atomicAdd(sums, s_sum);
        if (s_mx) atomicMax(counts + 3, s_mx);
    }
}

extern "C" int bmsp_compare_csr(bmsp_matrix_t m, const int32_t* row_ptr, const int32_t* col_idx, const float* vals, int32_t mem, void* stream,
                                int64_t* only_in_m, int64_t* only_in_csr, double* mean_rel_err, double* max_rel_err) {
    if (!m || !row_ptr) { set_error("bmsp_compare_csr: null argument"); return BMSP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    touch(m, st);
    DevBuf<int32_t> a_rp, a_ci; DevBuf<float> a_v; DevBuf<unsigned long long> acc; DevBuf<char> b_rp, b_ci, b_v;
    BMSP_TRY(a_rp.alloc((size_t)m->rows + 2, st));
    BMSP_TRY(a_ci.alloc((size_t)m->nnz + 1, st));
    BMSP_TRY(a_v.alloc((size_t)m->nnz + 1, st));
    BMSP_TRY(acc.alloc(8, st));
    BMSP_CUDA(cudaMemsetAsync(acc.get(), 0, 8 * sizeof(unsigned long long), st));
    BMSP_TRY(to_csr_device(m, a_rp.get(), a_ci.get(), a_v.get(), st));
    const int64_t n = mem == BMSP_DEVICE ? 0 : row_ptr[m->rows];     // the host CSR's entry count
    BMSP_TRY(stage(b_rp, row_ptr, sizeof(int32_t) * ((size_t)m->rows + 1), mem, st));
    BMSP_TRY(stage(b_ci, col_idx, sizeof(int32_t) * (size_t)n, mem, st));
    BMSP_TRY(stage(b_v, vals, sizeof(float) * (size_t)n, mem, st));
    if (m->rows > 0) {
        compare_rows_kernel<<<(unsigned)ceil_div(m->rows, 256), 256, 0, st>>>(m->rows, a_rp.get(), a_ci.get(), a_v.get(), row_ptr, col_idx, vals, acc.get(),
                                                                              reinterpret_cast<double*>(acc.get() + 4));
        BMSP_KERNEL_CHECK();
    }
    unsigned long long h[8];
    BMSP_CUDA(cudaMemcpyAsync(h, acc.get(), sizeof(h), cudaMemcpyDeviceToHost, st));
    BMSP_CUDA(cudaStreamSynchronize(st));
    double sum, mx;
    memcpy(&sum, &h[4], 8); memcpy(&mx, &h[3], 8);
    if (only_in_m) *only_in_m = (int64_t)h[0];
    if (only_in_csr) *only_in_csr = (int64_t)h[1];
    if (mean_rel_err) *mean_rel_err = h[2] ? sum / (double)h[2] : 0.0;
    if (max_rel_err) *max_rel_err = mx;
    return BMSP_OK;
}

extern "C" int bmsp_compare(bmsp_matrix_t m, int64_t nnz, const int32_t* rows, const int32_t* cols, const float* vals,
                            int64_t* only_in_m, int64_t* only_in_coo, double* mean_rel_err, double* max_rel_err) {
    if (!m || (nnz > 0 && (!rows || !cols || !vals))) { set_error("bmsp_compare: null argument"); return BMSP_ERR_INVALID; }
    // the COO (any order) becomes CSR on the host and the comparison itself runs on the device (bmsp_compare_csr).  Entries whose row
    // is outside the matrix count as "only in the COO".  Of entries with the same (row, col), the first in input order is the one
    // compared; the others count as "only in the COO" too.
    std::vector<int32_t> rp, ci;
    std::vector<float> v;
    const int64_t outside = coo_to_csr_host(m->rows, nnz, rows, cols, vals, rp, ci, v);
    int64_t ob = 0;
    BMSP_TRY(bmsp_compare_csr(m, rp.data(), ci.data(), v.data(), BMSP_HOST, m->last_stream, only_in_m, &ob, mean_rel_err, max_rel_err));
    if (only_in_coo) *only_in_coo = ob + outside;
    return BMSP_OK;
}
