/*
 * bmsparse_b200.h -- C ABI of the B200-native bmSparse SpMV / SpGEMM hot path.
 *
 * Drop-in boundary for GonzaBerger/bmSparse-SPGEMM-SPMV.  The reference has no C ABI: its
 * surface is the C++ class bmSpMatrix<T> (include/bmSpMatrix.h:20-40) with public device
 * vectors keys/bmps/offsets/values, two operator templates defined in the driver sources
 * (bmSparse_SpMV src/bmSparse_SPMV.cu:191-230, bmSparse_mult src/bmSparse_SPGEMM.cu:827-1223)
 * and the declared-only ingest entry points mmread_bmSparse (include/reader.h:14-15) and
 * CSRMatrix (include/CSRMatrix.h:13-21).  Every function below names the reference interface
 * it replaces.  include/bmSpMatrix.h, include/reader.h and include/CSRMatrix.h in this repo are
 * header-only C++ shims that re-create those class/function names on top of this ABI.
 *
 * Conventions
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = default).
 *   - every call returns a bmsp_status (0 = OK); no exit(), no prints.  bmsp_last_error() gives
 *     the message of the last failure on the calling thread.
 *   - matrices are opaque device-resident handles; bmsp_get() exposes raw device pointers whose
 *     contents are bit-identical to the reference's four vectors.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     BMSP_ERR_CUDA.
 */
#ifndef BMSPARSE_B200_H_
#define BMSPARSE_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMSP_ABI_VERSION 2

typedef enum {
    BMSP_OK = 0,
    BMSP_ERR_INVALID = 1,     /* bad argument / inconsistent sizes                               */
    BMSP_ERR_CUDA = 2,        /* CUDA runtime error or no device                                 */
    BMSP_ERR_UNSORTED = 3,    /* CSR column indices not strictly ascending inside a row          */
    BMSP_ERR_DUPLICATE = 4,   /* duplicate (row,col): the reference corrupts offsets, we reject  */
    BMSP_ERR_IO = 5,          /* MatrixMarket file unreadable / malformed                        */
    BMSP_ERR_TOO_LARGE = 6,   /* exceeds 2^31-1 blocks or 2^32-1 values                          */
    BMSP_ERR_UNSUPPORTED = 7, /* dtype / orientation combination not implemented                 */
    BMSP_ERR_RANGE = 8        /* row or column index outside the matrix                          */
} bmsp_status;

typedef enum { BMSP_F16 = 0, BMSP_F32 = 1 } bmsp_dtype;   /* bmSpMatrix<half>, bmSpMatrix<float> */
typedef enum { BMSP_HOST = 0, BMSP_DEVICE = 1 } bmsp_mem;

typedef struct bmsp_matrix_s* bmsp_matrix_t;

/* Raw view of a matrix (device pointers).  First eight fields mirror include/bmSpMatrix.h:28-32. */
typedef struct {
    int32_t num_rows, num_cols;
    int64_t nnz;                 /* values.size()                                                  */
    int64_t block_num;           /* keys.size()                                                    */
    const uint64_t* keys;        /* [block_num]  (brow << 32) | bcol, ascending                    */
    const uint64_t* bmps;        /* [block_num]  MSB-first 8x8 occupancy                            */
    const uint64_t* offsets;     /* [offsets_len] exclusive scan of popcount(bmps)                  */
    const void* values;          /* [nnz] fp16 or fp32, compacted in bitmap order                  */
    int64_t offsets_len;         /* block_num (ingested, bmSpMatrix.cu:190-194) or +1 (product, SPGEMM.cu:1087) */
    int32_t dtype;               /* bmsp_dtype of `values`                                          */
    int32_t transposed;          /* 1: transposed-operand form (bit = 63-(col%8*8+row%8))          */
    /* derived once at build time (the reference re-derives them on every call) */
    int32_t num_block_rows;      /* ceil(num_rows / 8)                                              */
    const int32_t* block_row_ptr;   /* [num_block_rows+1]                                           */
    const int32_t* block_col;       /* [block_num]                                                  */
    const uint32_t* block_row_val;  /* [num_block_rows+1] index of the block row's first value      */
} bmsp_view;

typedef struct {          /* per-phase device times of the last bmsp_spgemm (CUDA events), ms      */
    float symbolic_ms;    /* T_1..T_6,T_9 of SPGEMM.cu:835-1107                                     */
    float numeric_ms;     /* T_7 of SPGEMM.cu:1125-1158                                             */
    float total_ms;
    int64_t candidate_pairs, surviving_pairs, c_blocks, c_nnz;
    int32_t numeric_path; /* 0 scalar, 1 mma.sync                                                   */
    float count_ms;       /* symbolic, first pass: block-row spans, candidate pairs, filter, C blocks per row (T_1..T_4) */
    float fill_ms;        /* symbolic, second pass: pair list, keys in order, bitmaps, offsets (T_5, T_6, T_9)           */
} bmsp_spgemm_info;

typedef struct {
    int32_t mode;         /* accepted and ignored: `mode` of bmSparse_mult (SPGEMM.cu:828)         */
    int32_t tc_version;   /* accepted and ignored: multiplyV11..V15 selector (SPGEMM.cu:1132-1154)  */
    int32_t verbose;      /* 1: fill bmsp_spgemm_info with per-phase times (costs event syncs)      */
    int32_t numeric_path; /* -1 auto, 0 force scalar, 1 force mma.sync                              */
    int32_t brow_begin, brow_end;  /* A block-row range to multiply: multi-GPU shard / chunked product */
    int32_t brow_range_set;        /* 1: [brow_begin, brow_end) is taken literally (an empty range multiplies nothing);
                                      0: legacy rule, [0,0) = all block rows                                     */
} bmsp_spgemm_opts;

/* ---- library ------------------------------------------------------------------------------- */
int bmsp_abi_version(void);
const char* bmsp_last_error(void);
/* sm count, L2 bytes, total HBM bytes, compute capability of the current device */
int bmsp_device_info(int32_t* sm_count, int64_t* l2_bytes, int64_t* hbm_bytes, int32_t* cc_major, int32_t* cc_minor);

/* ---- construction -------------------------------------------------------------------------- */
/* CSR -> bmSparse.  Replaces CSRMatrix::CSRMatrix(cusp::csr_matrix*) (CSRMatrix.h:16) feeding the
 * COO->bmSparse conversion of bmSpMatrix.cu:163-216.  row_ptr int32[rows+1], col_idx int32[nnz]
 * strictly ascending per row, vals fp32 or fp16 ([nnz]).  mem says where the three arrays live. */
int bmsp_create_from_csr(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_ptr,
                         const int32_t* col_idx, const void* vals, int32_t vals_dtype, int32_t mem,
                         int32_t transposed, int32_t out_dtype, void* stream, bmsp_matrix_t* out);

/* Host COO (0-based, any order, no duplicates) -> bmSparse.  Replaces the body of
 * bmSpMatrix::bmSpMatrix(path, transposed) after parsing (bmSpMatrix.cu:161-216). */
int bmsp_create_from_coo(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_idx,
                         const int32_t* col_idx, const double* vals, int32_t transposed,
                         int32_t out_dtype, void* stream, bmsp_matrix_t* out);

/* MatrixMarket coordinate file -> bmSparse.  Replaces bmSpMatrix::bmSpMatrix(std::string, bool)
 * (bmSpMatrix.cu:111-219) and mmread_bmSparse (reader.cu:49-110).  `symmetric` banners are
 * mirrored (bmSpMatrix.cu:113-149), `pattern` files get value 1. */
int bmsp_create_from_mtx(const char* path, int32_t transposed, int32_t out_dtype, void* stream,
                         bmsp_matrix_t* out);

/* The same two with a flags word: BMSP_MERGE_DUPLICATES sums repeated (row, col) entries instead of rejecting them
 * (BMSP_ERR_DUPLICATE).  MatrixMarket banners: real / integer / pattern, general / symmetric / skew-symmetric (mirror negated);
 * complex, hermitian and array storage return BMSP_ERR_UNSUPPORTED (cusp/io/detail/matrix_market.inl:155-330 is the spec). */
#define BMSP_MERGE_DUPLICATES 1
int bmsp_create_from_coo_ex(int32_t rows, int32_t cols, int64_t nnz, const int32_t* row_idx,
                            const int32_t* col_idx, const double* vals, int32_t transposed,
                            int32_t out_dtype, int32_t flags, void* stream, bmsp_matrix_t* out);
int bmsp_create_from_mtx_ex(const char* path, int32_t transposed, int32_t out_dtype, int32_t flags, void* stream,
                            bmsp_matrix_t* out);

/* Adopt existing bmSparse arrays (copied).  Replaces the swap-in constructor bmSpMatrix.cu:30-43.
 * offsets_len is block_num or block_num+1. */
int bmsp_create_from_arrays(int32_t rows, int32_t cols, int64_t block_num, int64_t nnz,
                            const uint64_t* keys, const uint64_t* bmps, const uint64_t* offsets,
                            int64_t offsets_len, const void* values, int32_t dtype, int32_t mem,
                            int32_t transposed, void* stream, bmsp_matrix_t* out);

int bmsp_destroy(bmsp_matrix_t m);

/* New values, same structure.  Overwrite m's values; keys, bitmaps and offsets stay.  values: m's nnz entries in m's own compact
 * order (the order of bmsp_view.values), fp32 or fp16 (dtype), host or device memory (mem); converted to m's dtype with round to
 * nearest, as the constructors convert.  values == NULL: the caller has written m's values in place through bmsp_view.values, and
 * only the library's own copies of them are refreshed.  Every copy a product keeps (a B operand's packed records and fine index)
 * is rewritten; the SpMV plan holds no values and is kept.  A device source is asynchronous on `stream`; a host source is
 * synchronous.  No counterpart in the reference. */
int bmsp_set_values(bmsp_matrix_t m, const void* values, int32_t dtype, int32_t mem, void* stream);
/* The same, with the values given as a CSR that has exactly m's pattern: row_ptr int32[num_rows+1], col_idx int32 ascending in
 * each row, vals fp32 or fp16.  Works for both orientations: a plain A and a transposed-operand Bt built from the same CSR take
 * the same arrays.  A different pattern (an extra, missing or moved entry, a row_ptr that does not span nnz) fails with
 * BMSP_ERR_INVALID and leaves m's values as they were.  The pattern is checked on the device before anything is written, and the
 * check's result is read back once: the call synchronises `stream`. */
int bmsp_set_values_csr(bmsp_matrix_t m, const int32_t* row_ptr, const int32_t* col_idx, const void* vals, int32_t vals_dtype,
                        int32_t mem, void* stream);

/* ---- access -------------------------------------------------------------------------------- */
int bmsp_get(bmsp_matrix_t m, bmsp_view* view);
/* Copy the four interchange arrays to host buffers (any may be NULL).  offsets gets offsets_len. */
int bmsp_download(bmsp_matrix_t m, uint64_t* keys, uint64_t* bmps, uint64_t* offsets, void* values);
/* bmSparse -> COO on the device, copied to host; order = block order then bit order; vals fp32.
 * Replaces bmSpMatrix::generate_coo (bmSpMatrix.cu:320-363). */
int bmsp_to_coo(bmsp_matrix_t m, int32_t* rows, int32_t* cols, float* vals);
/* Compare with a host COO (any order): replaces bmSpMatrix::compare (bmSpMatrix.cu:381-432), but
 * returns real numbers: entries only in `m`, entries only in the COO, mean and max relative error
 * (|exp-real| / max(|exp|, 1e-8), the reference's metric :418) over the common entries. */
int bmsp_compare(bmsp_matrix_t m, int64_t nnz, const int32_t* rows, const int32_t* cols,
                 const float* vals, int64_t* only_in_m, int64_t* only_in_coo, double* mean_rel_err,
                 double* max_rel_err);

/* bmSparse -> CSR on the device (row-major decode: the blocks of a block row are already in column order, so no sort): row_ptr
 * int32[num_rows + 1], col_idx int32[nnz] ascending inside each row, vals fp32[nnz].  `mem` says where the three output arrays
 * live (BMSP_DEVICE: written in place, asynchronous on `stream`; BMSP_HOST: copied out, synchronous).  This is the export the
 * reference's CSRMatrix class was declared for (include/CSRMatrix.h:15-17) and what feeds cuSPARSE / cusp consumers. */
int bmsp_to_csr(bmsp_matrix_t m, int32_t* row_ptr, int32_t* col_idx, float* vals, int32_t mem, void* stream);
/* bmsp_compare against a CSR (columns ascending inside each row), on the device: both sides are in key order, so one thread
 * per row merges the two column lists -- nothing is sorted and nothing but four numbers comes back to the host. */
int bmsp_compare_csr(bmsp_matrix_t m, const int32_t* row_ptr, const int32_t* col_idx, const float* vals, int32_t mem,
                     void* stream, int64_t* only_in_m, int64_t* only_in_csr, double* mean_rel_err, double* max_rel_err);

/* ---- operators ----------------------------------------------------------------------------- */
/* y = A x.  Replaces bmSparse_SpMV<ValueIn,ValueOut>(A, v, u, batched) (SPMV.cu:191-230).
 * x: [num_cols] device, fp32 (x_dtype = BMSP_F32) or fp16; y: [num_rows] device fp32.
 * Asynchronous on `stream`; rows of empty block rows are written as 0. */
int bmsp_spmv(bmsp_matrix_t A, const void* x, int32_t x_dtype, float* y, void* stream);
/* y_host = A x_host with both vectors in HOST memory (pinned for full speed; pageable works but serialises).
 * The reference's driver does this by hand around the operator: cudaMemcpy of v to the device, bmSparse_SpMV,
 * cudaMemcpy of u back (SPMV.cu:276-285, :299, :308-309).  Here the three steps are one call and are pipelined:
 * the block rows run in chunks, each chunk starts as soon as the x columns it touches have arrived and its y
 * slice leaves while the next chunk runs (H2D and D2H share the full-duplex link).  Ordered after earlier work on
 * `stream`; y_host is complete once `stream` is synchronised.  One call at a time per matrix. */
int bmsp_spmv_host(bmsp_matrix_t A, const void* x_host, int32_t x_dtype, float* y_host, void* stream);
/* Algorithmic bytes of one SpMV on the compact surface (SURVEY.md section 8d). */
int bmsp_spmv_bytes(bmsp_matrix_t A, int32_t x_dtype, int64_t* bytes);

/* C = A * B, A plain, Bt = B in transposed-operand form, C plain fp32.  Replaces
 * bmSparse_mult<valueIn,valueOut>(A, B, C, mode, VERBOSE, tc_version) (SPGEMM.cu:827-1223).
 * opts and info may be NULL.  Synchronises the stream twice (C sizes must reach the host). */
int bmsp_spgemm(bmsp_matrix_t A, bmsp_matrix_t Bt, const bmsp_spgemm_opts* opts, void* stream,
                bmsp_matrix_t* C, bmsp_spgemm_info* info);

/* SpGEMM plans: the same A * B formed again and again with new values on an unchanged pattern (AMG set-up, Jacobian products,
 * iterations over a fixed graph).  C's structure depends on the operands' structure only, so a plan keeps C and what its NUMERIC
 * pass reads, and bmsp_spgemm_numeric recomputes C's values alone.  No counterpart in the reference. */
typedef struct bmsp_spgemm_plan_s* bmsp_spgemm_plan_t;
/* Runs C = A * Bt exactly as bmsp_spgemm does (same opts, errors, C and info; synchronises twice) and keeps what the numeric
 * pass needs.  The plan holds A, Bt and C by pointer: destroy it before any of them. */
int bmsp_spgemm_plan_create(bmsp_matrix_t A, bmsp_matrix_t Bt, const bmsp_spgemm_opts* opts, void* stream,
                            bmsp_spgemm_plan_t* plan, bmsp_matrix_t* C, bmsp_spgemm_info* info);
/* Recomputes C's values from A's and Bt's current values (bmsp_set_values / bmsp_set_values_csr).  Only enqueues work on
 * `stream`: no host synchronisation, no allocation, no read-back, so it can be captured into a CUDA graph.  A plan owns its
 * queue counters and scratch: its calls must be ordered on one stream at a time; different plans may run concurrently. */
int bmsp_spgemm_numeric(bmsp_spgemm_plan_t plan, void* stream);
/* Device memory the plan retains (bytes, allocation padding included; C and the operands not counted). */
int bmsp_spgemm_plan_bytes(bmsp_spgemm_plan_t plan, int64_t* bytes);
/* Frees the plan's memory, ordered behind its last bmsp_spgemm_numeric.  Call before A, Bt or C are destroyed. */
int bmsp_spgemm_plan_destroy(bmsp_spgemm_plan_t plan);

/* Plain form <-> transposed-operand form of the same matrix (bitmap 8x8 transpose + value
 * permutation inside each block; keys unchanged).  The reference can only get the B operand by
 * re-reading the file with transposed=true (SPGEMM.cu:1262); its transpose8 sketch
 * (SPGEMM.cu:759-781) is unused.  out_dtype lets an fp32 product feed the next multiply as fp16. */
int bmsp_block_transpose(bmsp_matrix_t A, int32_t out_dtype, void* stream, bmsp_matrix_t* At);

/* A^T as a new matrix: rows and columns swapped, stored plain (out_transposed = 0: SpMV operand, left SpGEMM operand) or in
 * transposed-operand form (out_transposed = 1: the B of X * A^T), values converted to out_dtype.  A may be in either form.
 * Enqueued on `stream` only: no host synchronisation, no read-back.  Transposing twice gives A's arrays bit for bit.
 * No counterpart in the reference. */
int bmsp_matrix_transpose(bmsp_matrix_t A, int32_t out_dtype, int32_t out_transposed, void* stream, bmsp_matrix_t* At);

/* C = alpha*A + beta*B as a new matrix.  A and B: same shape, same storage form (both plain or both transposed-operand), any
 * dtype each.  C's pattern is the UNION of A's and B's patterns: entries whose sum is zero are kept (the pattern depends on
 * the operands' patterns only).  Each value is fl(fl(alpha*a) + fl(beta*b)) in fp32, where a missing entry counts as 0. It is
 * rounded once to out_dtype.  C is stored in A's form with offsets_len = block_num.  Synchronises `stream` once, because C's
 * block and value counts must reach the host.  No counterpart in the reference. */
int bmsp_add(float alpha, bmsp_matrix_t A, float beta, bmsp_matrix_t B, int32_t out_dtype, void* stream, bmsp_matrix_t* C);

/* ---- multi-GPU helpers (block-row sharding, SURVEY.md section 8e) --------------------------- */
/* Split block rows into nparts contiguous ranges balanced by SpMV bytes (weight_spgemm = 0) or by
 * candidate SpGEMM pairs against Bt (weight_spgemm = 1, Bt required).  bounds: int32[nparts+1]. */
int bmsp_partition_block_rows(bmsp_matrix_t A, bmsp_matrix_t Bt, int32_t nparts,
                              int32_t weight_spgemm, int32_t* bounds, void* stream);
/* New matrix holding block rows [brow_begin, brow_end) of A (row indices kept global unless
 * rebase_rows != 0, in which case they start at 0 and num_rows shrinks). */
int bmsp_slice_block_rows(bmsp_matrix_t A, int32_t brow_begin, int32_t brow_end, int32_t rebase_rows,
                          void* stream, bmsp_matrix_t* out);

/* Multi-GPU SpMV with the halo exchange over peer memory (NVLink P2P stores), fused into the product.
 * Every rank owns a contiguous row range, keeps x for the columns it touches ("extended range") in three
 * rotating peer-mapped buffers and an inbox of epoch flags (bmsp_peer_alloc / bmsp_peer_open).  One step:
 *   bmsp_spmv_halo(A_local, x_ext[cur], own slice of x_ext[nxt], desc[nxt], e, e + 1, stream)
 * waits (in the kernel) until every peer published epoch e, computes y, stores the rows each peer needs straight
 * into that peer's x_ext[nxt] and publishes epoch e + 1.  No NCCL call, no extra launch (row-tiled kernel; the
 * block-parallel kernel uses a wait and a push kernel around the product).  Three buffers, not two: a peer may
 * write the next-but-one buffer while this rank's kernel still reads the current one.
 * Descriptor rules (BMSP_ERR_INVALID otherwise): n_push and n_peer in [0, BMSP_HALO_MAX]; every push range
 * 0 <= lo <= hi <= rows with lo a multiple of 4 and a 16-byte aligned push_dst; scratch set when n_peer > 0;
 * n_push > 0 only with n_peer > 0 (n_peer counts every peer of both directions, so it includes each peer
 * pushed to).  An empty range (lo == hi) pushes nothing.  With n_peer == 0 the call is the plain product. */
#define BMSP_HALO_MAX 8
typedef struct {
    int32_t n_push;                      /* row ranges of my y that some peer needs                          */
    int32_t push_lo[BMSP_HALO_MAX];      /* local rows [lo, hi), lo a multiple of 4                           */
    int32_t push_hi[BMSP_HALO_MAX];
    void* push_dst[BMSP_HALO_MAX];       /* peer-mapped address of row push_lo[i] inside the peer's x buffer  */
    int32_t n_peer;                      /* peers to signal and to wait for (union of both directions)        */
    void* peer_flag[BMSP_HALO_MAX];      /* my slot in the peer's inbox (peer-mapped uint32)                  */
    const void* my_flag[BMSP_HALO_MAX];  /* the peer's slot in my inbox (local uint32)                         */
    void* scratch;                       /* local device memory, 2 x uint32, zero-initialised                 */
    int32_t own_col_lo, own_col_hi;      /* columns of x_ext that are this rank's own slice: row tiles whose  */
                                         /* columns stay inside never wait for a peer                          */
} bmsp_halo_desc;
int bmsp_spmv_halo(bmsp_matrix_t A, const float* x_ext, float* y_own, const bmsp_halo_desc* halo,
                   uint32_t wait_epoch, uint32_t signal_epoch, void* stream);
/* Push rows of y_own to the peers and publish signal_epoch (first exchange after x is set). */
int bmsp_halo_push(const float* y_own, int32_t rows, const bmsp_halo_desc* halo, uint32_t signal_epoch, void* stream);
/* timed_out != 0: a wait gave up after 4 s (a peer died); results since then are invalid. */
int bmsp_halo_status(const bmsp_halo_desc* halo, void* stream, int32_t* timed_out);
/* Peer-mapped device memory: allocate + export a 64-byte CUDA IPC handle, open a peer's handle, close, free. */
int bmsp_peer_alloc(int64_t bytes, void** ptr, void* handle64);
int bmsp_peer_open(const void* handle64, void** ptr);
int bmsp_peer_close(void* ptr);
int bmsp_peer_free(void* ptr);

/* ---- test hook ------------------------------------------------------------------------------- */
/* Runs the device routine that forms the boolean 8x8 block product (bmp_calculator,
 * SPGEMM.cu:787-810) on n host pairs; used by the parity tests only. */
int bmsp_debug_pair_bitmap(int64_t n, const uint64_t* a, const uint64_t* bt, uint64_t* out);

/* What the SpMV plan of A chose, and how its tiles and work items fall into the kernels' branches: lets a test assert that its
 * input reaches the branch it is written for.  Builds the plan (on `stream`) if A has none, then reads it back (synchronises
 * `stream`).  A must be plain and non-empty.  Used by the tests only. */
typedef struct {
    int32_t path;              /* 0 row-tiled, 1 block-parallel                                                  */
    int32_t kernel;            /* row-tiled: 0 streaming kernel, 1 one CTA per tile                              */
    int32_t tile_rows, npal;   /* block rows per tile; palette entries (0: no palette)                           */
    int32_t cap_blk, cap_val, cap_lines;   /* a tile's shared-memory capacities: blocks, values, x lines         */
    int32_t ntiles;
    int32_t empty_tiles;       /* tiles without blocks                                                           */
    int32_t unplanned_tiles;   /* tiles the planner left to global memory: ...                                   */
    int32_t unplanned_blocks;  /*   ... because they have more blocks than it sorts (2048)                       */
    int32_t unplanned_lines;   /*   ... because they touch more x lines than it offsets (1900)                   */
    int32_t over_cap_tiles;    /* planned tiles above a capacity: read from global memory too                    */
    int32_t tail_line_tiles;   /* tiles whose last x line reaches past the last column (guarded load)            */
    int32_t runs[4];           /* non-empty planned tiles by runs of consecutive x lines (runs[0]: more than 3)  */
    int32_t n_work, n_bundles, n_split_rows;   /* block-parallel: work items, bundles of four short block rows,
                                                  block rows sliced into several items                          */
} bmsp_spmv_plan_info;
int bmsp_debug_spmv_plan(bmsp_matrix_t A, bmsp_spmv_plan_info* out, void* stream);

/* Whether the SpMV plan of A streams row shapes: the streaming kernel's palette layout in which every block row names one of a
 * per-matrix table of block-word sequences instead of streaming a word per block.  *nshapes = distinct shapes, *nwords = words of
 * the table (padded to a multiple of 4); both -1 when the plan uses another layout.  Builds the plan as bmsp_debug_spmv_plan does.
 * Used by the tests only. */
int bmsp_debug_spmv_shapes(bmsp_matrix_t A, int32_t* nshapes, int32_t* nwords, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BMSPARSE_B200_H_ */
