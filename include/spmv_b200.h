/* spmv_b200.h -- resident-matrix ("handle") API of libspmv_b200.
 *
 * NEW SURFACE, no reference counterpart.  The reference launchers
 * (src/cuda_csr.cu:180-233, src/cuda_hll.cu:154-260) upload the matrix, run
 * one launch and free everything on every call.  The entry points in
 * cuda_csr.h / cuda_hll.h keep that calling convention; underneath they use
 * the API below, which keeps a matrix resident in HBM, runs y = A*x on
 * DEVICE pointers on a caller-supplied stream, and times launches properly.
 * It is also what bench.py, the parity tests and the multi-GPU iterated SpMV
 * bind.  Plain C ABI: pointers, sizes, ints -- no CUDA or torch types
 * (a stream is a `void *` holding a cudaStream_t; NULL = default stream).
 *
 * Conventions
 *   - functions returning int: 0 = success, negative errno-style code on
 *     failure; functions returning a pointer: NULL on failure.  In both cases
 *     spmv_b200_last_error() holds a message for the calling thread.
 *   - "d_" parameters are device pointers, everything else is host memory.
 *   - there is NO CPU fallback: with no usable GPU every create/run fails.
 *   - threading: a handle is used by one thread at a time (launch plans are built lazily on
 *     first use of a kernel); different handles may be used concurrently; the reference-style
 *     entry points of cuda_csr.h / cuda_hll.h serialise on an internal lock.
 *   - devices: one process per GPU (spmv_b200_set_device once, early) or one process driving
 *     several GPUs (spmv_b200_dist_group_*).  Handles remember the device they were created on;
 *     the caller makes that device current (spmv_b200_set_device) before using a handle.  The
 *     scratch buffers of the host-pointer calls and of spmv_b200_flush_l2 exist per device.
 */
#ifndef SPMV_B200_H
#define SPMV_B200_H

#include <stddef.h>
#include <stdint.h>

#include "csr.h"
#include "hll.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- kernel selectors (same numbering as the CSV `kernel` column) -------- */
enum spmv_b200_csr_kernel {
      SPMV_B200_CSR_THREAD_ROW = 0, /* one thread per row */
      SPMV_B200_CSR_WARP_ROW = 1,   /* one warp per row */
      SPMV_B200_CSR_ADAPTIVE = 2,   /* chosen per matrix: staged tiles for regular rows, sorted
                                       slices (SELL-P) for ragged rows or scattered columns */
      SPMV_B200_CSR_BLOCK_ROW = 3,  /* one CTA per row */
      SPMV_B200_CSR_STREAM = 4,     /* cp.async.bulk staged row tiles (falls back to the
                                       adaptive choice where staging cannot win) */
      SPMV_B200_CSR_NUM_KERNELS = 5
};

enum spmv_b200_hll_kernel {
      SPMV_B200_HLL_THREAD_ROW_RM = 0, /* thread per row (row-major input) */
      SPMV_B200_HLL_THREAD_ROW = 1,    /* thread per row, scalar loads */
      SPMV_B200_HLL_WARP_HACK = 2,     /* warp per hack, lane = row (headline); column panels
                                          when x is larger than the L2 and the columns scatter */
      SPMV_B200_HLL_STREAM = 3,        /* cp.async.bulk staged hacks */
      SPMV_B200_HLL_NUM_KERNELS = 4
};

/* ---- library / device ---------------------------------------------------- */
const char *spmv_b200_last_error(void);
const char *spmv_b200_version(void);
int spmv_b200_device_count(void);
int spmv_b200_set_device(int ordinal);

typedef struct {
      char name[128];
      int cc_major, cc_minor;
      int sm_count;
      int l2_bytes_mb;
      int64_t hbm_bytes;
      int max_smem_per_block;
} spmv_b200_devinfo;
int spmv_b200_device_info(spmv_b200_devinfo *out);

/* ---- raw device memory (for C hosts and ctypes callers without torch) ---- */
void *spmv_b200_dmalloc(size_t bytes);
int spmv_b200_dfree(void *d_ptr);
int spmv_b200_h2d(void *d_dst, const void *src, size_t bytes, void *stream);
int spmv_b200_d2h(void *dst, const void *d_src, size_t bytes, void *stream);
int spmv_b200_dmemset(void *d_dst, int byte, size_t bytes, void *stream);
int spmv_b200_stream_sync(void *stream);
/* Pinned host staging memory (e2e path). */
void *spmv_b200_host_alloc(size_t bytes);
int spmv_b200_host_free(void *ptr);
/* Page-lock / release memory the caller owns (cudaHostRegister).  The caller must unregister
 * before freeing it; the host-pointer calls use registered buffers in place. */
int spmv_b200_host_register(void *ptr, size_t bytes);
int spmv_b200_host_unregister(void *ptr);
/* memcpy on the library's copy threads (what the host-buffer calls use between pageable memory
 * and their page-locked bounce buffers: non-temporal stores, the CPUs the cpuset allows;
 * SPMV_B200_COPY_THREADS overrides the team size). */
int spmv_b200_host_copy(void *dst, const void *src, size_t bytes);
/* Overwrite a scratch buffer four times the size of the L2, then read half of it back, so the
 * next launch starts cold AND the L2 holds no dirty lines whose write-back it would pay for. */
int spmv_b200_flush_l2(void *stream);

/* ---- resident CSR --------------------------------------------------------- */
typedef struct spmv_b200_csr spmv_b200_csr;

/* Upload a host CSR (copies; the host arrays may be freed afterwards) and
 * build the launch plan (row bins, stream tiles). */
spmv_b200_csr *spmv_b200_csr_create(const sparse_csr *A);

/* General form used for shards: `irp` holds M+1 row offsets of width
 * `irp_bytes` (4 or 8); column indices are stored as (JA[k] - col_offset) and
 * must land in [0, n_local): the shard multiplies a local slice of x that
 * starts at global column `col_offset`.  `cuts`/`n_cuts` (may be NULL/0) are
 * row indices at which launch tiles must break so that
 * spmv_b200_csr_spmv_rows() can be called on [cuts[i], cuts[i+1]). */
spmv_b200_csr *spmv_b200_csr_create_ex(int64_t M, int64_t n_local, int64_t NZ,
                                       const void *irp, int irp_bytes,
                                       const int *JA, const double *AS,
                                       int64_t col_offset, const int64_t *cuts,
                                       int n_cuts);

/* 27-point stencil on an nx*ny*nz grid (diag 26, others -1, lexicographic
 * numbering, x fastest, sorted columns), rows of planes [z0, z1) generated
 * directly in HBM.  Columns are stored relative to `col_offset`. */
spmv_b200_csr *spmv_b200_csr_gen_stencil27(int nx, int ny, int nz, int z0,
                                           int z1, int64_t col_offset,
                                           int64_t n_local,
                                           const int64_t *cuts, int n_cuts);

/* Aᵀ of a resident CSR as a new resident CSR, built on A's device: row j lists column j of A in
 * increasing row order (entries of one row with equal columns keep their order; values are copied,
 * never summed).  A shard transposes its local block (n_local rows, M columns, col_offset 0, no
 * cuts).  Synchronous; A is unchanged; destroy both handles separately.  NULL + last_error on
 * failure; -ENOTSUP for 2^31 or more entries. */
spmv_b200_csr *spmv_b200_csr_transpose(const spmv_b200_csr *A);

/* C = A * B of two resident CSR handles, built on their device as a new resident CSR.
 * Shape: C has A's M rows and B's N columns (N is n_local for a shard: a shard multiplies its
 * local block); it needs A.N == B.M.  C has col_offset 0 and no cuts.
 * Pattern: row i of C lists each column j once, in increasing column order, for every (i, j) with
 * at least one product, even when the sum is zero; explicit zeros of the inputs still produce
 * entries.  The inputs may have unsorted rows and repeated (row, col) entries.
 * Values: the products of row i are taken in the order p over A's row i, then q over B's row
 * ja_A[p], both in stored order; C[i][j] is the left-to-right sum of those that land in column j,
 * starting from the first, each product a_p * b_q rounded to FP64 before it is added (no fused
 * multiply-add).  So a lone -0.0 stays -0.0, NaN and Inf propagate, and the result is the same on
 * every run.
 * Synchronous, on A's device (the current device is restored); A and B are unchanged; destroy all
 * three handles separately.  Row offsets of either input may be 32- or 64-bit, and the number of
 * products may exceed 2^31.  NULL + last_error on failure: -EINVAL for a null handle, A.N != B.M
 * or handles on different devices; -ENOTSUP when C would have 2^31 - 64 or more entries (found
 * before C is allocated); -ENOMEM when the temporaries do not fit. */
spmv_b200_csr *spmv_b200_csr_spgemm(const spmv_b200_csr *A, const spmv_b200_csr *B);

#define SPMV_B200_COO_SUM_DUPLICATES 1
/* Resident CSR from n entries (d_row[k], d_col[k], d_val[k]) in device memory of the current
 * device.  idx_bytes = 4 or 8 (both index arrays; torch indices are int64).  Row r of the result
 * lists the entries of row r in increasing column order.  Entries with equal (row, col) keep
 * their input order, or, with SPMV_B200_COO_SUM_DUPLICATES, become one entry whose value is
 * their left-to-right sum in input order, starting from the first value.  Nothing is dropped for
 * being zero.  The build is ordered after earlier work on `stream` and is synchronous.  The
 * caller's arrays are not retained.  NULL + last_error on failure: -EINVAL for a bad shape, index
 * width or flag, a null array, an array that is not device memory of the current device, or an
 * index out of range (the message names the first such entry); -ENOTSUP for 2^31 - 64 or more
 * entries; -ENOMEM when the temporaries do not fit. */
spmv_b200_csr *spmv_b200_csr_from_coo(int64_t M, int64_t N, int64_t n, const void *d_row,
                                      const void *d_col, int idx_bytes, const double *d_val,
                                      int flags, void *stream);

int64_t spmv_b200_csr_rows(const spmv_b200_csr *h);
int64_t spmv_b200_csr_cols(const spmv_b200_csr *h);
int64_t spmv_b200_csr_nnz(const spmv_b200_csr *h);
/* Copy the device arrays back (any of the outputs may be NULL).  `irp64`
 * receives M+1 64-bit offsets. */
int spmv_b200_csr_download(const spmv_b200_csr *h, int64_t *irp64, int *JA,
                           double *AS);
/* Rows per adaptive bin: out[0..5] = {empty, sub-warp, warp, block, split,
 * tiles}.  Diagnostic. */
int spmv_b200_csr_plan_info(const spmv_b200_csr *h, int64_t *out, int n_out);
/* Column codes of the staged row-tile plans built so far (kernels 2 / 4): out[0..4) = {state
 * (0 none built, 1 coded, -1 some plan keeps int32 columns: a tile has more than 256 distinct
 * column offsets), coded tiles, largest dictionary of a tile, bytes of the code blocks}. */
int spmv_b200_csr_codes_info(const spmv_b200_csr *h, int64_t *out, int n_out);

/* y[0..M) = A * x on `stream` (asynchronous).  d_x has n_local entries. */
int spmv_b200_csr_spmv(spmv_b200_csr *h, int kernel, int warps_per_block,
                       const double *d_x, double *d_y, void *stream);
/* Same for rows [row0, row1) only; y is still indexed by local row. */
int spmv_b200_csr_spmv_rows(spmv_b200_csr *h, int kernel, int warps_per_block,
                            int64_t row0, int64_t row1, const double *d_x,
                            double *d_y, void *stream);
/* Fused epilogue for the multi-GPU halo exchange: besides y[row], rows in
 * [push_row0[i], push_row1[i]) are also stored to d_push_dst[i][row -
 * push_row0[i]] (a peer GPU's halo buffer mapped through CUDA IPC).  Up to 8
 * push ranges. */
int spmv_b200_csr_spmv_rows_push(spmv_b200_csr *h, int kernel,
                                 int warps_per_block, int64_t row0,
                                 int64_t row1, const double *d_x, double *d_y,
                                 int n_push, const int64_t *push_row0,
                                 const int64_t *push_row1,
                                 double *const *d_push_dst, void *stream);
/* K right-hand sides in one pass (SURVEY 8(f)3): Y = A X with X[n_local][k] and Y[M][k] row-major
 * (the k values of a row are adjacent), k = 2 or 4, d_X 16-byte aligned.  Same routes as kernel id 2
 * (sorted slices for ragged rows / scattered columns, rows straight from CSR otherwise); every
 * gather returns k useful values from the 32-byte sector it moves, so gather-bound matrices
 * (BASELINE configs[2], [3]) run close to k times the single-vector rate.  Asynchronous on `stream`. */
int spmv_b200_csr_spmm(spmv_b200_csr *h, int k, const double *d_X, double *d_Y, void *stream);
/* Fused iteration step (SURVEY 8(f)3; the loop around reference src/csr.c:182-199 when SpMV is
 * iterated): y = alpha * A x + beta * z in one pass over the matrix, and, when d_dot is
 * non-NULL, *d_dot = sum_i y_i * w_i (d_w may be d_y for ||y||^2; d_z and d_w may be NULL).
 * Kernels 2 and 4, whole matrix, no rows longer than a stage, no column panels: -ENOTSUP
 * otherwise.  The dot product is reduced in a fixed order (bit-reproducible run to run). */
int spmv_b200_csr_spmv_fused(spmv_b200_csr *h, int kernel, int warps_per_block,
                             const double *d_x, double *d_y, double alpha, double beta,
                             const double *d_z, const double *d_w, double *d_dot,
                             void *stream);
/* Host x in, host y out, in one call: x upload, row-chunk kernels and y download are pipelined
 * on three streams when the matrix is banded (see csrc/entry.cu).  Page-locked buffers
 * (spmv_b200_host_alloc / _register) are used in place, pageable ones go through page-locked
 * bounce buffers.  *kernel_ms (may be NULL) = span of the kernels.  Synchronous. */
int spmv_b200_csr_spmv_host(spmv_b200_csr *h, int kernel, int warps_per_block, const double *x,
                            double *y, double *kernel_ms);
/* SELL-P plan of this matrix (column-panelled, window-sorted slices; csrc/sell_kernels.cuh):
 * out[0..11) = {state (1 built), panels, sigma, slices, padded slots, entries in slices, rows
 * handled by the long-row kernels, gather span * 1e6, virtual-row chunk (0: none), rows split into
 * pieces, pieces}.
 * build != 0 builds the plan first. */
int spmv_b200_csr_sell_info(spmv_b200_csr *h, int build, int64_t *out, int n_out);
/* Device SELL-P arrays back to the host for bit-compare (any output may be NULL):
 * soff[panels*(slices+1)], perm[panels*slices*32], JA/AS[slots]. */
int spmv_b200_csr_sell_download(const spmv_b200_csr *h, int64_t *soff, int *perm, int *JA,
                                double *AS);
/* Host half of the SELL-P build (row order and slice offsets from per-panel row counts,
 * counts[p*M + r], -1 = row excluded); needs no GPU.  perm[K*S*32], soff[K*(S+1)], S = ceil(M/32). */
int spmv_b200_sell_plan(const int *counts, int64_t M, int K, int sigma, int *perm, int64_t *soff);
/* Host half of the virtual-row form (ragged matrices): sizes[4] = {virtual rows, slices, rows
 * split into pieces, pieces}; dest[slices*32] (row, -1, or -2-piece) and soff[slices+1] may be
 * NULL on a first call that only asks for the sizes.  `irp`: M+1 64-bit offsets.  No GPU. */
int spmv_b200_sell_plan_vrows(const int64_t *irp, int64_t M, int chunk, int sigma, int64_t *sizes,
                              int *dest, int64_t *soff);
/* Kernel launches one spmv call issues for this matrix/kernel. */
int spmv_b200_csr_launches(const spmv_b200_csr *h, int kernel);
/* Run `warmup` untimed + `reps` timed launches, each bracketed by CUDA events
 * on `stream`; ms_out[reps] receives per-launch milliseconds.  flush_l2 != 0
 * evicts L2 before every timed launch (outside the timed interval). */
int spmv_b200_csr_time(spmv_b200_csr *h, int kernel, int warps_per_block,
                       const double *d_x, double *d_y, int warmup, int reps,
                       int flush_l2, double *ms_out, void *stream);
void spmv_b200_csr_destroy(spmv_b200_csr *h);

/* ---- resident HLL --------------------------------------------------------- */
typedef struct spmv_b200_hll spmv_b200_hll;

/* Flatten + upload a host HLL of either layout. */
spmv_b200_hll *spmv_b200_hll_create(const sparse_hll *H, int is_col_major);
/* Build the device HLL straight from a resident CSR, on the GPU. */
spmv_b200_hll *spmv_b200_hll_from_csr(const spmv_b200_csr *A);

int64_t spmv_b200_hll_rows(const spmv_b200_hll *h);
int64_t spmv_b200_hll_cols(const spmv_b200_hll *h);
int64_t spmv_b200_hll_nnz(const spmv_b200_hll *h);
int64_t spmv_b200_hll_num_hacks(const spmv_b200_hll *h);
int64_t spmv_b200_hll_slots(const spmv_b200_hll *h); /* padded entries */
/* Device layout back to the host for bit-compare: hoff[num_hacks+1] slot
 * offsets, JA/AS[slots] column-major per hack with stride 32. */
int spmv_b200_hll_download(const spmv_b200_hll *h, int64_t *hoff, int *JA,
                           double *AS);

int spmv_b200_hll_spmv(spmv_b200_hll *h, int kernel, int warps_per_block,
                       const double *d_x, double *d_y, void *stream);
int spmv_b200_hll_spmv_fused(spmv_b200_hll *h, int kernel, int warps_per_block,
                             const double *d_x, double *d_y, double alpha, double beta,
                             const double *d_z, const double *d_w, double *d_dot,
                             void *stream);
int spmv_b200_hll_spmv_host(spmv_b200_hll *h, int kernel, int warps_per_block, const double *x,
                            double *y, double *kernel_ms);
int spmv_b200_hll_sell_info(spmv_b200_hll *h, int build, int64_t *out, int n_out);
int spmv_b200_hll_launches(const spmv_b200_hll *h, int kernel);
int spmv_b200_hll_time(spmv_b200_hll *h, int kernel, int warps_per_block,
                       const double *d_x, double *d_y, int warmup, int reps,
                       int flush_l2, double *ms_out, void *stream);
void spmv_b200_hll_destroy(spmv_b200_hll *h);

/* ---- cache used by the reference-style entry points ---------------------- */
/* The entry points of cuda_csr.h / cuda_hll.h keep the uploaded matrix resident between calls
 * (the reference uploads it on every call, src/cuda_csr.cu:180-195).  Policy:
 *   0  off    upload on every call
 *   1  hash   (default) re-hash the caller's arrays in full on every call, re-upload on change
 *   2  trust  key on host pointers + shape; call spmv_b200_invalidate() after editing in place
 * Also settable with SPMV_B200_CACHE=off|hash|trust. */
int spmv_b200_set_cache_policy(int policy);
/* Forget the device copy of one sparse_csr / sparse_hll (NULL: of all). */
void spmv_b200_invalidate(const void *matrix);
/* Drop every device copy and scratch buffer kept by the host-pointer calls. */
void spmv_b200_release_all(void);
/* Timing policy of the reference-style entry points (defaults 1 / 3; also
 * settable with SPMV_B200_WARMUP / SPMV_B200_REPS).  The returned duration is
 * the median of the timed repetitions.  reps = 0 asks for no separately timed
 * launches: the pipelined entry (banded matrix, page-locked x and y: x is
 * uploaded in column order while row chunks compute and y chunks travel back)
 * then returns the span of its single pass; other paths time one launch. */
void spmv_b200_set_timing(int warmup, int reps);
/* Counters since load: kernel launches issued, bytes copied H2D / D2H. */
void spmv_b200_counters(int64_t *launches, int64_t *h2d_bytes,
                        int64_t *d2h_bytes);

/* Experiment knobs used by bin/kbench sweeps and tests ("csr_stream_cfg", "hll_stream_cfg",
 * "force_wide", "pipeline", "pipe_chunks", "csr_pipe", "hll_pipe" (short rows / narrow hacks
 * through per-warp bulk-copy rings: -1 auto, 0 off, 1 whenever they fit), "csr_codes" (1, the
 * default: row-tile stream plans stream one-byte column codes where every tile allows; 0: int32
 * columns), "sell", "sell_panels",
 * "sell_sigma", "sell_panel_mb", "sell_max_row", "sell_chunk", "cache").
 * 0 or -EINVAL.  Knobs that change planning must be set before a handle is created. */
int spmv_b200_set_knob(const char *key, int value);

/* ---- inter-process peer memory (one process per GPU) --------------------- */
#define SPMV_B200_IPC_HANDLE_BYTES 64
int spmv_b200_ipc_export(void *d_ptr, unsigned char *handle64);
int spmv_b200_ipc_open(const unsigned char *handle64, void **d_ptr_out);
int spmv_b200_ipc_close(void *d_ptr);
int spmv_b200_enable_peer(int peer_device);

/* Step ordering between ranks without a host round trip (multi-GPU halo push):
 * spmv_b200_signal_peers  epoch := epoch + 1 (device word), then store it into
 *                         each of the n peer slots (peer HBM mapped through IPC);
 * spmv_b200_wait_peers    spin (at most max_spins polls per slot, then *d_error
 *                         is set to 1 + slot index and the kernel returns) until
 *                         each of my n slots holds a value >= my epoch.
 * Both are single-thread kernels on `stream`, capturable in a CUDA graph. */
int spmv_b200_signal_peers(void *d_epoch, int n, void *const *d_peer_slots,
                           void *stream);
int spmv_b200_wait_peers(const void *d_epoch, int n, void *const *d_my_slots,
                         uint64_t max_spins, int *d_error, void *stream);

/* ---- multi-GPU iterated SpMV: x_{k+1} = A x_k, rows partitioned over the GPUs of one box ----
 * NEW SURFACE (the reference is single-GPU); csrc/dist.cu describes the step.  Planning
 * functions are host-only and usable without a GPU. */
#define SPMV_B200_MAX_RANKS 16
#define SPMV_B200_DIST_BLOB_BYTES 512
enum spmv_b200_dist_mode {
      SPMV_B200_DIST_AUTO = 0, /* PUSH when the plan allows it (at most 8 peers per boundary segment and
                                  SPMV_B200_PUSH_ALL != 0 for more than 2), else NCCL */
      SPMV_B200_DIST_PUSH = 1, /* peer HBM written directly, epoch flags: halo rows by the SpMV epilogue;
                                  whole slices of a general matrix as row-block peer copies behind the
                                  running step (SPMV_B200_GATHER_BLOCKS, default 2) */
      SPMV_B200_DIST_NCCL = 2  /* ncclAllGather / grouped ncclSend+ncclRecv on a side stream */
};

/* Rows [r0, r1) of the global matrix, the global columns [c0, c1) they touch, and which local
 * rows read outside their own slice: rows [0, read_lo) may read columns < r0, rows
 * [read_hi, M) may read columns >= r1. */
typedef struct {
      int64_t r0, r1, c0, c1, read_lo, read_hi;
} spmv_b200_shard_desc;

typedef struct {
      int peer;
      int64_t g0, g1; /* global index range [g0, g1) */
} spmv_b200_xfer;

typedef struct {
      int rank, world;
      int mode;       /* SPMV_B200_DIST_PUSH or _NCCL, identical on every rank */
      int all_gather; /* every rank needs every slice and the slices are equal */
      int covered;    /* the row ranges tile this rank's column range */
      int n_send, n_recv, n_cuts;
      int64_t boundary_lo, boundary_hi; /* local rows [0,lo) and [hi,M) run before the exchange */
      int64_t cuts[2];                  /* pass to spmv_b200_csr_create_ex / _gen_stencil27 */
      int64_t halo_bytes;               /* received per step */
      spmv_b200_xfer send[SPMV_B200_MAX_RANKS], recv[SPMV_B200_MAX_RANKS];
} spmv_b200_dist_plan;

/* cuts[parts+1]: contiguous row ranges with balanced nnz -- a range is closed at the row whose
 * running nnz reaches total/parts, as the reference's partition_csr_rows (src/csr.c:218-276) --
 * each cut rounded up to a multiple of `align` rows.  `irp`: M+1 offsets of 4 or 8 bytes. */
int spmv_b200_partition_rows(int64_t M, const void *irp, int irp_bytes, int parts, int align,
                             int64_t *cuts);
/* Descriptor of rows [r0, r1): `irp` points at the r1-r0+1 offsets of those rows, `JA` at the
 * (global) columns of their first entry. */
int spmv_b200_shard_scan(int64_t r0, int64_t r1, const void *irp, int irp_bytes, const int *JA,
                         spmv_b200_shard_desc *out);
/* Descriptor of planes [z0, z1) of the 27-point stencil (no matrix needed). */
int spmv_b200_stencil27_shard_desc(int nx, int ny, int nz, int z0, int z1,
                                   spmv_b200_shard_desc *out);
/* Plan of `rank` from everybody's descriptor.  want_mode: enum spmv_b200_dist_mode. */
int spmv_b200_dist_make_plan(int rank, int world, const spmv_b200_shard_desc *table, int want_mode,
                             spmv_b200_dist_plan *out);

/* One rank (one process per GPU).  `shard` was created with col_offset = c0, n_local = c1-c0 and
 * plan->cuts; it is not owned.  Sequence: create -> export -> (caller gathers the blobs of all
 * ranks, rank-major) -> connect -> [barrier] set_x -> iterate ... -> sync / get_x -> destroy. */
typedef struct spmv_b200_dist spmv_b200_dist;
spmv_b200_dist *spmv_b200_dist_create(const spmv_b200_dist_plan *plan,
                                      const spmv_b200_shard_desc *table, spmv_b200_csr *shard,
                                      int kernel, int warps_per_block);
int spmv_b200_dist_export(spmv_b200_dist *d, unsigned char *blob);
int spmv_b200_dist_connect(spmv_b200_dist *d, const unsigned char *blobs);
/* x_0: own slice, host or device memory.  Collective; the whole job must be idle (sync +
 * barrier on the caller's side) before any rank calls it. */
int spmv_b200_dist_set_x(spmv_b200_dist *d, const double *x_own);
/* Queue k steps on the rank's stream (asynchronous). */
int spmv_b200_dist_iterate(spmv_b200_dist *d, int k);
/* `reps` regions of k steps, each bracketed by CUDA events on the rank's stream; ms_out[reps].
 * Returns after the stream has drained. */
int spmv_b200_dist_time(spmv_b200_dist *d, int k, int reps, double *ms_out);
/* Wait for the rank's streams; -ETIMEDOUT if a wait kernel gave up on a neighbour. */
int spmv_b200_dist_sync(spmv_b200_dist *d);
double *spmv_b200_dist_x(spmv_b200_dist *d);      /* device: own slice of the current x */
double *spmv_b200_dist_xlocal(spmv_b200_dist *d); /* device: current x over [c0, c1) */
int spmv_b200_dist_get_x(spmv_b200_dist *d, double *host_out); /* own slice, after a sync */
void *spmv_b200_dist_stream(spmv_b200_dist *d);   /* cudaStream_t the steps are queued on */
int64_t spmv_b200_dist_steps(const spmv_b200_dist *d);
int spmv_b200_dist_mode(const spmv_b200_dist *d);
int spmv_b200_dist_has_graph(const spmv_b200_dist *d);
void spmv_b200_dist_destroy(spmv_b200_dist *d);

/* One process driving n GPUs (devices 0..n-1, peer access): partition, shards, plans and wiring
 * in one call.  From a host CSR (square), or the 27-point stencil generated per shard in HBM. */
typedef struct spmv_b200_dist_group spmv_b200_dist_group;
spmv_b200_dist_group *spmv_b200_dist_group_create(const sparse_csr *A, int n_gpus, int kernel,
                                                  int warps_per_block, int mode);
spmv_b200_dist_group *spmv_b200_dist_group_stencil27(int nx, int ny, int nz, int n_gpus,
                                                     int kernel, int warps_per_block, int mode);
int spmv_b200_dist_group_size(const spmv_b200_dist_group *g);
spmv_b200_dist *spmv_b200_dist_group_rank(spmv_b200_dist_group *g, int rank);
int spmv_b200_dist_group_set_x(spmv_b200_dist_group *g, const double *x_host);
/* k steps on every GPU; *ms_out (may be NULL) = longest per-GPU CUDA-event time.  Synchronous. */
int spmv_b200_dist_group_iterate(spmv_b200_dist_group *g, int k, double *ms_out);
int spmv_b200_dist_group_get_x(spmv_b200_dist_group *g, double *x_host);
void spmv_b200_dist_group_destroy(spmv_b200_dist_group *g);

#ifdef __cplusplus
}
#endif

#endif /* SPMV_B200_H */
