/* cuda_hll.h -- GPU HLL SpMV entry points exported by libspmv_b200.
 *
 * Same five symbols as the reference (include/cuda_hll.h:10-22; callers
 * src/hll.c:226-256).  H, x, y are HOST pointers; the host layout of H is the
 * one the entry point implies (row-major for _threads_row_major and
 * _halfwarp_row, column-major for _threads_col_major and _warp_block,
 * reference src/main.c:324-325) and its padding is JA = -1 / AS = 0.0.  On
 * upload the library flattens all hacks into ONE value buffer and ONE index
 * buffer, column-major per hack with a fixed stride of 32 rows, and rewrites
 * each -1 to the previous valid column of the row (0 for an empty row) --
 * the same branch-free device convention as reference src/cuda_hll.cu:173-195.
 * Return value: kernel milliseconds; <= 0 on error.
 *
 * CSV `kernel` ids (reference src/main.c:310-315):
 *   0 hll_spmv_cuda_threads_row_major  thread per row, scalar loads
 *                                      (row-major input transposed on upload)
 *   1 hll_spmv_cuda_threads_col_major  thread per row, scalar loads
 *   2 hll_spmv_cuda_warp_block         warp per hack, lane = row, 64-bit value / 32-bit
 *                                      index loads (128- and 256-bit loads measured
 *                                      slower); narrow hacks (width <= 8) through
 *                                      per-warp cp.async.bulk rings; column panels (SELL-P) when x is larger than
 *                                      the L2 and the columns scatter
 *   3 hll_spmv_cuda_halfwarp_row       warp per hack, streams staged in shared
 *                                      memory by cp.async.bulk (TMA)
 */
#ifndef SPMV_B200_CUDA_HLL_H
#define SPMV_B200_CUDA_HLL_H

#include "hll.h"

#ifdef __cplusplus
extern "C" {
#endif

void set_hll_warps_per_block(int wppb);

/* one prototype per variant of SPMV_HLL_CUDA_VARIANTS (see hll.h):
 *   double hll_spmv_cuda_<variant>(const sparse_hll *matrix, const double *x_host,
 *                                    double *y_host, void *unused);                  */
#define SPMV_DECLARE(suffix)                                                          \
    double hll_spmv_cuda_##suffix(const sparse_hll *matrix, const double *x_host,        \
                                    double *y_host, void *unused);
SPMV_HLL_CUDA_VARIANTS(SPMV_DECLARE)
#undef SPMV_DECLARE

#ifdef __cplusplus
}
#endif

#endif /* SPMV_B200_CUDA_HLL_H */
