// transpose_kernels.cuh -- A^T of a resident CSR built in HBM (spmv_b200_csr_transpose).
//
// New code (no reference counterpart).  The transpose is a stable sort of A's entries by column:
// row j of A^T lists column j of A in increasing row order, and entries of one row of A that share
// a column keep their order.  The sort itself is cub::DeviceRadixSort over (column, entry index);
// the kernels here prepare its input and gather its output.  Nothing is combined with atomics
// except the exact integer column counts, so the result is the same on every run.
#pragma once

#include "common.cuh"

namespace b200 {

// One warp per row of A: for every entry k of row r, row_of[k] = r, key[k] = ja[k], idx[k] = k
// (the sort's key and value inputs), and count[ja[k]] += 1 (entries per column = per row of A^T).
template <typename OffT>
__global__ void transpose_prep_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                                      long long M, int *__restrict__ row_of, int *__restrict__ key,
                                      int *__restrict__ idx, int *__restrict__ count) {
      const int lane = threadIdx.x & 31;
      const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
      for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < M; r += warps) {
            const long long k1 = (long long)irp[r + 1];
            for (long long k = (long long)irp[r] + lane; k < k1; k += 32) {
                  const int c = ja[k];
                  row_of[k] = (int)r;
                  key[k] = c;
                  idx[k] = (int)k;
                  atomicAdd(count + c, 1);
            }
      }
}

// Output position p holds source entry k = perm[p]: t_ja[p] = row of k in A, t_as[p] = as[k].
// perm may alias t_ja (each position reads its own slot before writing it).
__global__ void transpose_fill_kernel(const int *perm, const int *__restrict__ row_of,
                                      const double *__restrict__ as, long long nz, int *t_ja,
                                      double *__restrict__ t_as) {
      for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nz;
           p += (long long)gridDim.x * blockDim.x) {
            const int k = perm[p];
            t_ja[p] = row_of[k];
            t_as[p] = as[k];
      }
}

} // namespace b200
