// coo_kernels.cuh -- resident CSR built in HBM from COO triplets (spmv_b200_csr_from_coo).
//
// New code (no reference counterpart).  Each entry gets the sort key row * 2^cb + col
// (cb = column bits), so that sorting the keys orders the entries by row and then by column.
// The sort itself is cub::DeviceRadixSort over (key, entry index), which is stable: entries with
// equal (row, col) keep their input order.  The kernels here prepare its input, mark where runs of
// equal keys start and write the CSR arrays.  Only the integer row counts use atomics; duplicate
// values are added by one thread, left to right, so the result is the same on every run.
#pragma once

#include "common.cuh"

namespace b200 {

// What the pack pass found: the first entry with an index out of range (INT_MAX: none), whether
// some key is smaller than the one before it, and whether some key equals the one before it.
struct CooStatus {
      int bad;
      int unsorted;
      int dup;
      int pad;
};

// One grid-stride pass over the n input entries: bounds check, key[k] = row << cb | col, and the
// comparison of each key with its predecessor.  Keys of out-of-range entries are not written (the
// build fails on them).
template <typename IdxT, typename KeyT>
__global__ void coo_pack_kernel(const IdxT *__restrict__ row, const IdxT *__restrict__ col, long long n,
                                long long M, long long N, int cb, KeyT *__restrict__ key,
                                CooStatus *__restrict__ st) {
      int bad = 0x7fffffff;
      bool unsorted = false, dup = false;
      for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n;
           k += (long long)gridDim.x * blockDim.x) {
            const long long r = (long long)row[k], c = (long long)col[k];
            if (r < 0 || r >= M || c < 0 || c >= N) {
                  bad = min(bad, (int)k);
                  continue;
            }
            const KeyT kk = (KeyT)r << cb | (KeyT)c;
            key[k] = kk;
            if (k > 0) {
                  const KeyT kp = (KeyT)(long long)row[k - 1] << cb | (KeyT)(long long)col[k - 1];
                  unsorted |= kk < kp;
                  dup |= kk == kp;
            }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
            bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, o));
      unsorted = __any_sync(0xffffffffu, unsorted);
      dup = __any_sync(0xffffffffu, dup);
      if ((threadIdx.x & 31) == 0) {
            if (bad != 0x7fffffff)
                  atomicMin(&st->bad, bad);
            if (unsorted)
                  st->unsorted = 1;
            if (dup)
                  st->dup = 1;
      }
}

// idx[k] = k: the value input of the sort, which comes out as the permutation.
__global__ void coo_iota_kernel(int *__restrict__ idx, long long n) {
      for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n;
           k += (long long)gridDim.x * blockDim.x)
            idx[k] = (int)k;
}

// head[p] = 1 where sorted position p starts a run of equal keys, for p < n; head[n] = 0.  An
// exclusive scan of head[0..n] then gives each run its output position and, in head[n], the
// number of output entries.
template <typename KeyT>
__global__ void coo_heads_kernel(const KeyT *__restrict__ key, long long n, int *__restrict__ head) {
      for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p <= n;
           p += (long long)gridDim.x * blockDim.x)
            head[p] = p < n && (p == 0 || key[p] != key[p - 1]);
}

// Sorted position p holds input entry perm[p] (perm == nullptr: the input was already sorted and
// p is the entry itself).  Without SUM every position is an output entry; with SUM the first
// position of each run writes output entry pos[p] and adds the run's values left to right,
// starting from the first one (so a lone -0.0 stays -0.0 and NaN / Inf propagate).  Each output
// entry counts itself in count[row].
template <typename KeyT, bool SUM>
__global__ void coo_fill_kernel(const KeyT *__restrict__ key, const int *__restrict__ perm,
                                const int *__restrict__ pos, const double *__restrict__ val, long long n,
                                int cb, int *__restrict__ ja, double *__restrict__ as,
                                int *__restrict__ count) {
      const KeyT col_mask = ((KeyT)1 << cb) - 1;
      for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n;
           p += (long long)gridDim.x * blockDim.x) {
            const KeyT k = key[p];
            if (SUM && p > 0 && key[p - 1] == k)
                  continue;
            double v = val[perm ? perm[p] : p];
            if (SUM)
                  for (long long j = p + 1; j < n && key[j] == k; ++j)
                        v += val[perm ? perm[j] : j];
            const long long q = SUM ? (long long)pos[p] : p;
            ja[q] = (int)(k & col_mask);
            as[q] = v;
            atomicAdd(count + (long long)(k >> cb), 1);
      }
}

} // namespace b200
