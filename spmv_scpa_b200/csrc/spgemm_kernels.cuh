// spgemm_kernels.cuh -- C = A * B of two resident CSR handles built in HBM (spmv_b200_csr_spgemm).
//
// New code (no reference counterpart).  Three passes over the products a_p * b_q of each row i of
// A, taken in the order p in A's row i, then q in B's row ja_A[p], both in stored order:
//   count     P_i = sum of len_B(ja_A[p]): the row's products, an upper bound on its columns;
//   symbolic  one warp per row inserts the column keys into an open-addressing hash table and counts
//             the distinct ones (C's entries per row);
//   numeric   the same walk again, adding each product into its column's slot, then the occupied
//             slots are written, unsorted, to the row's place in C.  A segmented sort orders them.
// A warp step covers 32 consecutive products of one 32-entry chunk of A's row: a warp scan of the B
// row lengths of the chunk's entries tells each lane its (p, q), as in merge-path.  Lanes whose
// products share a column are grouped with __match_any_sync; the group's lowest lane inserts the
// key and adds the group's products to the slot one at a time, in lane order.  So every column's
// value is the left-to-right sum of its products starting from the first, each rounded to FP64
// before it is added (__dmul_rn / __dadd_rn: no contraction into FMA).  Only the integer key
// insertion uses atomics; the result is the same on every run.
//
// Tables hold a power of two slots, at least twice the row's bound min(P_i, B.N), so they are at
// most half full.  A table is either per warp in shared memory (SharedTable: all rows of one launch
// have the same size) or a row's own region of one table in global memory (GlobalTable: regions
// given by an offset array, sized from each row's bound).
#pragma once

#include "common.cuh"

namespace b200 {

constexpr int kSpgemmEmpty = -1; // key of a free slot (columns are >= 0)

struct SharedTable {
      static constexpr bool kShared = true;
};
struct GlobalTable {
      static constexpr bool kShared = false;
};

// Where the table of row number w of a launch lives.  slots: a power of two; shift = 32 - log2.
struct SpgemmTable {
      int *keys;
      double *vals; // numeric pass only
      unsigned mask;
      int shift;
};

// Rows of one launch: `rows[0..n)` are rows of A.  SharedTable: every table has `slots` slots.
// GlobalTable: row w's region is [toff[w], toff[w + 1]) of gkeys / gvals.
struct SpgemmRows {
      const int *rows;
      long long n;
      long long slots;
      const long long *toff;
      int *gkeys;
      double *gvals;
};

__device__ __forceinline__ int spgemm_log2(unsigned long long s) { return 63 - __clzll((long long)s); }

// Slot of key c: insert it if absent.  Returns the slot; *fresh tells whether this call inserted it.
// Keys never move once written, and within a warp step every key has one inserting lane, so a
// plain read that finds c or another key is final; only a free slot needs the CAS.
__device__ __forceinline__ unsigned spgemm_insert(const SpgemmTable &t, int c, bool *fresh) {
      unsigned s = ((unsigned)c * 2654435761u) >> t.shift & t.mask;
      while (true) {
            const int k = *(volatile int *)(t.keys + s);
            if (k == c) {
                  *fresh = false;
                  return s;
            }
            if (k == kSpgemmEmpty) {
                  const int old = atomicCAS(t.keys + s, kSpgemmEmpty, c);
                  if (old == kSpgemmEmpty || old == c) {
                        *fresh = old == kSpgemmEmpty;
                        return s;
                  }
            }
            s = (s + 1) & t.mask;
      }
}

// One pass of a warp over the products of row r (see the file comment).  Symbolic: returns, on
// every lane, the number of distinct columns.  Numeric: leaves each column's sum in its slot; the
// staging array holds one product per lane for the group leaders.
template <bool NUMERIC, typename OffA, typename OffB>
__device__ __forceinline__ int spgemm_row(const OffA *__restrict__ irp_a, const int *__restrict__ ja_a,
                                          const double *__restrict__ as_a, const OffB *__restrict__ irp_b,
                                          const int *__restrict__ ja_b, const double *__restrict__ as_b,
                                          long long r, const SpgemmTable &t, double *stage) {
      const int lane = threadIdx.x & 31;
      for (unsigned s = lane; s <= t.mask; s += 32)
            t.keys[s] = kSpgemmEmpty;
      __syncwarp();
      int fresh_count = 0;
      const long long a1 = (long long)irp_a[r + 1];
      for (long long pb = (long long)irp_a[r]; pb < a1; pb += 32) {
            const long long p = pb + lane;
            long long q0 = 0, len = 0;
            double av = 0.0;
            if (p < a1) {
                  const int k = ja_a[p];
                  q0 = (long long)irp_b[k];
                  len = (long long)irp_b[k + 1] - q0;
                  if (NUMERIC)
                        av = as_a[p];
            }
            long long inc = len; // inclusive scan of the chunk's B row lengths
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                  const long long v = __shfl_up_sync(0xffffffffu, inc, d);
                  if (lane >= d)
                        inc += v;
            }
            const long long q_base = q0 - (inc - len); // q of the entry's product number g: q_base + g
            const long long total = __shfl_sync(0xffffffffu, inc, 31);
            for (long long g0 = 0; g0 < total; g0 += 32) {
                  const long long g = g0 + lane;
                  int j = 0; // the chunk entry of product g: the first j with inc_j > g
#pragma unroll
                  for (int step = 16; step; step >>= 1)
                        if (__shfl_sync(0xffffffffu, inc, j + step - 1) <= g)
                              j += step;
                  const long long q = __shfl_sync(0xffffffffu, q_base, j) + g;
                  const double a = NUMERIC ? __shfl_sync(0xffffffffu, av, j) : 0.0;
                  const bool act = g < total;
                  const int c = act ? ja_b[q] : kSpgemmEmpty;
                  const unsigned grp = __match_any_sync(0xffffffffu, c);
                  if (NUMERIC)
                        stage[lane] = act ? __dmul_rn(a, as_b[q]) : 0.0;
                  __syncwarp();
                  if (act && lane == __ffs(grp) - 1) {
                        bool fresh;
                        const unsigned s = spgemm_insert(t, c, &fresh);
                        if (NUMERIC) {
                              double v = fresh ? stage[lane] : __dadd_rn(t.vals[s], stage[lane]);
                              for (unsigned m = grp & (grp - 1); m; m &= m - 1)
                                    v = __dadd_rn(v, stage[__ffs(m) - 1]);
                              t.vals[s] = v;
                        }
                        fresh_count += fresh;
                  }
                  __syncwarp();
            }
      }
#pragma unroll
      for (int d = 16; d; d >>= 1)
            fresh_count += __shfl_xor_sync(0xffffffffu, fresh_count, d);
      return fresh_count;
}

// Table of the launch's row number w for this warp.  Shared tables: keys of the block's warps,
// then their values (numeric), then 32 staging doubles per warp.
template <typename TABLE, bool NUMERIC>
__device__ __forceinline__ SpgemmTable spgemm_table(const SpgemmRows &rs, long long w, double **stage) {
      extern __shared__ __align__(16) unsigned char spgemm_smem[];
      const int wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
      SpgemmTable t;
      long long slots;
      if constexpr (TABLE::kShared) {
            slots = rs.slots;
            int *keys = reinterpret_cast<int *>(spgemm_smem);
            double *vals = reinterpret_cast<double *>(keys + (size_t)wpb * slots);
            t.keys = keys + (size_t)wib * slots;
            t.vals = vals + (size_t)wib * slots;
            *stage = (NUMERIC ? vals + (size_t)wpb * slots : reinterpret_cast<double *>(keys + (size_t)wpb * slots)) +
                     wib * 32;
      } else {
            const long long o = rs.toff[w];
            slots = rs.toff[w + 1] - o;
            t.keys = rs.gkeys + o;
            t.vals = NUMERIC ? rs.gvals + o : nullptr;
            *stage = reinterpret_cast<double *>(spgemm_smem) + wib * 32;
      }
      t.mask = (unsigned)(slots - 1);
      t.shift = 32 - spgemm_log2((unsigned long long)slots);
      return t;
}

// One warp per row of A: P[r] = the row's products.
template <typename OffA, typename OffB>
__global__ void spgemm_count_kernel(const OffA *__restrict__ irp_a, const int *__restrict__ ja_a, long long M,
                                    const OffB *__restrict__ irp_b, long long *__restrict__ P) {
      const int lane = threadIdx.x & 31;
      const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
      for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < M; r += warps) {
            long long s = 0;
            const long long k1 = (long long)irp_a[r + 1];
            for (long long k = (long long)irp_a[r] + lane; k < k1; k += 32) {
                  const int c = ja_a[k];
                  s += (long long)irp_b[c + 1] - (long long)irp_b[c];
            }
#pragma unroll
            for (int d = 16; d; d >>= 1)
                  s += __shfl_xor_sync(0xffffffffu, s, d);
            if (lane == 0)
                  P[r] = s;
      }
}

// Symbolic pass over the launch's rows: count[r] = distinct columns of C's row r, and their sum
// over the launch's rows added to *total (64-bit, one atomic per warp).
template <typename TABLE, typename OffA, typename OffB>
__global__ void spgemm_symbolic_kernel(const OffA *__restrict__ irp_a, const int *__restrict__ ja_a,
                                       const OffB *__restrict__ irp_b, const int *__restrict__ ja_b,
                                       SpgemmRows rs, int *__restrict__ count,
                                       unsigned long long *__restrict__ total) {
      const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
      long long sum = 0;
      for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < rs.n; w += warps) {
            double *stage;
            const SpgemmTable t = spgemm_table<TABLE, false>(rs, w, &stage);
            const int r = rs.rows[w];
            const int n = spgemm_row<false>(irp_a, ja_a, nullptr, irp_b, ja_b, nullptr, r, t, stage);
            if ((threadIdx.x & 31) == 0)
                  count[r] = n;
            sum += n;
            __syncwarp();
      }
      if ((threadIdx.x & 31) == 0 && sum)
            atomicAdd(total, (unsigned long long)sum);
}

// Numeric pass over the launch's rows: C's row r, its columns in slot order, goes to
// [irp_c[r], irp_c[r + 1]) of (t_ja, t_as).
template <typename TABLE, typename OffA, typename OffB>
__global__ void spgemm_numeric_kernel(const OffA *__restrict__ irp_a, const int *__restrict__ ja_a,
                                      const double *__restrict__ as_a, const OffB *__restrict__ irp_b,
                                      const int *__restrict__ ja_b, const double *__restrict__ as_b,
                                      SpgemmRows rs, const void *__restrict__ irp_c, bool wide_c,
                                      int *__restrict__ t_ja, double *__restrict__ t_as) {
      const int lane = threadIdx.x & 31;
      const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
      for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < rs.n; w += warps) {
            double *stage;
            const SpgemmTable t = spgemm_table<TABLE, true>(rs, w, &stage);
            const int r = rs.rows[w];
            spgemm_row<true>(irp_a, ja_a, as_a, irp_b, ja_b, as_b, r, t, stage);
            long long o = wide_c ? static_cast<const long long *>(irp_c)[r] : static_cast<const int *>(irp_c)[r];
            for (unsigned s0 = 0; s0 <= t.mask; s0 += 32) {
                  const int k = t.keys[s0 + lane];
                  const unsigned occ = __ballot_sync(0xffffffffu, k != kSpgemmEmpty);
                  if (k != kSpgemmEmpty) {
                        const long long d = o + __popc(occ & ((1u << lane) - 1));
                        t_ja[d] = k;
                        t_as[d] = t.vals[s0 + lane];
                  }
                  o += __popc(occ);
            }
            __syncwarp();
      }
}

} // namespace b200
