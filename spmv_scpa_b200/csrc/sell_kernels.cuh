// sell_kernels.cuh -- column-panelled, window-sorted sliced ELLPACK ("SELL-P") for sm_100a.
//
// New code, no reference counterpart.  It generalises the device HLL layout (hll_kernels.cuh:
// hack = slice of 32 rows, column-major with a fixed stride of 32, branch-free pads) in the two
// directions the reference formats cannot cover (SURVEY.md section 7, hard parts 2 and 3):
//
//   * column panels.  When x is larger than the L2 and the columns of a row are scattered
//     (uniform random: BASELINE configs[2]), every gather is its own DRAM sector -- measured
//     4.7 x B_min of DRAM traffic in round 1.  Here the columns are cut into K panels whose x
//     slice fits the L2; panel p is one launch that touches only x[pc[p], pc[p+1]) and adds its
//     partial row sums into y (panel 0 stores, later panels accumulate; stream order makes the
//     sum deterministic).
//   * sigma-sorted windows.  Inside each window of `sigma` consecutive rows the rows are ordered
//     by their entry count in the panel (descending, ties by row index), so the 32 rows of a
//     slice have (nearly) equal length and padding disappears even for power-law rows
//     (BASELINE configs[3]); y is written through the permutation, and stays inside the window.
//
//   * virtual rows (one panel only).  A slice is walked by ONE warp, so a 4000-entry row in a
//     slice is a millisecond of serial latency at the tail of the launch.  For ragged matrices
//     every row longer than `chunk` entries is cut into virtual rows of at most `chunk` entries;
//     slices are built over virtual rows, every warp gets at most `chunk` steps, the hub rows
//     of a power-law matrix spread over thousands of lanes, and no separate long-row kernel is
//     left.  A virtual row of an unsplit row stores y directly; the pieces of a split row store
//     partial sums that csr_combine_kernel adds in piece order (deterministic, no atomics).
//     perm then holds the DESTINATION of a lane: row >= 0, -1 = none, -2-i = partial[i].
//
// Layout, per panel p and slice s (S = ceil(M/32) slices in every panel):
//   soff[p*(S+1) + s]        slot offset of the slice; (soff[..+1] - soff[..]) / 32 = width
//   perm[(p*S + s)*32 + i]   local row of lane i, or -1 (no row: tail of the last window, or a
//                            row that is too long for a slice and handled by the CSR long-row
//                            kernels)
//   ja/as[slot + j*32 + i]   j-th entry of that row inside the panel; pads: as = 0.0,
//                            ja = previous valid column of the row in the panel, or the panel's
//                            first column when the row has none (always inside the x slice)
#pragma once

#include "common.cuh"

namespace b200 {

// One warp per slice, lane = row (the mapping of hll_warp_kernel, which measured best
// whenever the gather is the limiter).  Slices [slice0, slice0 + n) of one panel.
template <int EPI, bool VROWS = false>
__global__ void __launch_bounds__(1024)
    sell_kernel(const long long *__restrict__ soff, const int *__restrict__ perm,
                const int *__restrict__ ja, const double *__restrict__ as, long long n_slices,
                const double *__restrict__ x, double *__restrict__ y,
                double *__restrict__ partial, EpiArgs epi) {
      const long long s = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (s >= n_slices)
            return; // whole warp
      const int lane = threadIdx.x & 31;
      const long long base = soff[s];
      const int width = (int)((soff[s + 1] - base) >> 5);
      if (EPI == EPI_ACC && width == 0)
            return; // nothing to add for these rows in this panel
      const int row = perm[s * 32 + lane];
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      const double *sas = as + base;
      const int *sja = ja + base;
      constexpr int U = 4;

      double acc0 = 0.0, acc1 = 0.0;
      for (int j = 0; j < width; j += U) {
            double a[U], xv[U];
            int c[U];
            bool okm[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const int k = (j + u) * 32 + lane;
                  const bool ok = j + u < width;
                  okm[u] = ok;
                  a[u] = ok ? ld_stream_f64(sas + k, pol_s) : 0.0;
                  c[u] = ok ? ld_stream_s32(sja + k, pol_s) : 0;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                  xv[u] = okm[u] ? ld_x(x + c[u], pol_x) : 0.0;
#pragma unroll
            for (int u = 0; u < U; u += 2) {
                  acc0 = fma(a[u], xv[u], acc0);
                  acc1 = fma(a[u + 1], xv[u + 1], acc1);
            }
      }
      double dot_acc = 0.0;
      if (row >= 0)
            store_y<EPI>(y, row, acc0 + acc1, epi, dot_acc);
      else if (VROWS && row < -1)
            partial[-2 - row] = acc0 + acc1; // a piece of a split row
      epi_finish_warp<EPI>(epi, dot_acc, s);
}

// K right-hand sides at once (SURVEY 8(f)3): Y[M][K] = A X[N][K], both row-major.  The slices are
// walked exactly as in sell_kernel; every gather now returns K useful values out of the sector it
// moves, which is the one way past the gather bound of DESIGN.md section 3 for callers that
// iterate on several vectors.  EPI_PLAIN stores, EPI_ACC adds (column panels after the first);
// pieces of split rows write K partial sums each.
template <int K, int EPI, bool VROWS>
__global__ void __launch_bounds__(512)
    sell_mm_kernel(const long long *__restrict__ soff, const int *__restrict__ perm,
                   const int *__restrict__ ja, const double *__restrict__ as, long long n_slices,
                   const double *__restrict__ X, double *__restrict__ Y, double *__restrict__ partial) {
      static_assert(EPI == EPI_PLAIN || EPI == EPI_ACC, "SpMM epilogues");
      const long long s = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (s >= n_slices)
            return; // whole warp
      const int lane = threadIdx.x & 31;
      const long long base = soff[s];
      const int width = (int)((soff[s + 1] - base) >> 5);
      if (EPI == EPI_ACC && width == 0)
            return;
      const int row = perm[s * 32 + lane];
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      const double *sas = as + base;
      const int *sja = ja + base;
      constexpr int U = 4;
      double acc[K];
#pragma unroll
      for (int k = 0; k < K; ++k)
            acc[k] = 0.0;
      for (int j = 0; j < width; j += U) {
            double a[U], xv[U][K];
            int c[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const int kk = (j + u) * 32 + lane;
                  const bool ok = j + u < width;
                  a[u] = ok ? ld_stream_f64(sas + kk, pol_s) : 0.0;
                  c[u] = ok ? ld_stream_s32(sja + kk, pol_s) : -1;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                  ld_xk<K>(X, c[u], pol_x, xv[u]);
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                  for (int k = 0; k < K; ++k)
                        acc[k] = fma(a[u], xv[u][k], acc[k]);
      }
      double *out = row >= 0 ? Y + (long long)row * K : (VROWS && row < -1 ? partial + (long long)(-2 - row) * K : nullptr);
      if (out) {
#pragma unroll
            for (int k = 0; k < K; ++k)
                  out[k] = (EPI == EPI_ACC && row >= 0) ? out[k] + acc[k] : acc[k];
      }
}

// ------------------------------------------------------------------ build --
// Row sources: the resident CSR or the resident device HLL.
template <typename OffT>
struct CsrSrc {
      const OffT *irp;
      const int *ja;
      const double *as;
      __device__ __forceinline__ int len(long long r) const { return (int)(irp[r + 1] - irp[r]); }
      __device__ __forceinline__ long long at(long long r, int j) const { return (long long)irp[r] + j; }
};
struct HllSrc {
      const long long *hoff;
      const int *ja;
      const double *as;
      const int *rowlen;
      __device__ __forceinline__ int len(long long r) const { return rowlen[r]; }
      __device__ __forceinline__ long long at(long long r, int j) const {
            return hoff[r >> 5] + (long long)j * 32 + (r & 31);
      }
};

// Panel of a column: pc[] has K+1 ascending bounds, K <= 64.
struct PanelBounds {
      int K;
      int pc[65];
};
__device__ __forceinline__ int panel_of(const PanelBounds &pb, int col) {
      int p = 0;
      while (p + 1 < pb.K && col >= pb.pc[p + 1])
            ++p;
      return p;
}

// counts[p*M + r] = entries of row r whose column lies in panel p; rows longer than max_row get
// -1 in every panel (they are not part of any slice).
template <typename Src>
__global__ void sell_count_kernel(Src src, long long M, PanelBounds pb, int max_row,
                                  int *__restrict__ counts) {
      const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
      if (r >= M)
            return;
      const int len = src.len(r);
      if (len > max_row) {
            for (int p = 0; p < pb.K; ++p)
                  counts[(long long)p * M + r] = -1;
            return;
      }
      if (pb.K == 1) {
            counts[r] = len;
            return;
      }
      int cnt[64];
      for (int p = 0; p < pb.K; ++p)
            cnt[p] = 0;
      for (int j = 0; j < len; ++j)
            ++cnt[panel_of(pb, src.ja[src.at(r, j)])];
      for (int p = 0; p < pb.K; ++p)
            counts[(long long)p * M + r] = cnt[p];
}

// Fill the slices of every panel: warp per (panel, slice), lane = row perm[...].  A lane walks its
// row in storage order and keeps the entries of its panel, so the order of a row's entries inside
// a panel is the reference's CSR order.
template <typename Src>
__global__ void sell_fill_kernel(Src src, long long n_slices, PanelBounds pb,
                                 const long long *__restrict__ soff, const int *__restrict__ perm,
                                 int *__restrict__ ja, double *__restrict__ as) {
      const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (w >= n_slices * pb.K)
            return;
      const int lane = threadIdx.x & 31;
      const int p = (int)(w / n_slices);
      const long long s = w % n_slices;
      const long long base = soff[(long long)p * (n_slices + 1) + s];
      const int width = (int)((soff[(long long)p * (n_slices + 1) + s + 1] - base) >> 5);
      const int row = perm[((long long)p * n_slices + s) * 32 + lane];
      const int lo = pb.pc[p], hi = pb.pc[p + 1];
      const int len = row >= 0 ? src.len(row) : 0;
      int last_col = lo, j = 0, out = 0;
      for (; out < width; ++out) {
            double a = 0.0;
            while (j < len) {
                  const long long k = src.at(row, j);
                  const int c = src.ja[k];
                  ++j;
                  if (pb.K == 1 || (c >= lo && c < hi)) {
                        a = src.as[k];
                        last_col = c;
                        break;
                  }
            }
            as[base + (long long)out * 32 + lane] = a;
            ja[base + (long long)out * 32 + lane] = last_col;
      }
}

// Virtual-row fill (one panel): lane = virtual row perm_v[...] = entries [j0, j0 + len) of row
// vr_row[v], len = min(chunk, row length - j0).
template <typename Src>
__global__ void sell_fill_vrow_kernel(Src src, long long n_slices, const long long *__restrict__ soff,
                                      const int *__restrict__ perm_v, const int *__restrict__ vr_row,
                                      const int *__restrict__ vr_j0, int chunk, int *__restrict__ ja,
                                      double *__restrict__ as) {
      const long long s = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (s >= n_slices)
            return;
      const int lane = threadIdx.x & 31;
      const long long base = soff[s];
      const int width = (int)((soff[s + 1] - base) >> 5);
      const int v = perm_v[s * 32 + lane];
      long long row = 0;
      int j0 = 0, len = 0;
      if (v >= 0) {
            row = vr_row[v];
            j0 = vr_j0[v];
            len = min(chunk, src.len(row) - j0);
      }
      int last_col = 0;
      for (int out = 0; out < width; ++out) {
            double a = 0.0;
            if (out < len) {
                  const long long k = src.at(row, j0 + out);
                  a = src.as[k];
                  last_col = src.ja[k];
            }
            as[base + (long long)out * 32 + lane] = a;
            ja[base + (long long)out * 32 + lane] = last_col;
      }
}

// Largest |first column - last column| distance statistics are taken on the host from a sample;
// this kernel only extracts, for `n` sampled row blocks of `block` rows, the smallest and largest
// column index each block touches (is the gather local, or scattered over all of x?).
template <typename Src>
__global__ void col_extent_kernel(Src src, long long M, long long block, long long stride, int n,
                                  int *__restrict__ lo_out, int *__restrict__ hi_out) {
      const int b = blockIdx.x;
      if (b >= n)
            return;
      const long long r0 = (long long)b * stride;
      int lo = 0x7fffffff, hi = -1;
      for (long long r = r0 + threadIdx.x; r < r0 + block && r < M; r += blockDim.x) {
            const int len = src.len(r);
            for (int j = 0; j < len; ++j) {
                  const int c = src.ja[src.at(r, j)];
                  lo = min(lo, c);
                  hi = max(hi, c);
            }
      }
      __shared__ int s_lo[32], s_hi[32];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
      }
      if ((threadIdx.x & 31) == 0)
            s_lo[threadIdx.x >> 5] = lo, s_hi[threadIdx.x >> 5] = hi;
      __syncthreads();
      if (threadIdx.x == 0) {
            for (unsigned w = 1; w < (blockDim.x >> 5); ++w)
                  lo = min(lo, s_lo[w]), hi = max(hi, s_hi[w]);
            lo_out[b] = lo;
            hi_out[b] = hi;
      }
}

} // namespace b200
