// hll_kernels.cuh -- FP64 HLL (hacked ELLPACK, hack = 32) y = A*x for sm_100a.
//
// Device format (one per matrix, built on upload or on the GPU from CSR):
//   hoff[h]   slot offset of hack h, hoff[h+1]-hoff[h] = 32 * width_h
//   ja, as    column-major per hack with a FIXED stride of 32 rows:
//             slot(h, i, j) = hoff[h] + j*32 + i      (i = row in hack)
//   pads      as = 0.0, ja = previous valid column of the row (0 if none),
//             i.e. the branch-free convention of the reference upload
//             (src/cuda_hll.cu:173-195); rows past M in the last hack are
//             all pads.
// Every hack therefore starts on a 256-byte (values) / 128-byte (indices)
// boundary and a warp reads whole 256-byte lines.
//
// Kernels (reference counterparts: src/cuda_hll.cu:19-152):
//   hll_warp_kernel       warp per hack, lane = row, 64-bit value and 32-bit
//                         index loads.
//   hll_stream_kernel     persistent CTAs; groups of consecutive hacks are
//                         staged in shared memory by cp.async.bulk (TMA)
//                         through an mbarrier ring; warp per hack, lane = row.
#pragma once

#include "common.cuh"

namespace b200 {

template <int EPI>
__global__ void __launch_bounds__(1024)
    hll_warp_kernel(const long long *__restrict__ hoff, const int *__restrict__ ja,
                    const double *__restrict__ as, long long hack0, long long n_hacks, long long M,
                    const double *__restrict__ x, double *__restrict__ y, EpiArgs epi) {
      static_assert(EPI == EPI_PLAIN || EPI == EPI_FUSED, "HLL epilogues");
      const long long wslot = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      const long long h = hack0 + wslot;
      if (h >= n_hacks)
            return; // whole warp
      double dot_acc = 0.0;
      const int lane = threadIdx.x & 31;
      const long long base = hoff[h];
      const int width = (int)((hoff[h + 1] - base) >> 5);
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      const double *has = as + base;
      const int *hja = ja + base;
      const long long row_base = h * kHack;

      constexpr int U = 4;
      double acc0 = 0.0, acc1 = 0.0;
      for (int j = 0; j < width; j += U) {
            double a[U], xv[U];
            int c[U];
            bool okm[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const int s = (j + u) * 32 + lane;
                  const bool ok = j + u < width;
                  okm[u] = ok;
                  a[u] = ok ? ld_stream_f64(has + s, pol_s) : 0.0;
                  c[u] = ok ? ld_stream_s32(hja + s, pol_s) : 0;
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
      const double acc = acc0 + acc1;
      if (row_base + lane < M)
            store_y<EPI>(y, row_base + lane, acc, epi, dot_acc);
      epi_finish_warp<EPI>(epi, dot_acc, wslot);
}

// ------------------------------------------------------------------------
// TMA-staged hack groups.  Plan (host): tile t = hacks [tile_h[t], tile_h[t+1])
// with at most WARPS hacks and at most CAP slots in total.  A single hack
// wider than CAP slots forms its own tile and is read straight from global
// memory by all warps of the CTA (slot columns dealt round-robin to warps).
// ------------------------------------------------------------------------
template <int WARPS, int STAGES, int CAP>
__global__ void __launch_bounds__(WARPS * 32)
    hll_stream_kernel(const long long *__restrict__ hoff, const int *__restrict__ ja,
                      const double *__restrict__ as, const int *__restrict__ tile_h, int n_tiles,
                      long long M, const double *__restrict__ x, double *__restrict__ y) {
      const EpiArgs epi{};
      double dot_acc = 0.0;
      extern __shared__ __align__(128) unsigned char smem_raw[];
      double *s_as = reinterpret_cast<double *>(smem_raw);
      int *s_ja = reinterpret_cast<int *>(smem_raw + (size_t)STAGES * CAP * 8);
      uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)STAGES * CAP * 12);
      __shared__ double big_part[WARPS][32];

      const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();

      if (tid == 0) {
            for (int s = 0; s < STAGES; ++s)
                  mbar_init(&bars[s], 1);
            mbar_fence_init();
      }
      __syncthreads();

      const int first = blockIdx.x, stride = gridDim.x;

      auto issue = [&](int t, int stage) {
            const long long s0 = hoff[tile_h[t]], s1 = hoff[tile_h[t + 1]];
            const long long cnt = s1 - s0;
            if (cnt > 0 && cnt <= CAP) {
                  mbar_expect_tx(&bars[stage], (uint32_t)(cnt * 12));
                  bulk_g2s(s_as + (size_t)stage * CAP, as + s0, (uint32_t)(cnt * 8), &bars[stage],
                           pol_s);
                  bulk_g2s(s_ja + (size_t)stage * CAP, ja + s0, (uint32_t)(cnt * 4), &bars[stage],
                           pol_s);
            } else {
                  mbar_expect_tx(&bars[stage], 0);
            }
      };

      if (tid == 0) {
            int t = first;
            for (int s = 0; s < STAGES && t < n_tiles; ++s, t += stride)
                  issue(t, s);
      }

      int it = 0;
      for (int t = first; t < n_tiles; t += stride, ++it) {
            const int stage = it % STAGES;
            const uint32_t parity = (uint32_t)(it / STAGES) & 1u;
            const int h0 = tile_h[t], h1 = tile_h[t + 1];
            const long long s0 = hoff[h0];
            const long long cnt = hoff[h1] - s0;
            // this warp's hack (if any): offsets fetched before the wait
            const int h = h0 + warp;
            long long hb = 0;
            int width = 0;
            if (h < h1) {
                  hb = hoff[h];
                  width = (int)((hoff[h + 1] - hb) >> 5);
            }
            mbar_wait(&bars[stage], parity);

            if (cnt <= CAP) {
                  if (h < h1) {
                        const double *tas = s_as + (size_t)stage * CAP + (hb - s0);
                        const int *tja = s_ja + (size_t)stage * CAP + (hb - s0);
                        constexpr int U = 8;
                        double acc0 = 0.0, acc1 = 0.0;
                        for (int j = 0; j < width; j += U) {
                              double a[U], xv[U];
                              int c[U];
                              bool okm[U];
#pragma unroll
                              for (int u = 0; u < U; ++u) {
                                    const bool ok = j + u < width;
                                    okm[u] = ok;
                                    c[u] = ok ? tja[(j + u) * 32 + lane] : 0;
                                    a[u] = ok ? tas[(j + u) * 32 + lane] : 0.0;
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
                        const double acc = acc0 + acc1;
                        const long long r = (long long)h * kHack + lane;
                        if (r < M)
                              store_y<EPI_PLAIN>(y, r, acc, epi, dot_acc);
                  }
            } else {
                  // one oversized hack: all warps share its slot columns
                  const int bw = (int)(cnt >> 5);
                  double acc = 0.0;
#pragma unroll 4
                  for (int j = warp; j < bw; j += WARPS) {
                        const long long s = s0 + (long long)j * 32 + lane;
                        acc = fma(ld_stream_f64(as + s, pol_s),
                                  ld_x(x + ld_stream_s32(ja + s, pol_s), pol_x), acc);
                  }
                  big_part[warp][lane] = acc;
                  __syncthreads();
                  if (warp == 0) {
                        double v = 0.0;
#pragma unroll
                        for (int w = 0; w < WARPS; ++w)
                              v += big_part[w][lane];
                        const long long r = (long long)h0 * kHack + lane;
                        if (r < M)
                              store_y<EPI_PLAIN>(y, r, v, epi, dot_acc);
                  }
            }
            __syncthreads();
            if (tid == 0) {
                  const int tn = t + STAGES * stride;
                  if (tn < n_tiles)
                        issue(tn, stage);
            }
      }
}

// ------------------------------------------------------------------------
// Narrow hacks (5-point stencils: width 5, BASELINE configs[0]).  A warp that owns ONE 2 KB hack
// lives through a chain of dependent loads -- hoff -> values/indices (two batches) -> x -> y, each
// a DRAM round trip (~1.1 us) while the matrix is cold -- and the SM's 64 warps only have 2 KB
// each to hide it with: 3.3 waves x 5.5 us = the 20 us measured on the L2-flushed 80 MB matrix
// (59 %, whatever the lane mapping or group size; profiles/r2_kbench_c1_*.txt, r2_c1_ncu_summary.md).
// Here every warp is persistent and runs its OWN software pipeline: lane 0 fetches the values and
// indices of the warp's next hacks with bulk copies into a private ring of STAGES shared-memory
// buffers (one mbarrier per stage, no CTA-wide synchronisation anywhere), the offsets of the hack
// after those are already in registers, and the only latency left on the critical path of a hack
// is its gather of x.  Hacks are dealt round-robin (warp w: w, w + W, ...), so neighbouring warps
// stream neighbouring memory.
// One hack of exactly W slot columns out of a shared-memory stage, lane = row.
template <int W>
__device__ __forceinline__ double hll_pipe_cols(const double *__restrict__ tas, const int *__restrict__ tja,
                                                int lane, const double *__restrict__ x, uint64_t pol_x) {
      double a[W], xv[W];
      int c[W];
#pragma unroll
      for (int u = 0; u < W; ++u) {
            c[u] = tja[u * 32 + lane];
            a[u] = tas[u * 32 + lane];
      }
#pragma unroll
      for (int u = 0; u < W; ++u)
            xv[u] = ld_x(x + c[u], pol_x);
      double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
      for (int u = 0; u < W; ++u) { // even slot columns into acc0, odd into acc1, like hll_warp_kernel
            if (u & 1)
                  acc1 = fma(a[u], xv[u], acc1);
            else
                  acc0 = fma(a[u], xv[u], acc0);
      }
      return acc0 + acc1;
}

template <int STAGES, int EPI>
__global__ void __launch_bounds__(256)
    hll_pipe_kernel(const long long *__restrict__ hoff, const int *__restrict__ ja,
                    const double *__restrict__ as, long long hack0, long long hack1, int capw,
                    long long M, const double *__restrict__ x, double *__restrict__ y, EpiArgs epi) {
      extern __shared__ __align__(128) unsigned char smem_raw[];
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
      unsigned char *ring = smem_raw + (size_t)warp * STAGES * capw * 12;
      uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)wpc * STAGES * capw * 12) + warp * STAGES;
      const long long W = (long long)gridDim.x * wpc;
      const long long first = hack0 + (long long)blockIdx.x * wpc + warp;
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      if (lane == 0) {
#pragma unroll
            for (int s = 0; s < STAGES; ++s)
                  mbar_init(&bars[s], 1);
            mbar_fence_init();
      }
      __syncwarp();

      long long b0[STAGES] = {0}, b1[STAGES] = {0}; // slot range of the hack in flight in each stage
      auto fetch = [&](int s) {         // lane 0: start the copies of stage s (b0/b1 already loaded)
            if (lane == 0) {
                  const long long cnt = b1[s] - b0[s];
                  mbar_expect_tx(&bars[s], (uint32_t)(cnt * 12));
                  if (cnt > 0) {
                        bulk_g2s(ring + (size_t)s * capw * 12, as + b0[s], (uint32_t)(cnt * 8), &bars[s], pol_s);
                        bulk_g2s(ring + (size_t)s * capw * 12 + (size_t)capw * 8, ja + b0[s], (uint32_t)(cnt * 4),
                                 &bars[s], pol_s);
                  }
            }
      };
#pragma unroll
      for (int s = 0; s < STAGES; ++s) {
            const long long h = first + s * W;
            b0[s] = b1[s] = 0;
            if (h < hack1) {
                  b0[s] = hoff[h], b1[s] = hoff[h + 1];
                  fetch(s);
            }
      }
      for (long long i = 0;; i += STAGES) {
            const uint32_t parity = (uint32_t)(i / STAGES) & 1u;
#pragma unroll
            for (int s = 0; s < STAGES; ++s) {
                  const long long h = first + (i + s) * W;
                  if (h >= hack1)
                        return; // whole warp
                  // offsets of the hack that takes this stage next: on their way while this one is computed
                  const long long hn = h + STAGES * W;
                  long long n0 = 0, n1 = 0;
                  if (hn < hack1)
                        n0 = hoff[hn], n1 = hoff[hn + 1];
                  const int width = (int)((b1[s] - b0[s]) >> 5);
                  mbar_wait(&bars[s], parity);
                  const double *tas = reinterpret_cast<const double *>(ring + (size_t)s * capw * 12);
                  const int *tja = reinterpret_cast<const int *>(ring + (size_t)s * capw * 12 + (size_t)capw * 8);
                  // exactly `width` slot columns (<= 8 by the launcher's choice): no predicated spares
                  double acc;
                  switch (width) {
                  case 0: acc = 0.0; break;
                  case 1: acc = hll_pipe_cols<1>(tas, tja, lane, x, pol_x); break;
                  case 2: acc = hll_pipe_cols<2>(tas, tja, lane, x, pol_x); break;
                  case 3: acc = hll_pipe_cols<3>(tas, tja, lane, x, pol_x); break;
                  case 4: acc = hll_pipe_cols<4>(tas, tja, lane, x, pol_x); break;
                  case 5: acc = hll_pipe_cols<5>(tas, tja, lane, x, pol_x); break;
                  case 6: acc = hll_pipe_cols<6>(tas, tja, lane, x, pol_x); break;
                  case 7: acc = hll_pipe_cols<7>(tas, tja, lane, x, pol_x); break;
                  default: acc = hll_pipe_cols<8>(tas, tja, lane, x, pol_x); break;
                  }
                  __syncwarp(); // every lane has read the stage: it may be overwritten
                  b0[s] = n0, b1[s] = n1;
                  if (hn < hack1)
                        fetch(s);
                  double dot_acc = 0.0;
                  const long long r = h * kHack + lane;
                  if (r < M)
                        store_y<EPI>(y, r, acc, epi, dot_acc);
                  epi_finish_warp<EPI>(epi, dot_acc, h - hack0);
            }
      }
}

// ------------------------------------------------------------------------
// Device-side format conversion.
// ------------------------------------------------------------------------

// width[h] = longest row of hack h (CSR input).
template <typename OffT>
__global__ void hll_width_kernel(const OffT *__restrict__ irp, long long M, long long n_hacks,
                                 int *__restrict__ width) {
      const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (h >= n_hacks)
            return;
      const int lane = threadIdx.x & 31;
      const long long r = h * kHack + lane;
      int len = r < M ? (int)(irp[r + 1] - irp[r]) : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
            len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
      if (lane == 0)
            width[h] = len;
}

// CSR -> device HLL: warp per hack, lane = row; writes are coalesced
// (32 consecutive slots per step), reads walk each row.
template <typename OffT>
__global__ void hll_fill_from_csr_kernel(const OffT *__restrict__ irp, const int *__restrict__ cja,
                                         const double *__restrict__ cas, long long M,
                                         long long n_hacks, const long long *__restrict__ hoff,
                                         int *__restrict__ ja, double *__restrict__ as,
                                         int *__restrict__ rowlen) {
      const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (h >= n_hacks)
            return;
      const int lane = threadIdx.x & 31;
      const long long r = h * kHack + lane;
      const long long base = hoff[h];
      const int width = (int)((hoff[h + 1] - base) >> 5);
      OffT k0 = 0;
      int len = 0;
      if (r < M) {
            k0 = irp[r];
            len = (int)(irp[r + 1] - k0);
      }
      rowlen[r] = len; // allocated for n_hacks * 32 rows
      int last_col = 0;
      for (int j = 0; j < width; ++j) {
            double a = 0.0;
            if (j < len) {
                  a = cas[k0 + j];
                  last_col = cja[k0 + j];
            }
            as[base + (long long)j * 32 + lane] = a;
            ja[base + (long long)j * 32 + lane] = last_col;
      }
}

// Host HLL (either layout, pads = -1) staged on the device as a flat copy
// -> device HLL.  `src_off[h]` is the offset of hack h in the staged arrays,
// rows[h] its row count (stride of the column-major host layout).
__global__ void hll_fill_from_host_layout_kernel(const long long *__restrict__ src_off,
                                                 const int *__restrict__ src_ja,
                                                 const double *__restrict__ src_as,
                                                 int col_major, long long M, long long n_hacks,
                                                 const long long *__restrict__ hoff,
                                                 int *__restrict__ ja, double *__restrict__ as,
                                                 int *__restrict__ rowlen) {
      const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
      if (h >= n_hacks)
            return;
      const int lane = threadIdx.x & 31;
      const long long base = hoff[h];
      const int width = (int)((hoff[h + 1] - base) >> 5);
      const long long rows_left = M - h * kHack;
      const int rows = rows_left < kHack ? (int)rows_left : kHack;
      const int *sja = src_ja + src_off[h];
      const double *sas = src_as + src_off[h];
      int last_col = 0, len = 0;
      for (int j = 0; j < width; ++j) {
            double a = 0.0;
            if (lane < rows) {
                  const long long s = col_major ? (long long)j * rows + lane
                                                : (long long)lane * width + j;
                  const int c = sja[s];
                  a = sas[s];
                  if (c != -1) {
                        last_col = c;
                        len = j + 1; // the host packer fills a row left to right (src/hll.c:78-91)
                  } else {
                        a = 0.0;
                  }
            }
            as[base + (long long)j * 32 + lane] = a;
            ja[base + (long long)j * 32 + lane] = last_col;
      }
      rowlen[h * kHack + lane] = len;
}

} // namespace b200
