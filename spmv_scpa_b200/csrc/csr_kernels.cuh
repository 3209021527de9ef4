// csr_kernels.cuh -- FP64 CSR y = A*x kernels for sm_100a.
//
// New designs; the reference kernels they stand in for are
// src/cuda_csr.cu:19-178 (thread / warp / half-warp / block per row, plain
// LDG).  Families here:
//   csr_vec_kernel<LPR>     LPR = 1,2,4,...,32 lanes cooperate on one row
//                           (LPR=1 is thread-per-row, LPR=32 warp-per-row),
//                           shuffle reduction; matrix streams bypass L1.
//   csr_block_row_kernel    one CTA per row, shuffle + shared-memory reduce.
//   csr_split_kernel        rows too long for one CTA are cut into chunks,
//   csr_combine_kernel      partial sums combined deterministically.
//   csr_stream_kernel       persistent CTAs; the value/index streams of a
//                           tile of consecutive rows are staged in shared
//                           memory by cp.async.bulk (TMA) through an
//                           mbarrier ring, then each thread walks its own row
//                           in shared memory, so the x gather of a warp hits
//                           neighbouring columns (ELL-like access on CSR).
// Every kernel takes the matrix as (irp, ja, as) with OffT row offsets
// (int32, or int64 for shards beyond 2^31 entries) and column indices
// already relative to the local x slice.
#pragma once

#include "common.cuh"

namespace b200 {

// ------------------------------------------------------------------------
// LPR lanes per row.  `rowlist` == nullptr: rows [row0, row0+nrows) in order;
// otherwise rows rowlist[0..nrows).  Rows longer than `max_len` are skipped
// (they belong to another bin's launch); max_len < 0 disables the test.
// ------------------------------------------------------------------------
template <int LPR, typename OffT, int EPI>
__global__ void __launch_bounds__(1024)
    csr_vec_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                   const double *__restrict__ as, long long row0, long long nrows,
                   const int *__restrict__ rowlist, long long max_len,
                   const double *__restrict__ x, double *__restrict__ y, EpiArgs epi) {
      static_assert(EPI == EPI_PLAIN || EPI == EPI_PUSH, "direct kernels: plain or push epilogue");
      const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
      const long long g = gid / LPR;
      const int sub = (int)(gid % LPR);
      // whole groups leave together, so the shuffles below stay convergent
      if (g >= nrows)
            return;
      const long long row = rowlist ? (long long)rowlist[g] : row0 + g;
      const OffT s = irp[row], e = irp[row + 1];
      if (max_len >= 0 && (long long)(e - s) > max_len)
            return;

      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      // Batches of U entries per lane: all index/value loads of a batch are
      // issued before the first gather, all gathers before the first FMA, so
      // U independent memory round trips overlap instead of chaining.
      constexpr int U = LPR == 32 ? 8 : 4; // a whole warp on a long row: deeper batches
      double acc0 = 0.0, acc1 = 0.0;
      for (OffT k = s + sub; k < e; k += LPR * U) {
            double a[U], xv[U];
            int c[U];
            bool okm[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const OffT kk = k + u * LPR;
                  const bool ok = kk < e;
                  okm[u] = ok;
                  if (LPR >= 16) {
                        a[u] = ok ? ld_stream_f64(as + kk, pol_s) : 0.0;
                        c[u] = ok ? ld_stream_s32(ja + kk, pol_s) : 0;
                  } else {
                        a[u] = ok ? ld_stream_l1_f64(as + kk, pol_s) : 0.0;
                        c[u] = ok ? ld_stream_l1_s32(ja + kk, pol_s) : 0;
                  }
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
      double acc = acc0 + acc1;
      acc = group_sum<LPR>(acc);
      double unused = 0.0;
      if (sub == 0)
            store_y<EPI>(y, row, acc, epi, unused);
}

// Strided partial dot product of one long row: entries first, first+step, ...
// below `end`, in batches of 4 independent load -> gather -> FMA chains.
template <typename OffT>
__device__ __forceinline__ double long_row_partial(const double *__restrict__ as,
                                                   const int *__restrict__ ja,
                                                   const double *__restrict__ x, OffT first,
                                                   OffT end, int step, uint64_t pol_s,
                                                   uint64_t pol_x) {
      constexpr int U = 4;
      double acc0 = 0.0, acc1 = 0.0;
      for (OffT k = first; k < end; k += (OffT)step * U) {
            double a[U], xv[U];
            int c[U];
            bool okm[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const OffT kk = k + (OffT)u * step;
                  const bool ok = kk < end;
                  okm[u] = ok;
                  a[u] = ok ? ld_stream_f64(as + kk, pol_s) : 0.0;
                  c[u] = ok ? ld_stream_s32(ja + kk, pol_s) : 0;
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
      return acc0 + acc1;
}

// ------------------------------------------------------------------------
// One CTA per row (blockDim.x = 32*wpb).  Row = rowlist[blockIdx.x] or
// row0 + blockIdx.x.
// ------------------------------------------------------------------------
template <typename OffT, int EPI>
__global__ void __launch_bounds__(1024)
    csr_block_row_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                         const double *__restrict__ as, long long row0,
                         const int *__restrict__ rowlist, const double *__restrict__ x,
                         double *__restrict__ y, EpiArgs epi) {
      __shared__ double warp_part[32];
      const long long row = rowlist ? (long long)rowlist[blockIdx.x] : row0 + blockIdx.x;
      const OffT s = irp[row], e = irp[row + 1];
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();

      double acc = long_row_partial<OffT>(as, ja, x, s + threadIdx.x, e, blockDim.x, pol_s, pol_x);
      acc = group_sum<32>(acc);

      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      const int nwarps = blockDim.x >> 5;
      if (lane == 0)
            warp_part[warp] = acc;
      __syncthreads();
      if (warp == 0) {
            double v = lane < nwarps ? warp_part[lane] : 0.0;
            v = group_sum<32>(v);
            double unused = 0.0;
            if (lane == 0)
                  store_y<EPI>(y, row, v, epi, unused);
      }
}

// ------------------------------------------------------------------------
// Very long rows: chunk c covers entries [chunk_k[c], chunk_k[c+1]) of one
// row and produces partial[c]; csr_combine_kernel then adds the partials of
// each split row in chunk order (deterministic, no atomics).
// ------------------------------------------------------------------------
static __global__ void __launch_bounds__(1024)
    csr_split_kernel(const long long *__restrict__ chunk_k0, const long long *__restrict__ chunk_k1,
                     const int *__restrict__ ja, const double *__restrict__ as,
                     const double *__restrict__ x, double *__restrict__ partial) {
      __shared__ double warp_part[32];
      const long long s = chunk_k0[blockIdx.x], e = chunk_k1[blockIdx.x];
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      double acc =
          long_row_partial<long long>(as, ja, x, s + threadIdx.x, e, blockDim.x, pol_s, pol_x);
      acc = group_sum<32>(acc);
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      if (lane == 0)
            warp_part[warp] = acc;
      __syncthreads();
      if (warp == 0) {
            double v = lane < (int)(blockDim.x >> 5) ? warp_part[lane] : 0.0;
            v = group_sum<32>(v);
            if (lane == 0)
                  partial[blockIdx.x] = v;
      }
}

template <int EPI>
__global__ void csr_combine_kernel(const int *__restrict__ split_row,
                                   const int *__restrict__ split_first_chunk, int n_split,
                                   const double *__restrict__ partial, double *__restrict__ y,
                                   EpiArgs epi) {
      const int i = blockIdx.x * blockDim.x + threadIdx.x;
      if (i >= n_split)
            return;
      double acc = 0.0;
      for (int c = split_first_chunk[i]; c < split_first_chunk[i + 1]; ++c)
            acc += partial[c];
      double unused = 0.0;
      store_y<EPI>(y, split_row[i], acc, epi, unused);
}

// ------------------------------------------------------------------------
// TMA-staged row tiles.
//
// Plan (host): tile t = rows [tile_row[t], tile_row[t+1]) with at most
// MAXROWS rows and (after rounding the entry range out to multiples of 4)
// at most CAP entries; tile_k[t] = irp[tile_row[t]].  A tile that is a single
// row with more than CAP entries is skipped here (long-row launch).
//
// Kernel: persistent CTAs, CTA b owns tiles b, b+G, b+2G, ...  A ring of
// STAGES shared-memory buffers, each filled by two cp.async.bulk copies
// (values, indices) that complete on the stage's "full" mbarrier.
//   WS = false  every thread computes; thread 0 also issues the copies; one
//               __syncthreads per tile hands the stage back.
//   WS = true   warp-specialised: one extra producer warp issues copies as
//               soon as a stage's "empty" mbarrier (one arrival per consumer
//               warp) completes; consumer warps never meet at a CTA barrier,
//               so they drift apart and overlap each other's gather latency.
//
// Compute: LPR lanes per row (LPR = 1: thread per row).  Rows of a warp are
// neighbours, so for banded matrices the 32 x-gathers of one step fall in a
// few contiguous sectors (ELL-like access on CSR).  For even row lengths the
// walk through the row is rotated by the row's index so lanes start in
// different shared-memory banks.
//
// Column codes (CODES = true, row-tile mode only): in place of the int32
// index stream a tile brings one block, built once per plan by
// stream_codes_kernel: a uint8 code per staged entry, in the positions of
// the value stage, padded to 16 bytes, then the tile's dictionary of
// distinct column offsets d = col - row (int32, ascending, at most
// kCodeDict, padded to 16 bytes).  The column of an entry is row +
// dict[code], exactly the stored index, so results do not change; a banded
// or stencil tile streams 9 bytes per entry instead of 12.
// ------------------------------------------------------------------------
constexpr int kCodeDict = 256; // distinct column offsets a coded tile may hold

__host__ __device__ constexpr long long round16(long long n) { return (n + 15) & ~15ll; }

template <int THREADS, int LPR, int STAGES, int CAP, int PASSES, bool WS, bool SPLIT = false,
          bool CODES = false>
struct StreamCfg {
      static_assert(!(SPLIT && CODES), "column codes exist for the row-tile mode only");
      static constexpr int kConsumers = THREADS;
      static constexpr int kThreads = THREADS + (WS ? 32 : 0);
      static constexpr int kRowsPerPass = THREADS / LPR;
      static constexpr int kMaxRows = kRowsPerPass * PASSES;
      static constexpr int kCap = CAP; // entries per stage (multiple of 16)
      // bytes of the index part of a stage: int32 columns, or a code block
      static constexpr int kIdxBytes = CODES ? CAP + kCodeDict * 4 : CAP * 4;
      static constexpr int kQueue = CAP / 32 + 8; // rows longer than 32 entries per tile
      static constexpr int kIrpSlots = kMaxRows + 8; // staged row offsets per stage (SPLIT)
      template <typename OffT>
      static constexpr size_t smem() {
            return (size_t)STAGES * (CAP * 8 + kIdxBytes) + 2 * STAGES * 8 + 16 +
                   (SPLIT ? (size_t)(kQueue + 4) * 4 + 16 + (size_t)STAGES * kIrpSlots * sizeof(OffT) : 0);
      }
};

// All rows of one staged tile.  `gi` = row slot of this thread, `sub` = lane
// within the row group.  Columns come from `tja`, or with CODES from
// row + tdict[tcode[...]].
template <int LPR, int RPP, int PASSES, int EPI, bool CODES, typename OffT>
__device__ __forceinline__ void stream_tile_rows(const OffT *__restrict__ irp,
                                                 const double *__restrict__ tas,
                                                 const int *__restrict__ tja,
                                                 const unsigned char *__restrict__ tcode,
                                                 const int *__restrict__ tdict, int r0, int r1,
                                                 long long kbase, int gi, int sub, long long ks,
                                                 long long ke, const double *__restrict__ x,
                                                 double *__restrict__ y, uint64_t pol_x,
                                                 const EpiArgs &epi, double &dot_acc) {
      int row = r0 + gi;
#pragma unroll 1
      for (int p = 0; p < PASSES; ++p) {
            if (p > 0) {
                  if (r0 + p * RPP >= r1)
                        break; // uniform over the CTA
                  row = r0 + p * RPP + gi;
                  if (row < r1) {
                        ks = (long long)irp[row] - kbase;
                        ke = (long long)irp[row + 1] - kbase;
                  }
            }
            const int len = row < r1 ? (int)(ke - ks) : 0;
            const int base = (int)ks;
            // Even row lengths put the rows of a warp in the same banks:
            // start each row's walk at a different entry (two contiguous
            // runs [start,len) + [0,start)).
            int start = 0;
            if (LPR == 1 && len > 1 && (len & 1) == 0)
                  start = gi % len;
            constexpr int U = 8;
            double acc0 = 0.0, acc1 = 0.0;
            auto walk = [&](int from, int to) {
                  for (int j = from + sub; j < to; j += LPR * U) {
                        double a[U], xv[U];
                        int c[U];
                        bool okm[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                              const int jj = j + u * LPR;
                              const bool ok = jj < to;
                              okm[u] = ok;
                              // (codes: the byte now, its dictionary entry in a second sweep)
                              c[u] = ok ? (CODES ? (int)tcode[base + jj] : tja[base + jj]) : 0;
                              a[u] = ok ? tas[base + jj] : 0.0;
                        }
                        if (CODES) {
#pragma unroll
                              for (int u = 0; u < U; ++u)
                                    c[u] = row + tdict[c[u]];
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
            };
            walk(start, len);
            if (start)
                  walk(0, start);
            double acc = acc0 + acc1;
            if (LPR > 1)
                  acc = group_sum<LPR>(acc);
            if (sub == 0 && row < r1)
                  store_y<EPI>(y, row, acc, epi, dot_acc);
      }
}

// Irregular tiles (power-law matrices): rows of wildly different lengths share
// a tile, so the work is split by ENTRY, not by row.
//   phase 1  every consumer thread strides over the staged entries and
//            overwrites each value with value * x[col]   (balanced, gathers
//            batched 4 deep);
//   phase 2  thread per row adds up its (short) run of products; rows longer
//            than 32 entries are queued in shared memory instead;
//   phase 3  warps drain the queue, one warp per long row, shuffle reduction.
// Named barrier 1 (consumer threads only) separates the phases.
template <int THREADS, int PASSES, int CAP, int EPI, typename OffT>
__device__ __forceinline__ void stream_tile_products(const OffT *s_irp, double *tas, const int *tja,
                                                     int r0, int r1, int r0a, long long kbase,
                                                     int cnt, int tid,
                                                     const double *__restrict__ x,
                                                     double *__restrict__ y, uint64_t pol_x,
                                                     const EpiArgs &epi, double &dot_acc,
                                                     int *s_queue, int *s_queue_n,
                                                     int *s_queue_n_other) {
      // batches of up to 8 entries per thread (deeper batches measured slower:
      // profiles/r1_c4_*): loads, then gathers, then products back in place
      constexpr int PER = (CAP + THREADS - 1) / THREADS;
      constexpr int U = PER < 8 ? PER : 8;
      for (int j = tid; j < cnt; j += THREADS * U) {
            double a[U], xv[U];
            int c[U];
            bool okm[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const int jj = j + u * THREADS;
                  okm[u] = jj < cnt;
                  c[u] = okm[u] ? tja[jj] : 0;
                  a[u] = okm[u] ? tas[jj] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                  xv[u] = okm[u] ? ld_x(x + c[u], pol_x) : 0.0;
#pragma unroll
            for (int u = 0; u < U; ++u)
                  if (okm[u])
                        tas[j + u * THREADS] = a[u] * xv[u];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(THREADS) : "memory");
      // The long-row counter alternates between two words by tile parity.  Every thread is past
      // the previous tile's phase 3 (its last reader) once it has crossed the barrier above, and
      // the next tile's phase 2 (its next writer) lies behind that tile's first barrier, which
      // this thread reaches only after this store: resetting it here races with nobody.
      if (tid == 0)
            *s_queue_n_other = 0;

#pragma unroll 1
      for (int p = 0; p < PASSES; ++p) {
            const int row = r0 + p * THREADS + tid;
            if (r0 + p * THREADS >= r1)
                  break;
            if (row < r1) {
                  const int s = (int)((long long)s_irp[row - r0a] - kbase);
                  const int e = (int)((long long)s_irp[row - r0a + 1] - kbase);
                  if (e - s <= 32) {
                        // four independent shared-memory loads per step
                        double acc0 = 0.0, acc1 = 0.0;
                        for (int j = s; j < e; j += 4) {
                              const double p0 = tas[j];
                              const double p1 = j + 1 < e ? tas[j + 1] : 0.0;
                              const double p2 = j + 2 < e ? tas[j + 2] : 0.0;
                              const double p3 = j + 3 < e ? tas[j + 3] : 0.0;
                              acc0 += p0 + p2;
                              acc1 += p1 + p3;
                        }
                        store_y<EPI>(y, row, acc0 + acc1, epi, dot_acc);
                  } else {
                        s_queue[atomicAdd(s_queue_n, 1)] = row;
                  }
            }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(THREADS) : "memory");

      const int nq = *s_queue_n;
      const int warp = tid >> 5, lane = tid & 31;
      for (int q = warp; q < nq; q += THREADS / 32) {
            const int row = s_queue[q];
            const int s = (int)((long long)s_irp[row - r0a] - kbase);
            const int e = (int)((long long)s_irp[row - r0a + 1] - kbase);
            double acc = 0.0;
            for (int j = s + lane; j < e; j += 32)
                  acc += tas[j];
            acc = group_sum<32>(acc);
            if (lane == 0)
                  store_y<EPI>(y, row, acc, epi, dot_acc);
      }
      // the stage was written through the generic proxy; order those writes
      // before the bulk copy (async proxy) that refills it
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// code_off / codes: the code blocks of the tiles (CODES only; tile t's block is
// codes[code_off[t], code_off[t+1])).
template <int THREADS, int LPR, int STAGES, int CAP, int PASSES, bool WS, bool SPLIT, int EPI,
          bool CODES, typename OffT>
__global__ void __launch_bounds__(THREADS + (WS ? 32 : 0))
    csr_stream_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                      const double *__restrict__ as, const int *__restrict__ tile_row,
                      const long long *__restrict__ tile_k, const long long *__restrict__ code_off,
                      const unsigned char *__restrict__ codes, int tile0, int n_tiles,
                      const double *__restrict__ x, double *__restrict__ y, EpiArgs epi) {
      using Cfg = StreamCfg<THREADS, LPR, STAGES, CAP, PASSES, WS, SPLIT, CODES>;
      extern __shared__ __align__(128) unsigned char smem_raw[];
      double *s_as = reinterpret_cast<double *>(smem_raw);
      // index part of the stages: int32 columns, or code blocks
      unsigned char *s_idx = smem_raw + (size_t)STAGES * CAP * 8;
      uint64_t *full = reinterpret_cast<uint64_t *>(s_idx + (size_t)STAGES * Cfg::kIdxBytes);
      uint64_t *empty = full + STAGES;
      int *s_queue_n = reinterpret_cast<int *>(empty + STAGES + 1);
      int *s_queue = s_queue_n + 4;
      // staged row offsets (entry-split mode only), 16-byte aligned
      OffT *s_irp = reinterpret_cast<OffT *>(
          (reinterpret_cast<uintptr_t>(s_queue + Cfg::kQueue) + 15) & ~uintptr_t(15));
      constexpr int IRP_ALIGN = 16 / (int)sizeof(OffT); // rows per 16 bytes
      static_assert(!SPLIT || WS, "the entry-split mode is only built warp-specialised");

      constexpr int RPP = THREADS / LPR;
      constexpr int CWARPS = THREADS / 32;
      const int tid = threadIdx.x;
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();

      if (tid == 0) {
            for (int s = 0; s < STAGES; ++s) {
                  mbar_init(&full[s], 1);
                  mbar_init(&empty[s], CWARPS);
            }
            mbar_fence_init();
            if (SPLIT)
                  s_queue_n[0] = s_queue_n[1] = 0;
      }
      __syncthreads();
      double dot_acc = 0.0;

      const int first = tile0 + blockIdx.x;
      const int last = tile0 + n_tiles;
      const int stride = gridDim.x;

      auto issue = [&](int t, int stage) {
            const long long k0 = tile_k[t] & ~3ll;
            const long long k1 = (tile_k[t + 1] + 3) & ~3ll;
            const long long cnt = k1 - k0;
            if (cnt > CAP) {
                  // a long row handled elsewhere: complete the phase with a
                  // zero-byte arrival
                  mbar_expect_tx(&full[stage], 0);
                  return;
            }
            uint32_t irp_bytes = 0;
            int r0a = 0;
            if (SPLIT) {
                  r0a = tile_row[t] & ~(IRP_ALIGN - 1);
                  const int n = (tile_row[t + 1] + 1 - r0a + IRP_ALIGN - 1) & ~(IRP_ALIGN - 1);
                  irp_bytes = (uint32_t)n * (uint32_t)sizeof(OffT);
            }
            long long idx_off = k0 * 4, idx_bytes = cnt * 4;
            const unsigned char *idx_src = reinterpret_cast<const unsigned char *>(ja);
            if (CODES) {
                  idx_off = code_off[t];
                  idx_bytes = code_off[t + 1] - idx_off;
                  idx_src = codes;
            }
            mbar_expect_tx(&full[stage], (uint32_t)(cnt * 8 + idx_bytes) + irp_bytes);
            if (cnt > 0) {
                  bulk_g2s(s_as + (size_t)stage * CAP, as + k0, (uint32_t)(cnt * 8), &full[stage],
                           pol_s);
                  bulk_g2s(s_idx + (size_t)stage * Cfg::kIdxBytes, idx_src + idx_off,
                           (uint32_t)idx_bytes, &full[stage], pol_s);
            }
            if (SPLIT)
                  bulk_g2s(s_irp + (size_t)stage * Cfg::kIrpSlots, irp + r0a, irp_bytes,
                           &full[stage], pol_s);
      };

      if (WS && tid >= THREADS) {
            // ---------------- producer warp: one lane drives the ring ----------
            if (tid == THREADS) {
                  int it = 0;
                  for (int t = first; t < last; t += stride, ++it) {
                        const int stage = it % STAGES;
                        if (it >= STAGES)
                              mbar_wait(&empty[stage], (uint32_t)(it / STAGES - 1) & 1u);
                        issue(t, stage);
                  }
            }
            return;
      }

      if (!WS && tid == 0) {
            int t = first;
            for (int s = 0; s < STAGES && t < last; ++s, t += stride)
                  issue(t, s);
      }

      const int gi = tid / LPR, sub = tid % LPR;
      int it = 0;
      int n_split = 0; // entry-split tiles done so far: selects the long-row counter (tiles that
                       // hold one oversized row are skipped and must not advance the alternation)
      for (int t = first; t < last; t += stride, ++it) {
            const int stage = it % STAGES;
            const uint32_t parity = (uint32_t)(it / STAGES) & 1u;
            const int r0 = tile_row[t], r1 = tile_row[t + 1];
            const long long kbase = tile_k[t] & ~3ll;
            const bool staged = ((tile_k[t + 1] + 3) & ~3ll) - kbase <= CAP;

            // row extent of pass 0 is fetched before waiting on the copy
            long long ks = 0, ke = 0;
            if (!SPLIT && r0 + gi < r1) {
                  ks = (long long)irp[r0 + gi] - kbase;
                  ke = (long long)irp[r0 + gi + 1] - kbase;
            }
            mbar_wait(&full[stage], parity);

            if (SPLIT) {
                  const int cnt = (int)(((tile_k[t + 1] + 3) & ~3ll) - kbase);
                  if (staged) {
                        stream_tile_products<THREADS, PASSES, CAP, EPI, OffT>(
                            s_irp + (size_t)stage * Cfg::kIrpSlots, s_as + (size_t)stage * CAP,
                            reinterpret_cast<const int *>(s_idx + (size_t)stage * Cfg::kIdxBytes),
                            r0, r1, r0 & ~(IRP_ALIGN - 1), kbase, cnt,
                            tid, x, y, pol_x, epi, dot_acc, s_queue, s_queue_n + (n_split & 1),
                            s_queue_n + ((n_split + 1) & 1));
                        ++n_split;
                  }
            } else if (staged) {
                  const unsigned char *t_idx = s_idx + (size_t)stage * Cfg::kIdxBytes;
                  // the dictionary follows the codes of the tile's staged entries
                  const long long cnt = ((tile_k[t + 1] + 3) & ~3ll) - kbase;
                  stream_tile_rows<LPR, RPP, PASSES, EPI, CODES, OffT>(
                      irp, s_as + (size_t)stage * CAP, reinterpret_cast<const int *>(t_idx), t_idx,
                      reinterpret_cast<const int *>(t_idx + round16(cnt)), r0, r1, kbase, gi, sub,
                      ks, ke, x, y, pol_x, epi, dot_acc);
            }
            if (WS) {
                  __syncwarp();
                  if ((tid & 31) == 0)
                        mbar_arrive(&empty[stage]);
            } else {
                  __syncthreads();
                  if (tid == 0) {
                        const int tn = t + STAGES * stride;
                        if (tn < last)
                              issue(tn, stage);
                  }
            }
      }
      epi_finish_warp<EPI>(epi, dot_acc, (long long)blockIdx.x * CWARPS + (tid >> 5));
}

// Code blocks of the staged tiles (layout above), one CTA of 256 threads per tile.  The tile's
// distinct offsets d = ja[k] - row go into a shared-memory hash set; a code is the rank of d among
// them, so the blocks depend on the matrix only, not on the order the set was filled in.
//   codes == nullptr  count pass: n_dict[t] = distinct offsets (kCodeDict + 1: too many) and
//                     bytes[t] = size of the block (0 for a tile holding one row beyond `cap`)
//   otherwise         fill pass: write block t at codes + code_off[t], every byte of it (entries
//                     staged with the tile that belong to its neighbours, and padding: code 0)
constexpr int kCodeHash = 1024; // hash slots: > 2 * kCodeDict
template <typename OffT>
__global__ void __launch_bounds__(256)
    stream_codes_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                        const int *__restrict__ tile_row, const long long *__restrict__ tile_k,
                        int cap, int *__restrict__ n_dict, long long *__restrict__ bytes,
                        const long long *__restrict__ code_off, unsigned char *__restrict__ codes) {
      constexpr int kEmpty = -0x7fffffff - 1; // no offset: col >= 0 and row < 2^31 give d > -2^31
      __shared__ int s_key[kCodeHash];
      __shared__ unsigned char s_rank[kCodeHash];
      __shared__ short s_slot[kCodeDict]; // occupied slots, in claim order
      __shared__ int s_n, s_over;
      const int t = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
      const long long k0 = tile_k[t] & ~3ll, k1 = (tile_k[t + 1] + 3) & ~3ll;
      if (k1 - k0 > cap) { // one long row: the long-row kernels take it, no block
            if (!codes && tid == 0)
                  n_dict[t] = 0, bytes[t] = 0;
            return;
      }
      for (int i = tid; i < kCodeHash; i += 256)
            s_key[i] = kEmpty;
      if (tid == 0)
            s_n = 0, s_over = 0;
      __syncthreads();
      auto hash = [](int d) { return (int)(((unsigned)d * 2654435761u) >> 22); }; // 10 bits
      const int r0 = tile_row[t], r1 = tile_row[t + 1];
      for (int row = r0 + warp; row < r1; row += 8) {
            const long long e = (long long)irp[row + 1];
            for (long long k = (long long)irp[row] + lane; k < e; k += 32) {
                  // past kCodeDict offsets the answer is known: stop before the table fills (at
                  // most one more claim per thread follows, 257 + 256 < kCodeHash)
                  if (*(volatile int *)&s_n > kCodeDict)
                        break;
                  const int d = ja[k] - row;
                  int h = hash(d), i = 0;
                  for (; i < kCodeHash; ++i, h = (h + 1) & (kCodeHash - 1)) {
                        int v = *(volatile int *)&s_key[h];
                        if (v == kEmpty) {
                              v = atomicCAS(&s_key[h], kEmpty, d);
                              if (v == kEmpty) {
                                    const int n = atomicAdd(&s_n, 1);
                                    if (n < kCodeDict)
                                          s_slot[n] = (short)h;
                                    break;
                              }
                        }
                        if (v == d)
                              break;
                  }
                  if (i == kCodeHash)
                        s_over = 1; // the table is full: far more than kCodeDict offsets
            }
      }
      __syncthreads();
      const int n = s_over ? kCodeDict + 1 : min(s_n, kCodeDict + 1);
      const long long code_bytes = round16(k1 - k0);
      if (!codes) {
            if (tid == 0)
                  n_dict[t] = n, bytes[t] = code_bytes + round16(4ll * n);
            return;
      }
      if (n > kCodeDict)
            return; // the plan is not coded: the host never asks for this
      unsigned char *blk = codes + code_off[t];
      int *dict = reinterpret_cast<int *>(blk + code_bytes);
      for (int i = tid; i < n; i += 256) {
            const int v = s_key[s_slot[i]];
            int r = 0;
            for (int j = 0; j < n; ++j)
                  r += s_key[s_slot[j]] < v;
            s_rank[s_slot[i]] = (unsigned char)r;
            dict[r] = v;
      }
      for (int i = n + tid; i < (int)(round16(4ll * n) / 4); i += 256)
            dict[i] = 0;
      // staged positions outside the tile's own entries
      const int lead = (int)(tile_k[t] - k0), tail = (int)(tile_k[t + 1] - k0);
      for (int p = tid; p < (int)code_bytes; p += 256)
            if (p < lead || p >= tail)
                  blk[p] = 0;
      __syncthreads();
      for (int row = r0 + warp; row < r1; row += 8) {
            const long long e = (long long)irp[row + 1];
            for (long long k = (long long)irp[row] + lane; k < e; k += 32) {
                  const int d = ja[k] - row;
                  int h = hash(d);
                  while (s_key[h] != d)
                        h = (h + 1) & (kCodeHash - 1);
                  blk[k - k0] = s_rank[h];
            }
      }
}

// ------------------------------------------------------------------------
// K right-hand sides straight from CSR (Y[M][K] = A X[N][K], row-major): LPR lanes per row, the
// lanes of a row combined with shuffles.  The route of matrices that have no SELL-P plan (regular
// rows with local columns) and of rows too long for a slice.
template <int K, int LPR, typename OffT>
__global__ void __launch_bounds__(512)
    csr_mm_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                  const double *__restrict__ as, long long row0, long long nrows,
                  const int *__restrict__ rowlist, const double *__restrict__ X,
                  double *__restrict__ Y) {
      const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
      const long long g = gid / LPR;
      const int sub = (int)(gid % LPR);
      if (g >= nrows)
            return; // whole groups leave together
      const long long row = rowlist ? (long long)rowlist[g] : row0 + g;
      const OffT s = irp[row], e = irp[row + 1];
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      constexpr int U = 4;
      double acc[K];
#pragma unroll
      for (int k = 0; k < K; ++k)
            acc[k] = 0.0;
      for (OffT k0 = s + sub; k0 < e; k0 += LPR * U) {
            double a[U], xv[U][K];
            int c[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                  const OffT kk = k0 + u * LPR;
                  const bool ok = kk < e;
                  a[u] = ok ? ld_stream_f64(as + kk, pol_s) : 0.0;
                  c[u] = ok ? ld_stream_s32(ja + kk, pol_s) : -1;
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
#pragma unroll
      for (int k = 0; k < K; ++k)
            acc[k] = group_sum<LPR>(acc[k]);
      if (sub == 0) {
#pragma unroll
            for (int k = 0; k < K; ++k)
                  Y[row * K + k] = acc[k];
      }
}

// Y[split_row[i]][0..K) = sum of the row's pieces, in piece order
template <int K>
__global__ void csr_combine_mm_kernel(const int *__restrict__ split_row,
                                      const int *__restrict__ split_first, int n_split,
                                      const double *__restrict__ partial, double *__restrict__ Y) {
      const int i = blockIdx.x * blockDim.x + threadIdx.x;
      if (i >= n_split)
            return;
      double acc[K];
#pragma unroll
      for (int k = 0; k < K; ++k)
            acc[k] = 0.0;
      for (int c = split_first[i]; c < split_first[i + 1]; ++c)
#pragma unroll
            for (int k = 0; k < K; ++k)
                  acc[k] += partial[(long long)c * K + k];
#pragma unroll
      for (int k = 0; k < K; ++k)
            Y[(long long)split_row[i] * K + k] = acc[k];
}

// ------------------------------------------------------------------------
// Short regular rows (5-point stencils, BASELINE configs[0]): the CSR twin of hll_pipe_kernel.
// Persistent warps; a warp owns groups of 32 consecutive rows (g, g + W, ...), whose entries are
// one contiguous piece of ja / as: lane 0 fetches it (rounded out to multiples of 4 entries, the
// arrays carry 16 spare entries) with two bulk copies into the warp's private ring of STAGES
// buffers, every lane then walks its own row in shared memory (row starts are ~5 words apart:
// conflict-free), and the row offsets of the group after next are loaded while the current one is
// computed.  No CTA-wide synchronisation, no plan arrays.  The launcher guarantees rows <= 8.
// One group of the pipelined short-row kernel: W (compile time, 1..8) entries per lane at most.
template <int W>
__device__ __forceinline__ double csr_pipe_rows(const double *__restrict__ tas, const int *__restrict__ tja,
                                                int k0, int len, const double *__restrict__ x,
                                                uint64_t pol_x) {
      double a[W], xv[W];
      int c[W];
#pragma unroll
      for (int u = 0; u < W; ++u) {
            const bool ok = u < len;
            c[u] = ok ? tja[k0 + u] : -1;
            a[u] = ok ? tas[k0 + u] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < W; ++u)
            xv[u] = c[u] >= 0 ? ld_x(x + c[u], pol_x) : 0.0;
      double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
      for (int u = 0; u < W; ++u) { // even entries into acc0, odd ones into acc1: the order of every other kernel
            if (u & 1)
                  acc1 = fma(a[u], xv[u], acc1);
            else
                  acc0 = fma(a[u], xv[u], acc0);
      }
      return acc0 + acc1;
}

template <int STAGES, int CAPW, typename OffT>
__global__ void __launch_bounds__(256)
    csr_pipe_kernel(const OffT *__restrict__ irp, const int *__restrict__ ja,
                    const double *__restrict__ as, long long row0, int n_rows,
                    const double *__restrict__ x, double *__restrict__ y) {
      extern __shared__ __align__(128) unsigned char smem_raw[];
      constexpr int kStageBytes = CAPW * 12;
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
      unsigned char *ring = smem_raw + warp * (STAGES * kStageBytes);
      uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + wpc * (STAGES * kStageBytes)) + warp * STAGES;
      // groups of 32 rows, dealt round-robin to the warps of the grid; 32-bit arithmetic throughout
      // (a shard has fewer than 2^31 rows), the row offsets themselves are OffT
      const int W = (int)gridDim.x * wpc;
      const int first = (int)blockIdx.x * wpc + warp;
      const int n_groups = (n_rows + 31) >> 5;
      irp += row0;
      y += row0;
      const uint64_t pol_s = policy_evict_first();
      const uint64_t pol_x = policy_evict_last();
      if (lane == 0) {
#pragma unroll
            for (int s = 0; s < STAGES; ++s)
                  mbar_init(&bars[s], 1);
            mbar_fence_init();
      }
      __syncwarp();

      // row offsets of group g: this lane's row [lo, hi), the group's entries [k_lo, k_hi)
      auto offsets = [&](int g, OffT &lo, OffT &hi, OffT &k_lo, OffT &k_hi) {
            lo = irp[min(g * 32 + lane, n_rows)];
            k_hi = irp[min(g * 32 + 32, n_rows)];
            hi = __shfl_down_sync(0xffffffffu, lo, 1);
            if (lane == 31)
                  hi = k_hi;
            k_lo = __shfl_sync(0xffffffffu, lo, 0);
      };
      int s0[STAGES] = {0}, len[STAGES] = {0}; // this lane's entries inside the stage's buffer
      auto fetch = [&](int s, OffT lo, OffT hi, OffT k_lo, OffT k_hi) {
            // (rounding out to 128-byte lines instead measured the same: profiles/r2_kbench_poisson3000_pipe.txt)
            const OffT ka = k_lo & ~(OffT)3, kb = (k_hi + 3) & ~(OffT)3;
            s0[s] = (int)(lo - ka), len[s] = (int)(hi - lo);
            if (lane == 0) {
                  const uint32_t cnt = (uint32_t)(kb - ka);
                  mbar_expect_tx(&bars[s], cnt * 12);
                  if (cnt > 0) {
                        bulk_g2s(ring + s * kStageBytes, as + ka, cnt * 8, &bars[s], pol_s);
                        bulk_g2s(ring + s * kStageBytes + CAPW * 8, ja + ka, cnt * 4, &bars[s], pol_s);
                  }
            }
      };
#pragma unroll
      for (int s = 0; s < STAGES; ++s) {
            const int g = first + s * W;
            if (g < n_groups) {
                  OffT lo, hi, k_lo, k_hi;
                  offsets(g, lo, hi, k_lo, k_hi);
                  fetch(s, lo, hi, k_lo, k_hi);
            }
      }
      uint32_t parity = 0;
      for (int g0 = first;; g0 += STAGES * W, parity ^= 1u) {
#pragma unroll
            for (int s = 0; s < STAGES; ++s) {
                  const int g = g0 + s * W;
                  if (g >= n_groups)
                        return; // whole warp
                  const int gn = g + STAGES * W;
                  OffT lo = 0, hi = 0, k_lo = 0, k_hi = 0;
                  if (gn < n_groups)
                        offsets(gn, lo, hi, k_lo, k_hi); // on their way while this group is computed
                  mbar_wait(&bars[s], parity);
                  const double *tas = reinterpret_cast<const double *>(ring + s * kStageBytes);
                  const int *tja = reinterpret_cast<const int *>(ring + s * kStageBytes + CAPW * 8);
                  const int k0 = s0[s], n = len[s];
                  // exactly as many entry slots as the longest row of the group needs (<= 8 by the
                  // launcher's guarantee): a 5-point row costs 5 gathers, not 8 predicated ones
                  const int wmax = __reduce_max_sync(0xffffffffu, n);
                  double acc;
                  switch (wmax) {
                  case 0: acc = 0.0; break;
                  case 1: acc = csr_pipe_rows<1>(tas, tja, k0, n, x, pol_x); break;
                  case 2: acc = csr_pipe_rows<2>(tas, tja, k0, n, x, pol_x); break;
                  case 3: acc = csr_pipe_rows<3>(tas, tja, k0, n, x, pol_x); break;
                  case 4: acc = csr_pipe_rows<4>(tas, tja, k0, n, x, pol_x); break;
                  case 5: acc = csr_pipe_rows<5>(tas, tja, k0, n, x, pol_x); break;
                  case 6: acc = csr_pipe_rows<6>(tas, tja, k0, n, x, pol_x); break;
                  case 7: acc = csr_pipe_rows<7>(tas, tja, k0, n, x, pol_x); break;
                  default: acc = csr_pipe_rows<8>(tas, tja, k0, n, x, pol_x); break;
                  }
                  __syncwarp(); // every lane has read the stage: it may be overwritten
                  if (gn < n_groups)
                        fetch(s, lo, hi, k_lo, k_hi);
                  const int r = g * 32 + lane;
                  if (r < n_rows)
                        y[r] = acc;
            }
      }
}

} // namespace b200
