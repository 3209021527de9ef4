// spmv_b200.cu -- libspmv_b200 core: resident matrices, launch plans, kernel launchers and the
// handle API of include/spmv_b200.h.
//
// The other translation units: entry.cu (the reference's GPU boundary -- include/cuda_csr.h,
// include/cuda_hll.h, include/cuda_timer.h -- replacing reference src/cuda_csr.cu,
// src/cuda_hll.cu and src/cuda_timer.cu, plus the host-buffer pipelines) and dist.cu (multi-GPU
// iterated SpMV).  There is no CPU fallback anywhere: without a usable GPU every entry point
// fails loudly.
#include "internal.cuh"

#include <cub/cub.cuh>
#include <memory>
#include <type_traits>
#include <new>

#include "coo_kernels.cuh"
#include "csr_kernels.cuh"
#include "gen_kernels.cuh"
#include "hll_kernels.cuh"
#include "sell_kernels.cuh"
#include "spgemm_kernels.cuh"
#include "transpose_kernels.cuh"

using namespace b200;

// ===================================================================== state
namespace b200 {

Counters g_counters;
Knobs g_knobs;
int g_sm_count = 0;

int ensure_device() {
      static std::once_flag once;
      static int rc = 0;
      std::call_once(once, [] {
            int n = 0;
            cudaError_t e = cudaGetDeviceCount(&n);
            if (e != cudaSuccess || n == 0) {
                  rc = fail(-ENODEV, "no CUDA device available (%s); libspmv_b200 has no CPU path",
                            e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
                  return;
            }
            const char *env;
            if ((env = getenv("SPMV_B200_WARMUP")))
                  g_knobs.warmup = std::max(0, atoi(env));
            if ((env = getenv("SPMV_B200_REPS")))
                  g_knobs.reps = std::max(1, atoi(env));
            if ((env = getenv("SPMV_B200_CACHE"))) {
                  if (!strcmp(env, "off") || !strcmp(env, "0"))
                        g_knobs.cache = 0;
                  else if (!strcmp(env, "trust") || !strcmp(env, "2"))
                        g_knobs.cache = 2;
                  else
                        g_knobs.cache = 1;
            }
      });
      if (rc)
            return rc;
      if (!g_sm_count) {
            int dev = 0;
            cudaDeviceProp p;
            if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&p, dev) != cudaSuccess)
                  return fail(-EIO, "cudaGetDeviceProperties failed");
            if (p.major < 10)
                  return fail(-ENODEV, "device %s is sm_%d%d; this library is built for sm_100a only",
                              p.name, p.major, p.minor);
            g_sm_count = p.multiProcessorCount;
      }
      return 0;
}

// (An L2 access-policy window that pins part of a large x was tried in round 1 and removed:
// reserving the persisting carve-out shrinks the L2 left for everything else -- C2 dropped from
// 97 % to 89 % of peak -- and C3/C4, whose gathers it was meant to help, did not move at all:
// profiles/r1_kbench_c3_l2window_{on,off}.txt.  The per-load evict_last / evict_first policies
// and, for x larger than the L2, the column panels of sell_kernels.cuh are what is used.)

} // namespace b200

namespace {
void *g_flush_buf[kMaxDevices] = {nullptr};
constexpr size_t kFlushBytes = 512ull << 20; // > 126 MB L2
} // namespace

// ============================================================ build helpers
namespace {

template <typename T> struct OffTag { using type = T; };

// f(OffTag<OffT>{}) with OffT the row offset type of a handle: long long when `wide`, else int.
template <typename F> auto with_offsets(bool wide, F &&f) {
      return wide ? f(OffTag<long long>{}) : f(OffTag<int>{});
}

// Device temporaries of one build, freed on every way out.
struct DeviceTemps {
      std::vector<void *> ptrs;
      long long bytes = 0; // requested so far, for the -ENOMEM message
      ~DeviceTemps() { release_all(); }
      template <typename T>
      int alloc(T **out, size_t n_bytes, const char *what) {
            bytes += (long long)n_bytes;
            void *p = nullptr;
            if (cudaMalloc(&p, std::max<size_t>(n_bytes, 1)) != cudaSuccess) {
                  cudaGetLastError(); // clear the allocation error
                  return fail(-ENOMEM, "%s: cudaMalloc of %lld bytes of temporaries failed", what, bytes);
            }
            ptrs.push_back(p);
            *out = static_cast<T *>(p);
            return 0;
      }
      // alloc() holding a copy of `h`, counted in the h2d bytes as upload() counts it
      template <typename T>
      int upload(T **d, const std::vector<T> &h, const char *what) {
            const size_t n_bytes = h.size() * sizeof(T);
            if (alloc(d, n_bytes, what))
                  return -ENOMEM;
            B200_CUDA(cudaMemcpy(*d, h.data(), n_bytes, cudaMemcpyHostToDevice));
            g_counters.h2d += (long long)n_bytes;
            return 0;
      }
      void release(const void *p) {
            for (auto &q : ptrs)
                  if (q == p) {
                        cudaFree(q);
                        q = nullptr;
                  }
      }
      void release_all() {
            for (void *p : ptrs)
                  cudaFree(p);
            ptrs.clear();
      }
};

} // namespace

// ================================================================ CSR plans
namespace b200 {

void free_list(RowList &l) {
      cudaFree(l.d_rows);
      l = RowList();
}
void free_split(SplitPlan &s) {
      cudaFree(s.d_k0), cudaFree(s.d_k1), cudaFree(s.d_row), cudaFree(s.d_first),
          cudaFree(s.d_partial);
      s = SplitPlan();
}
void free_sell(SellPlan &sp) {
      cudaFree(sp.d_soff), cudaFree(sp.d_perm), cudaFree(sp.d_ja), cudaFree(sp.d_as);
      free_list(sp.long_warp);
      free_list(sp.long_block);
      free_split(sp.long_split);
      cudaFree(sp.d_split_row), cudaFree(sp.d_split_first), cudaFree(sp.d_partial), cudaFree(sp.d_partial_mm);
      sp = SellPlan();
}
void free_segment(Segment &sg) {
      for (auto &l : sg.lists)
            free_list(l);
      free_split(sg.split);
      for (auto &kv : sg.stream) {
            cudaFree(kv.second.d_code_off);
            cudaFree(kv.second.d_codes);
            cudaFree(kv.second.d_tile_row);
            cudaFree(kv.second.d_tile_k);
            for (auto &l : kv.second.long_lists)
                  free_list(l);
            free_split(kv.second.split);
      }
      sg.stream.clear();
}

static int build_split(const spmv_b200_csr *h, const std::vector<int> &rows, SplitPlan &sp) {
      std::vector<long long> k0, k1;
      std::vector<int> first;
      for (int r : rows) {
            first.push_back((int)k0.size());
            for (long long k = h->h_irp[r]; k < h->h_irp[r + 1]; k += kSplitChunk) {
                  k0.push_back(k);
                  k1.push_back(std::min(k + kSplitChunk, h->h_irp[r + 1]));
            }
      }
      first.push_back((int)k0.size());
      sp.n_rows = (int)rows.size();
      sp.n_chunks = (int)k0.size();
      if (!sp.n_rows)
            return 0;
      int rc = upload(&sp.d_k0, k0);
      rc = rc ? rc : upload(&sp.d_k1, k1);
      rc = rc ? rc : upload(&sp.d_row, rows);
      rc = rc ? rc : upload(&sp.d_first, first);
      if (rc)
            return rc;
      B200_CUDA(cudaMalloc(&sp.d_partial, sizeof(double) * (size_t)sp.n_chunks));
      return 0;
}

// Classify the rows of one segment into length bins (counts only; the per-bin row lists are
// built on first use of the direct binned kernels, build_bin_lists).
int build_adaptive(spmv_b200_csr *h, Segment &sg) {
      const long long rows = sg.r1 - sg.r0;
      std::fill(sg.kind_rows, sg.kind_rows + kNumKinds, 0);
      sg.max_len = 0;
      for (long long r = sg.r0; r < sg.r1; ++r) {
            const long long len = h->h_irp[r + 1] - h->h_irp[r];
            ++sg.kind_rows[kind_of(len)];
            sg.max_len = std::max(sg.max_len, len);
      }

      // "regular" matrix: one bin holds the bulk of the rows and nearly all
      // other rows are shorter -> run ONE launch over the contiguous range
      // with that bin's lanes-per-row (no row list, y written in order);
      // only longer rows go through lists.
      int dom = 0;
      for (int k = 1; k < 6; ++k)
            if (sg.kind_rows[k] > sg.kind_rows[dom])
                  dom = k;
      long long below = 0;
      for (int k = 0; k <= dom; ++k)
            below += sg.kind_rows[k];
      sg.regular = rows > 0 && below * 10 >= rows * 9;
      sg.base_kind = dom;
      return 0;
}

static int build_bin_lists(spmv_b200_csr *h, Segment &sg) {
      if (sg.lists_built)
            return 0;
      std::vector<int> lists[kNumKinds];
      for (long long r = sg.r0; r < sg.r1; ++r) {
            const int k = kind_of(h->h_irp[r + 1] - h->h_irp[r]);
            if (sg.regular && k <= sg.base_kind)
                  continue;
            lists[k].push_back((int)r);
      }
      for (int k = 0; k < kNumKinds; ++k) {
            sg.lists[k].n = (long long)lists[k].size();
            if (k == kNumKinds - 1) {
                  int rc = build_split(h, lists[k], sg.split);
                  if (rc)
                        return rc;
            } else {
                  int rc = upload(&sg.lists[k].d_rows, lists[k]);
                  if (rc)
                        return rc;
            }
      }
      sg.lists_built = true;
      return 0;
}

// Tiles of consecutive rows for the TMA-staged kernel.
static int build_stream(spmv_b200_csr *h, Segment &sg, int max_rows, int cap, StreamPlan &sp) {
      std::vector<int> tile_row;
      std::vector<long long> tile_k;
      std::vector<int> longs[kNumKinds];
      long long r = sg.r0;
      while (r < sg.r1) {
            const long long kstart = h->h_irp[r];
            const long long kbase = kstart & ~3ll;
            long long e = r;
            while (e < sg.r1 && e - r < max_rows &&
                   ((h->h_irp[e + 1] + 3) & ~3ll) - kbase <= cap)
                  ++e;
            if (e == r) { // a single row that does not fit a stage
                  const long long len = h->h_irp[r + 1] - kstart;
                  longs[std::max(5, kind_of(len))].push_back((int)r);
                  e = r + 1;
            }
            tile_row.push_back((int)r);
            tile_k.push_back(kstart);
            r = e;
      }
      tile_row.push_back((int)sg.r1);
      tile_k.push_back(h->h_irp[sg.r1]);
      sp.n_tiles = (int)tile_row.size() - 1;
      int rc = upload(&sp.d_tile_row, tile_row);
      rc = rc ? rc : upload(&sp.d_tile_k, tile_k);
      for (int k = 5; k < kNumKinds - 1 && !rc; ++k) {
            sp.long_lists[k].n = (long long)longs[k].size();
            rc = upload(&sp.long_lists[k].d_rows, longs[k]);
      }
      rc = rc ? rc : build_split(h, longs[kNumKinds - 1], sp.split);
      sp.built = rc == 0;
      return rc;
}

// Column codes of a row-tile plan (stream_codes_kernel), all or nothing: codes_state = 1 when
// every staged tile has at most kCodeDict distinct column offsets, else -1 and the plan keeps
// its int32 columns.  The codes only save bytes, so when device memory for them or for the build
// runs short the plan also keeps its int32 columns (-1, no error).  Every buffer stays in the
// temporaries guard until the build has succeeded, so no way out leaks one.  Synchronous on the
// legacy stream, so never inside a graph capture (plans are built on a handle's first launches).
template <typename OffT>
static int build_codes(spmv_b200_csr *h, int cap, StreamPlan &sp) {
      sp.codes_state = -1; // until the blocks exist
      const int T = sp.n_tiles;
      if (T <= 0)
            return 0;
      DeviceTemps tmp;
      // quiet allocation: running short is not an error here
      auto grab = [&](auto **out, size_t n_bytes) {
            void *p = nullptr;
            if (cudaMalloc(&p, std::max<size_t>(n_bytes, 1)) != cudaSuccess) {
                  cudaGetLastError(); // clear the allocation error
                  return false;
            }
            tmp.ptrs.push_back(p);
            *out = static_cast<std::remove_pointer_t<decltype(out)>>(p);
            return true;
      };
      int *d_nd = nullptr, *d_max = nullptr;
      long long *d_bytes = nullptr, *d_code_off = nullptr;
      unsigned char *d_codes = nullptr;
      void *d_scratch = nullptr;
      size_t scan_b = 0, max_b = 0;
      B200_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_b, d_bytes, d_code_off, T + 1));
      B200_CUDA(cub::DeviceReduce::Max(nullptr, max_b, d_nd, d_max, T));
      if (!grab(&d_nd, (size_t)T * sizeof(int)) || !grab(&d_max, sizeof(int)) ||
          !grab(&d_bytes, (size_t)(T + 1) * sizeof(long long)) ||
          !grab(&d_scratch, std::max(scan_b, max_b)) ||
          !grab(&d_code_off, (size_t)(T + 1) * sizeof(long long)))
            return 0;
      const OffT *irp = static_cast<const OffT *>(h->d_irp);
      int max_nd = 0;
      long long total = 0;
      cudaError_t e = cudaMemset(d_bytes + T, 0, sizeof(long long));
      if (e == cudaSuccess) {
            stream_codes_kernel<OffT><<<T, 256>>>(irp, h->d_ja, sp.d_tile_row, sp.d_tile_k, cap,
                                                   d_nd, d_bytes, nullptr, nullptr);
            e = cub::DeviceScan::ExclusiveSum(d_scratch, scan_b, d_bytes, d_code_off, T + 1);
      }
      if (e == cudaSuccess)
            e = cub::DeviceReduce::Max(d_scratch, max_b, d_nd, d_max, T);
      if (e == cudaSuccess)
            e = cudaMemcpy(&max_nd, d_max, sizeof(int), cudaMemcpyDeviceToHost);
      if (e == cudaSuccess)
            e = cudaMemcpy(&total, d_code_off + T, sizeof(long long), cudaMemcpyDeviceToHost);
      if (e != cudaSuccess)
            return fail(-EIO, "column codes: count pass failed: %s", cudaGetErrorString(e));
      if (max_nd > kCodeDict || !grab(&d_codes, (size_t)total))
            return 0;
      stream_codes_kernel<OffT><<<T, 256>>>(irp, h->d_ja, sp.d_tile_row, sp.d_tile_k, cap, d_nd,
                                             d_bytes, d_code_off, d_codes);
      e = cudaStreamSynchronize(nullptr);
      if (e == cudaSuccess)
            e = cudaGetLastError();
      if (e != cudaSuccess)
            return fail(-EIO, "column codes: fill pass failed: %s", cudaGetErrorString(e));
      tmp.ptrs.pop_back(), tmp.ptrs.pop_back(); // d_codes and d_code_off belong to the plan now
      sp.d_code_off = d_code_off, sp.d_codes = d_codes;
      sp.code_bytes = total, sp.max_dict = max_nd, sp.codes_state = 1;
      return 0;
}

static int finish_create(spmv_b200_csr *h, const long long *cuts, int n_cuts) {
      std::vector<long long> bounds;
      bounds.push_back(0);
      for (int i = 0; i < n_cuts; ++i)
            if (cuts[i] > bounds.back() && cuts[i] < h->M)
                  bounds.push_back(cuts[i]);
      bounds.push_back(h->M);
      for (size_t i = 0; i + 1 < bounds.size(); ++i) {
            if (bounds[i + 1] == bounds[i] && h->M > 0)
                  continue;
            Segment sg;
            sg.r0 = bounds[i], sg.r1 = bounds[i + 1];
            h->segs.push_back(sg);
      }
      for (auto &sg : h->segs) {
            int rc = build_adaptive(h, sg);
            if (rc)
                  return rc;
      }
      return 0;
}

} // namespace b200

// ================================================================ launchers
namespace {

struct CsrArgs {
      const spmv_b200_csr *h;
      const double *x;
      double *y;
      int epi_mode; // EPI_PLAIN / EPI_PUSH / EPI_FUSED
      EpiArgs epi;
      cudaStream_t st;
      int threads;
};

// The direct (non-staged) kernels exist with the plain and the push epilogue only.
#define DIRECT_EPI_SWITCH(mode, STMT)                                                              \
      do {                                                                                         \
            if ((mode) == EPI_PUSH) {                                                              \
                  constexpr int E = EPI_PUSH;                                                      \
                  STMT;                                                                            \
            } else {                                                                               \
                  constexpr int E = EPI_PLAIN;                                                     \
                  STMT;                                                                            \
            }                                                                                      \
      } while (0)

template <int LPR, typename OffT>
void launch_vec_t(const CsrArgs &a, long long row0, long long nrows, const int *list,
                  long long max_len) {
      if (nrows <= 0)
            return;
      const int grid = blocks_for(nrows * LPR, a.threads);
      const OffT *irp = static_cast<const OffT *>(a.h->d_irp);
      DIRECT_EPI_SWITCH(a.epi_mode, (csr_vec_kernel<LPR, OffT, E><<<grid, a.threads, 0, a.st>>>(
                                        irp, a.h->d_ja, a.h->d_as, row0, nrows, list, max_len, a.x,
                                        a.y, a.epi)));
      ++g_counters.launches;
}

template <typename OffT>
void launch_vec(const CsrArgs &a, int lpr_log2, long long row0, long long nrows, const int *list,
                long long max_len) {
      switch (lpr_log2) {
      case 0: launch_vec_t<1, OffT>(a, row0, nrows, list, max_len); break;
      case 1: launch_vec_t<2, OffT>(a, row0, nrows, list, max_len); break;
      case 2: launch_vec_t<4, OffT>(a, row0, nrows, list, max_len); break;
      case 3: launch_vec_t<8, OffT>(a, row0, nrows, list, max_len); break;
      case 4: launch_vec_t<16, OffT>(a, row0, nrows, list, max_len); break;
      default: launch_vec_t<32, OffT>(a, row0, nrows, list, max_len); break;
      }
}

template <typename OffT>
void launch_block_rows(const CsrArgs &a, long long row0, long long nrows, const int *list) {
      if (nrows <= 0)
            return;
      // gridDim.x limit is 2^31-1, enough for any row count we accept
      DIRECT_EPI_SWITCH(a.epi_mode,
                        (csr_block_row_kernel<OffT, E><<<(unsigned)nrows, a.threads, 0, a.st>>>(
                            static_cast<const OffT *>(a.h->d_irp), a.h->d_ja, a.h->d_as, row0, list,
                            a.x, a.y, a.epi)));
      ++g_counters.launches;
}

void launch_split(const CsrArgs &a, const SplitPlan &sp) {
      if (!sp.n_rows)
            return;
      csr_split_kernel<<<sp.n_chunks, 512, 0, a.st>>>(sp.d_k0, sp.d_k1, a.h->d_ja, a.h->d_as, a.x,
                                                      sp.d_partial);
      DIRECT_EPI_SWITCH(a.epi_mode,
                        (csr_combine_kernel<E><<<blocks_for(sp.n_rows, 128), 128, 0, a.st>>>(
                            sp.d_row, sp.d_first, sp.n_rows, sp.d_partial, a.y, a.epi)));
      g_counters.launches += 2;
}

template <typename OffT>
void launch_long_lists(const CsrArgs &a, const RowList *lists, const SplitPlan &sp) {
      launch_vec<OffT>(a, 5, 0, lists[5].n, lists[5].d_rows, -1);
      CsrArgs b = a;
      b.threads = 512;
      launch_block_rows<OffT>(b, 0, lists[6].n, lists[6].d_rows);
      launch_split(a, sp);
}

template <typename OffT>
void run_adaptive(const CsrArgs &a, const Segment &sg) {
      if (sg.regular)
            launch_vec<OffT>(a, sg.base_kind, sg.r0, sg.r1 - sg.r0, nullptr,
                             kKindMax[sg.base_kind]);
      for (int k = 0; k < 5; ++k)
            if (!(sg.regular && k <= sg.base_kind))
                  launch_vec<OffT>(a, k, 0, sg.lists[k].n, sg.lists[k].d_rows, -1);
      if (!(sg.regular && sg.base_kind >= 5))
            launch_vec<OffT>(a, 5, 0, sg.lists[5].n, sg.lists[5].d_rows, -1);
      CsrArgs b = a;
      b.threads = 512;
      launch_block_rows<OffT>(b, 0, sg.lists[6].n, sg.lists[6].d_rows);
      launch_split(a, sg.split);
}

// Stream kernel configurations reachable from stream_cfg_for() (the ids are those of the
// round-1 sweeps under profiles/, 35 shapes were tried; these seven won their class):
// {id, consumer threads, lanes/row, stages, cap, passes, entry-split}.  All warp-specialised.
#define STREAM_CONFIGS(X)                                                                          \
      X(10, 256, 2, 2, 4096, 1, false)                                                             \
      X(12, 512, 4, 2, 4096, 1, false)                                                             \
      X(13, 512, 2, 2, 8192, 1, false)                                                             \
      X(24, 256, 1, 2, 4096, 8, true)                                                              \
      X(25, 512, 1, 3, 4096, 2, true)                                                              \
      X(26, 512, 1, 4, 2048, 2, true)                                                              \
      X(33, 256, 1, 2, 2048, 4, true)

struct StreamShape {
      int id, threads, lpr, stages, cap, passes;
      bool split;
};
constexpr StreamShape kStreamShapes[] = {
#define X(id, t, l, s, c, p, sp) {id, t, l, s, c, p, sp},
    STREAM_CONFIGS(X)
#undef X
};
const StreamShape *stream_shape(int cfg) {
      for (const auto &s : kStreamShapes)
            if (s.id == cfg)
                  return &s;
      return nullptr;
}

template <typename Kern>
int stream_occupancy(Kern kern, int threads, size_t smem, int device, int *occ_cache) {
      int &occ = occ_cache[device % kMaxDevices];
      if (!occ) {
            B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem));
            B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
            if (occ < 1)
                  return fail(-EINVAL, "stream kernel does not fit on an SM");
      }
      return 0;
}

// One launch of the staged kernel over the tiles of `sp`, streaming column codes when the plan
// has them (row-tile configurations only) and the csr_codes knob is on.  *grid_out = CTAs
// launched.
template <typename OffT>
int launch_stream_cfg(int cfg, const CsrArgs &a, const StreamPlan &sp, int *grid_out) {
      if (grid_out)
            *grid_out = 0;
      if (sp.n_tiles <= 0)
            return 0;
      const OffT *irp = static_cast<const OffT *>(a.h->d_irp);
      const bool coded = sp.codes_state == 1 && g_knobs.csr_codes != 0;
      switch (cfg) {
#define LAUNCH_ONE(E, T, L, S, C, P, SP, CODES)                                                    \
      {                                                                                            \
            auto kern = csr_stream_kernel<T, L, S, C, P, true, SP, E, CODES, OffT>;                \
            using Cfg = StreamCfg<T, L, S, C, P, true, SP, CODES>;                                 \
            constexpr size_t smem = Cfg::template smem<OffT>();                                    \
            static int occ_by_dev[kMaxDevices] = {0}; /* the attribute is per device */            \
            int rc = stream_occupancy(kern, Cfg::kThreads, smem, a.h->device, occ_by_dev);         \
            if (rc)                                                                                \
                  return rc;                                                                       \
            const int grid =                                                                       \
                std::min(sp.n_tiles, occ_by_dev[a.h->device % kMaxDevices] * g_sm_count);          \
            kern<<<grid, Cfg::kThreads, smem, a.st>>>(irp, a.h->d_ja, a.h->d_as, sp.d_tile_row,    \
                                                      sp.d_tile_k, sp.d_code_off, sp.d_codes, 0,   \
                                                      sp.n_tiles, a.x, a.y, a.epi);                \
            if (grid_out)                                                                          \
                  *grid_out = grid;                                                                \
      }
#define LAUNCH_CODED(E, T, L, S, C, P, SP)                                                         \
      {                                                                                            \
            if (coded && !SP) /* entry-split plans have no codes */                                \
                  LAUNCH_ONE(E, T, L, S, C, P, SP, !SP)                                            \
            else                                                                                   \
                  LAUNCH_ONE(E, T, L, S, C, P, SP, false)                                          \
      }
#define X(id, T, L, S, C, P, SP)                                                                   \
      case id:                                                                                     \
            if (a.epi_mode == EPI_PUSH)                                                            \
                  LAUNCH_CODED(EPI_PUSH, T, L, S, C, P, SP)                                        \
            else if (a.epi_mode == EPI_FUSED)                                                      \
                  LAUNCH_CODED(EPI_FUSED, T, L, S, C, P, SP)                                       \
            else                                                                                   \
                  LAUNCH_CODED(EPI_PLAIN, T, L, S, C, P, SP)                                       \
            break;
            STREAM_CONFIGS(X)
#undef X
#undef LAUNCH_CODED
#undef LAUNCH_ONE
      default:
            return fail(-EINVAL, "unknown stream configuration %d", cfg);
      }
      ++g_counters.launches;
      return 0;
}

// Configuration of the TMA-staged kernel for one segment.  Measured on B200
// (profiles/r1_kbench_*.txt): warp-specialised variants win everywhere; rows of
// ~16+ entries want several lanes per row (more gathers in flight), short rows
// want one thread per row and several passes per tile so a tile still carries
// a few thousand entries.  warps_per_block picks the CTA size within a class.
int stream_cfg_for(int wpb, double mean_len, bool regular) {
      if (g_knobs.csr_stream_cfg >= 0 && stream_shape(g_knobs.csr_stream_cfg))
            return g_knobs.csr_stream_cfg;
      if (!regular) // power-law / ragged: split tiles by entry, not by row (cfg 33: 30 % vs 26 %
                    // for cfg 22 on R-MAT 22, profiles/r1_kbench_rmat22_split_cfgs2.txt)
            return wpb <= 4 ? 33 : 25;
      if (mean_len >= 12.0)
            return wpb <= 2 ? 10 : (wpb <= 4 ? 12 : 13);
      // short rows (5-point stencils ...): the entry-split tiles win here too -- 70 % vs 59 % of
      // peak on a 3000^2 Poisson matrix (profiles/r1_kbench_poisson3000.txt)
      return wpb <= 2 ? 24 : 26;
}

int ensure_dot(double **buf, long long *cap, long long n) {
      if (n <= *cap)
            return 0;
      cudaFree(*buf);
      *buf = nullptr, *cap = 0;
      B200_CUDA(cudaMalloc(buf, (size_t)n * sizeof(double)));
      *cap = n;
      return 0;
}

} // namespace

// =================================================================== SELL-P
namespace {

// Gather locality: how much of x does a block of 256 consecutive rows span?  Median over up to
// 64 sampled blocks, as a fraction of N.  Stencils and banded matrices: ~0; uniform random
// columns: ~1.
template <typename Src>
double measure_gather_span(const Src &src, long long M, long long N) {
      if (M <= 0 || N <= 0)
            return 0.0;
      constexpr int kSamples = 64;
      constexpr long long kBlock = 256;
      const int n = (int)std::min<long long>(kSamples, (M + kBlock - 1) / kBlock);
      const long long stride = std::max<long long>(kBlock, M / n / kBlock * kBlock);
      DeviceTemps tmp;
      int *d_lo = nullptr, *d_hi = nullptr;
      if (tmp.alloc(&d_lo, n * sizeof(int), "gather span") || tmp.alloc(&d_hi, n * sizeof(int), "gather span"))
            return 0.0;
      col_extent_kernel<<<n, 256>>>(src, M, kBlock, stride, n, d_lo, d_hi);
      std::vector<int> lo(n), hi(n);
      cudaMemcpy(lo.data(), d_lo, n * sizeof(int), cudaMemcpyDeviceToHost);
      cudaMemcpy(hi.data(), d_hi, n * sizeof(int), cudaMemcpyDeviceToHost);
      if (cudaGetLastError() != cudaSuccess)
            return 0.0;
      std::vector<double> span;
      for (int i = 0; i < n; ++i)
            span.push_back(hi[i] >= lo[i] ? (double)(hi[i] - lo[i] + 1) / (double)N : 0.0);
      std::sort(span.begin(), span.end());
      return span[span.size() / 2];
}

int sell_panels_for(long long N, double gather_span) {
      if (g_knobs.sell_panels > 0)
            return std::min(64, g_knobs.sell_panels);
      const double x_mb = (double)N * 8.0 / (1 << 20);
      // x fits the L2 beside the matrix streams, or the rows only touch a narrow band of it
      if (x_mb <= 48.0 || gather_span * x_mb <= 24.0)
            return 1;
      const int k = (int)((x_mb + g_knobs.sell_panel_mb - 1) / g_knobs.sell_panel_mb);
      return std::max(1, std::min(64, k));
}

// Host part of the build: per panel and window, order the rows by their entry count
// (descending, ties by row index -- a stable counting sort), emit perm and the slice offsets.
void sell_plan_host(const std::vector<int> &counts, long long M, int K, int sigma,
                    std::vector<int> &perm, std::vector<long long> &soff, long long *nnz_in,
                    std::vector<int> *long_rows) {
      const long long S = (M + 31) / 32;
      perm.assign((size_t)K * S * 32, -1);
      std::vector<long long> width((size_t)K * S, 0);
      const long long n_win = (M + sigma - 1) / sigma;
      long long nnz_total = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : nnz_total) collapse(2)
      for (int p = 0; p < K; ++p) {
            for (long long w = 0; w < n_win; ++w) {
                  const long long r0 = w * sigma, r1 = std::min(M, r0 + sigma);
                  const int *cnt = counts.data() + (size_t)p * M;
                  int maxc = 0;
                  for (long long r = r0; r < r1; ++r)
                        maxc = std::max(maxc, cnt[r]);
                  // bucket b holds the rows with count maxc - b; excluded rows (-1) come last
                  std::vector<int> start((size_t)maxc + 3, 0);
                  for (long long r = r0; r < r1; ++r)
                        ++start[(size_t)(cnt[r] < 0 ? maxc + 1 : maxc - cnt[r]) + 1];
                  for (size_t b = 1; b < start.size(); ++b)
                        start[b] += start[b - 1];
                  const long long base = ((long long)p * S + r0 / 32) * 32;
                  for (long long r = r0; r < r1; ++r) {
                        const size_t b = (size_t)(cnt[r] < 0 ? maxc + 1 : maxc - cnt[r]);
                        const int pos = start[b]++;
                        if (cnt[r] >= 0) {
                              perm[(size_t)(base + pos)] = (int)r;
                              nnz_total += cnt[r];
                        }
                  }
                  // slice width = count of its first (longest) row
                  for (long long s = r0 / 32; s < (r1 + 31) / 32; ++s) {
                        const int first = perm[(size_t)(((long long)p * S + s) * 32)];
                        width[(size_t)p * S + s] = first >= 0 ? cnt[first] : 0;
                  }
            }
      }
      *nnz_in = nnz_total;
      soff.assign((size_t)K * (S + 1), 0);
      long long run = 0;
      for (int p = 0; p < K; ++p) {
            for (long long s = 0; s < S; ++s) {
                  soff[(size_t)p * (S + 1) + s] = run;
                  run += 32 * width[(size_t)p * S + s];
            }
            soff[(size_t)p * (S + 1) + S] = run;
      }
      if (long_rows) {
            long_rows->clear();
            for (long long r = 0; r < M; ++r)
                  if (counts[r] < 0)
                        long_rows->push_back((int)r);
      }
}

template <typename Src>
int sell_build(const Src &src, long long M, long long N, int K, int max_row, SellPlan &sp,
               std::vector<int> *long_rows) {
      if (M <= 0 || M >= (1ll << 31) - 64)
            return 0;
      const int sigma = std::max(32, g_knobs.sell_sigma / 32 * 32);
      const long long S = (M + 31) / 32;
      PanelBounds pb{};
      pb.K = K;
      for (int p = 0; p <= K; ++p)
            pb.pc[p] = (int)(N * p / K);
      sp.pc.assign(pb.pc, pb.pc + K + 1);

      DeviceTemps tmp;
      int *d_counts = nullptr;
      if (tmp.alloc(&d_counts, (size_t)K * M * sizeof(int), "SELL row counts"))
            return -ENOMEM;
      sell_count_kernel<<<blocks_for(M, 256), 256>>>(src, M, pb, max_row, d_counts);
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess)
            return fail(-EIO, "SELL count kernel launch failed: %s", cudaGetErrorString(e));
      std::vector<int> counts((size_t)K * M);
      e = cudaMemcpy(counts.data(), d_counts, counts.size() * sizeof(int), cudaMemcpyDeviceToHost);
      tmp.release_all();
      if (e != cudaSuccess)
            return fail(-EIO, "SELL row counts failed: %s", cudaGetErrorString(e));
      g_counters.launches += 1;
      g_counters.d2h += (long long)counts.size() * 4;

      std::vector<int> perm;
      std::vector<long long> soff;
      sell_plan_host(counts, M, K, sigma, perm, soff, &sp.nnz_in_slices, long_rows);
      sp.K = K, sp.sigma = sigma, sp.M = M, sp.n_slices = S;
      sp.slots = soff.back();
      int rc = upload(&sp.d_perm, perm);
      rc = rc ? rc : upload(&sp.d_soff, soff);
      if (rc)
            return rc;
      B200_CUDA(cudaMalloc(&sp.d_ja, ((size_t)sp.slots + 32) * sizeof(int)));
      B200_CUDA(cudaMalloc(&sp.d_as, ((size_t)sp.slots + 32) * sizeof(double)));
      sell_fill_kernel<<<blocks_for(S * K * 32, 256), 256>>>(src, S, pb, sp.d_soff, sp.d_perm,
                                                             sp.d_ja, sp.d_as);
      g_counters.launches += 1;
      e = cudaDeviceSynchronize();
      if (e != cudaSuccess)
            return fail(-EIO, "SELL fill kernel failed: %s", cudaGetErrorString(e));
      sp.state = 1;
      return 0;
}

// Virtual rows of a ragged CSR (see sell_kernels.cuh): rows longer than `chunk` become
// ceil(len / chunk) pieces.  vr_row / vr_j0 describe the pieces, dest[v] where a piece stores
// (row, or -2-i for partial i), split_row / split_first the rows whose partials are combined.
void sell_virtual_rows(const std::vector<long long> &irp, long long M, int chunk,
                       std::vector<int> &vr_row, std::vector<int> &vr_j0, std::vector<int> &vr_len,
                       std::vector<int> &dest, std::vector<int> &split_row,
                       std::vector<int> &split_first) {
      long long V = 0, P = 0;
      for (long long r = 0; r < M; ++r) {
            const long long len = irp[r + 1] - irp[r];
            const long long pieces = len > chunk ? (len + chunk - 1) / chunk : 1;
            V += pieces;
            P += pieces > 1 ? pieces : 0;
      }
      vr_row.resize((size_t)V), vr_j0.resize((size_t)V), vr_len.resize((size_t)V), dest.resize((size_t)V);
      split_row.clear(), split_first.clear();
      long long v = 0, p = 0;
      for (long long r = 0; r < M; ++r) {
            const long long len = irp[r + 1] - irp[r];
            if (len <= chunk) {
                  vr_row[v] = (int)r, vr_j0[v] = 0, vr_len[v] = (int)len, dest[v] = (int)r;
                  ++v;
                  continue;
            }
            split_row.push_back((int)r);
            split_first.push_back((int)p);
            for (long long j0 = 0; j0 < len; j0 += chunk, ++v, ++p) {
                  vr_row[v] = (int)r, vr_j0[v] = (int)j0;
                  vr_len[v] = (int)std::min<long long>(chunk, len - j0);
                  dest[v] = (int)(-2 - p);
            }
      }
      split_first.push_back((int)p);
}

template <typename Src>
int sell_build_vrows(const Src &src, const std::vector<long long> &irp, long long M, long long N,
                     int chunk, SellPlan &sp) {
      if (M <= 0 || irp[M] + M >= (1ll << 31) - 64)
            return 0;
      const int sigma = std::max(32, g_knobs.sell_sigma / 32 * 32);
      std::vector<int> vr_row, vr_j0, vr_len, dest, split_row, split_first;
      sell_virtual_rows(irp, M, chunk, vr_row, vr_j0, vr_len, dest, split_row, split_first);
      const long long V = (long long)vr_row.size(), S = (V + 31) / 32;
      std::vector<int> perm_v;
      std::vector<long long> soff;
      sell_plan_host(vr_len, V, 1, sigma, perm_v, soff, &sp.nnz_in_slices, nullptr);
      std::vector<int> perm_dest(perm_v.size());
      for (size_t i = 0; i < perm_v.size(); ++i)
            perm_dest[i] = perm_v[i] >= 0 ? dest[perm_v[i]] : -1;
      sp.K = 1, sp.sigma = sigma, sp.M = V, sp.n_slices = S, sp.chunk = chunk, sp.n_rows = M;
      sp.pc = {0, (int)N};
      sp.slots = soff.back();
      sp.n_split_rows = (long long)split_row.size();
      sp.n_partials = split_first.back();
      static const char *what = "SELL virtual rows";
      DeviceTemps tmp;
      int *d_perm_v = nullptr, *d_vr_row = nullptr, *d_vr_j0 = nullptr;
      int rc = tmp.upload(&d_perm_v, perm_v, what);
      rc = rc ? rc : tmp.upload(&d_vr_row, vr_row, what);
      rc = rc ? rc : tmp.upload(&d_vr_j0, vr_j0, what);
      rc = rc ? rc : upload(&sp.d_perm, perm_dest);
      rc = rc ? rc : upload(&sp.d_soff, soff);
      if (!rc && sp.n_split_rows) {
            rc = upload(&sp.d_split_row, split_row);
            rc = rc ? rc : upload(&sp.d_split_first, split_first);
            if (!rc && cudaMalloc(&sp.d_partial, (size_t)sp.n_partials * sizeof(double)) != cudaSuccess)
                  rc = fail(-ENOMEM, "SELL partial sums: out of device memory");
      }
      if (!rc && (cudaMalloc(&sp.d_ja, ((size_t)sp.slots + 32) * sizeof(int)) != cudaSuccess ||
                  cudaMalloc(&sp.d_as, ((size_t)sp.slots + 32) * sizeof(double)) != cudaSuccess))
            rc = fail(-ENOMEM, "SELL slices: out of device memory");
      if (rc)
            return rc;
      sell_fill_vrow_kernel<<<blocks_for(S * 32, 256), 256>>>(src, S, sp.d_soff, d_perm_v, d_vr_row, d_vr_j0,
                                                              chunk, sp.d_ja, sp.d_as);
      g_counters.launches += 1;
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess)
            return fail(-EIO, "SELL fill kernel failed: %s", cudaGetErrorString(e));
      sp.state = 1;
      return 0;
}

// y = A x through the panels: panel 0 stores, later panels accumulate (stream order).
int sell_run(const SellPlan &sp, int wpb, const double *d_x, double *d_y, int epi_mode,
             const EpiArgs &epi, cudaStream_t st, int blocks = 0,
             const std::function<void(long long, long long)> *block_done = nullptr) {
      const int threads = 32 * wpb;
      const int grid = blocks_for(sp.n_slices * 32, threads);
      if (sp.chunk > 0) { // virtual rows: one panel, pieces of split rows go to partial sums
            if (epi_mode == EPI_FUSED)
                  sell_kernel<EPI_FUSED, true><<<grid, threads, 0, st>>>(
                      sp.d_soff, sp.d_perm, sp.d_ja, sp.d_as, sp.n_slices, d_x, d_y, sp.d_partial, epi);
            else
                  sell_kernel<EPI_PLAIN, true><<<grid, threads, 0, st>>>(
                      sp.d_soff, sp.d_perm, sp.d_ja, sp.d_as, sp.n_slices, d_x, d_y, sp.d_partial, epi);
            ++g_counters.launches;
            if (sp.n_split_rows) {
                  csr_combine_kernel<EPI_PLAIN><<<blocks_for(sp.n_split_rows, 128), 128, 0, st>>>(
                      sp.d_split_row, sp.d_split_first, (int)sp.n_split_rows, sp.d_partial, d_y, EpiArgs{});
                  ++g_counters.launches;
            }
            return 0;
      }
      // The last panel may run as `blocks` launches over runs of whole windows, `block_done(r0, r1)`
      // called after each: rows [r0, r1) of y are final from then on in stream order (rows never
      // leave their window).  The multi-GPU all-gather sends finished blocks while later ones compute.
      const int n_blocks = block_done && blocks ? std::max(1, blocks) : 1;
      const long long win_slices = std::max<long long>(1, sp.sigma / 32);
      const long long n_win = (sp.n_slices + win_slices - 1) / win_slices;
      for (int p = 0; p < sp.K; ++p)
            for (int b = 0; b < (p == sp.K - 1 ? n_blocks : 1); ++b) {
            const bool last = p == sp.K - 1;
            const long long s0 = last ? std::min(sp.n_slices, n_win * b / n_blocks * win_slices) : 0;
            const long long s1 = last ? std::min(sp.n_slices, n_win * (b + 1) / n_blocks * win_slices) : sp.n_slices;
            if (s1 <= s0)
                  continue;
            const long long *soff = sp.d_soff + (size_t)p * (sp.n_slices + 1) + s0;
            const int *perm = sp.d_perm + ((size_t)p * sp.n_slices + s0) * 32;
            const long long ns = s1 - s0;
            const int grid = blocks_for(ns * 32, threads);
            const bool push = epi_mode == EPI_PUSH && last; // finished sums also go to the peers
#define SELL_LAUNCH(E)                                                                             \
      sell_kernel<E><<<grid, threads, 0, st>>>(soff, perm, sp.d_ja, sp.d_as, ns, d_x, d_y, nullptr, epi)
            if (push && p > 0)
                  SELL_LAUNCH(EPI_ACC_PUSH);
            else if (push)
                  SELL_LAUNCH(EPI_PUSH);
            else if (p > 0)
                  SELL_LAUNCH(EPI_ACC);
            else if (epi_mode == EPI_FUSED)
                  SELL_LAUNCH(EPI_FUSED);
            else
                  SELL_LAUNCH(EPI_PLAIN);
#undef SELL_LAUNCH
            ++g_counters.launches;
            if (last && block_done && blocks)
                  (*block_done)(s0 * 32, std::min(sp.M, s1 * 32));
      }
      return 0;
}

// Should ids 2 / 4 of this CSR go through SELL-P?  (whole-matrix calls on single-segment handles)
bool csr_wants_sell(spmv_b200_csr *h) {
      if (g_knobs.sell == 0 || h->segs.size() != 1 || h->M < 64)
            return false;
      if (g_knobs.sell == 1)
            return true;
      const Segment &sg = h->segs[0];
      if (!sg.regular)
            return true; // ragged / power-law rows: sorted slices instead of per-bin row lists
      // regular rows, but x is too large for the L2 and the columns are scattered
      return sell_panels_for(h->N, h->gather_span) > 1;
}

// A plan not built (not applicable, or a step failed) holds no device memory and is not tried again.
int sell_not_built(SellPlan &plan) {
      free_sell(plan);
      plan.state = -1;
      return -1;
}

// `rhs` right-hand sides share one pass (SpMM): the x a panel must keep in the L2 is rhs times as large
int csr_build_sell(spmv_b200_csr *h, SellPlan &plan, int rhs) {
      if (plan.state != 0)
            return plan.state == 1 ? 0 : -1;
      // Ragged / power-law rows take ONE panel whatever the size of x: their columns are as
      // skewed as their rows (R-MAT: a few hot columns serve most gathers), panels measured no
      // gain there and cost a pass over y and the row order each (profiles/r2_kbench_c4_sell.txt).
      const bool ragged = !h->segs.empty() && !h->segs[0].regular;
      const int K = ragged && g_knobs.sell_panels <= 0 ? 1 : sell_panels_for(h->N * rhs, h->gather_span);
      // virtual rows: ragged matrices, or any one-panel plan when SELL-P is forced by the knob
      const bool vrows =
          (ragged || g_knobs.sell == 1) && K == 1 && g_knobs.sell_panels <= 0 && g_knobs.sell_chunk > 0;
      std::vector<int> long_rows; // stays empty for virtual rows: no row is too long for them
      const int rc = with_offsets(h->wide, [&](auto t) {
            using OffT = typename decltype(t)::type;
            const CsrSrc<OffT> src{(const OffT *)h->d_irp, h->d_ja, h->d_as};
            return vrows ? sell_build_vrows(src, h->h_irp, h->M, h->N, g_knobs.sell_chunk, plan)
                         : sell_build(src, h->M, h->N, K, g_knobs.sell_max_row, plan, &long_rows);
      });
      if (rc || plan.state != 1)
            return sell_not_built(plan);
      // rows too long for a slice: a warp per row up to 2048 entries, a CTA per row up to 65 536,
      // split into chunks beyond (the bins of the direct path)
      std::vector<int> wrp, blk, spl;
      for (int r : long_rows) {
            const long long len = h->h_irp[r + 1] - h->h_irp[r];
            (len <= kKindMax[5] ? wrp : (len <= kKindMax[6] ? blk : spl)).push_back(r);
      }
      plan.n_long = (long long)long_rows.size();
      plan.long_warp.n = (long long)wrp.size();
      plan.long_block.n = (long long)blk.size();
      if (upload(&plan.long_warp.d_rows, wrp) || upload(&plan.long_block.d_rows, blk) ||
          build_split(h, spl, plan.long_split))
            return sell_not_built(plan);
      return 0;
}

int csr_ensure_sell(spmv_b200_csr *h) { return csr_build_sell(h, h->sell, 1); }

} // namespace

// ================================================================== routing
namespace b200 {

// 0 launched, < 0 error.  CAPW = entries a warp's buffer holds: 32 rows of at most MAXROW entries,
// rounded out to multiples of 4 at both ends.  Two sizes: rows <= 5 (5-point stencils: 4.2 KB per
// warp, 48 warps per SM) and rows <= 8 (6.5 KB, 32 warps).
template <typename OffT, int MAXROW>
static int launch_csr_pipe_cap(const CsrArgs &a, long long r0, long long r1) {
      constexpr int kStages = 2, kWarps = 8;
      constexpr int capw = 32 * MAXROW + 16;
      constexpr size_t smem = (size_t)kWarps * kStages * capw * 12 + (size_t)kWarps * kStages * 8;
      auto kern = csr_pipe_kernel<kStages, capw, OffT>;
      static int occ_by_dev[kMaxDevices] = {0};
      int &occ = occ_by_dev[a.h->device % kMaxDevices];
      if (!occ) {
            B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kWarps * 32, smem));
            if (occ < 1)
                  return fail(-EINVAL, "csr_pipe_kernel does not fit on an SM");
      }
      if (r1 - r0 >= (1ll << 31) - 64)
            return fail(-EINVAL, "csr_pipe_kernel: more than 2^31 rows in one segment");
      const long long groups = (r1 - r0 + 31) / 32;
      const int g = (int)std::min<long long>((groups + kWarps - 1) / kWarps, (long long)occ * g_sm_count);
      kern<<<g, kWarps * 32, smem, a.st>>>((const OffT *)a.h->d_irp, a.h->d_ja, a.h->d_as, r0, (int)(r1 - r0), a.x, a.y);
      ++g_counters.launches;
      return 0;
}
template <typename OffT>
static int launch_csr_pipe(const CsrArgs &a, const Segment &sg) {
      return sg.max_len <= 5 ? launch_csr_pipe_cap<OffT, 5>(a, sg.r0, sg.r1)
                             : launch_csr_pipe_cap<OffT, kCsrPipeMaxRow>(a, sg.r0, sg.r1);
}

constexpr long long kStreamDotSlots = 32768; // >= CTAs * consumer warps of any stream launch

template <typename OffT>
static int run_kernel(spmv_b200_csr *h, int kernel, int wpb, Segment &sg, const CsrArgs &a) {
      if (a.epi_mode == EPI_FUSED && kernel != SPMV_B200_CSR_ADAPTIVE &&
          kernel != SPMV_B200_CSR_STREAM)
            return fail(-ENOTSUP, "the fused epilogue exists for CSR kernels 2 and 4 only");
      switch (kernel) {
      case SPMV_B200_CSR_THREAD_ROW:
            launch_vec<OffT>(a, 0, sg.r0, sg.r1 - sg.r0, nullptr, -1);
            return 0;
      case SPMV_B200_CSR_WARP_ROW:
            launch_vec<OffT>(a, 5, sg.r0, sg.r1 - sg.r0, nullptr, -1);
            return 0;
      case SPMV_B200_CSR_ADAPTIVE:
            // Adaptive = per segment, the kernel family that measures best for its row-length
            // profile: a regular segment (one length bin holds >= 90 % of the rows) streams
            // through the TMA-staged tile kernel, which also bins its own long rows; an
            // irregular one goes through the direct binned kernels (whole irregular matrices
            // never get here: csr_run routes them to the sorted slices of SELL-P).
            if (a.epi_mode != EPI_FUSED && !sg.regular) {
                  int rc = build_bin_lists(h, sg);
                  if (rc)
                        return rc;
                  run_adaptive<OffT>(a, sg);
                  return 0;
            }
            return run_kernel<OffT>(h, SPMV_B200_CSR_STREAM, wpb, sg, a);
      case SPMV_B200_CSR_BLOCK_ROW:
            launch_block_rows<OffT>(a, sg.r0, sg.r1 - sg.r0, nullptr);
            return 0;
      case SPMV_B200_CSR_STREAM: {
            // short regular rows: persistent warps with private bulk-copy rings (csr_pipe_kernel)
            if (a.epi_mode == EPI_PLAIN && g_knobs.csr_pipe != 0 && g_knobs.csr_stream_cfg < 0 &&
                sg.r1 > sg.r0 && sg.r1 - sg.r0 < (1ll << 31) - 64 && sg.max_len <= kCsrPipeMaxRow &&
                (g_knobs.csr_pipe > 0 || (sg.regular && sg.r1 - sg.r0 >= 32ll * 4 * g_sm_count * 8))) {
                  return launch_csr_pipe<OffT>(a, sg);
            }
            const double mean_len = sg.r1 > sg.r0 ? (double)(h->h_irp[sg.r1] - h->h_irp[sg.r0]) /
                                                        (double)(sg.r1 - sg.r0)
                                                  : 0.0;
            const int cfg = stream_cfg_for(wpb, mean_len, sg.regular);
            StreamPlan &sp = sg.stream[cfg];
            const StreamShape &s = *stream_shape(cfg);
            if (!sp.built) {
                  int rc = build_stream(h, sg, s.threads / s.lpr * s.passes, s.cap, sp);
                  if (rc)
                        return rc;
            }
            if (!s.split && g_knobs.csr_codes != 0 && sp.codes_state == 0) {
                  int rc = build_codes<OffT>(h, s.cap, sp);
                  if (rc)
                        return rc;
            }
            if (a.epi_mode == EPI_FUSED &&
                (sp.long_lists[5].n || sp.long_lists[6].n || sp.split.n_rows))
                  return fail(-ENOTSUP, "fused epilogue: the matrix has rows longer than a stage");
            int rc = launch_stream_cfg<OffT>(cfg, a, sp, nullptr);
            if (rc)
                  return rc;
            launch_long_lists<OffT>(a, sp.long_lists, sp.split);
            return 0;
      }
      default:
            return fail(-EINVAL, "unknown CSR kernel id %d", kernel);
      }
}

int csr_run_segment(spmv_b200_csr *h, Segment &sg, int kernel, int wpb, const double *d_x,
                    double *d_y, int epi_mode, const EpiArgs &epi, cudaStream_t st) {
      CsrArgs a{h, d_x, d_y, epi_mode, epi, st, 32 * wpb};
      return h->wide ? run_kernel<long long>(h, kernel, wpb, sg, a)
                     : run_kernel<int>(h, kernel, wpb, sg, a);
}

int csr_run(spmv_b200_csr *h, int kernel, int wpb, long long row0, long long row1,
            const double *d_x, double *d_y, int epi_mode, const EpiArgs &epi_in, void *stream) {
      if (!h)
            return fail(-EINVAL, "null CSR handle");
      wpb = clamp_wpb(wpb);
      cudaStream_t st = as_stream(stream);
      EpiArgs epi = epi_in;
      const bool whole = row0 == 0 && row1 == h->M;
      const bool want_dot = epi_mode == EPI_FUSED && epi.w && epi.dot_partial; // dot_partial = out
      double *dot_out = epi.dot_partial;
      long long dot_slots = 0;
      if (epi_mode == EPI_FUSED) {
            if (!whole || h->segs.size() > 1)
                  return fail(-ENOTSUP, "fused epilogue: whole-matrix calls on uncut handles only");
            epi.dot_partial = nullptr;
      }

      const bool sell_kernel_id = kernel == SPMV_B200_CSR_ADAPTIVE || kernel == SPMV_B200_CSR_STREAM;
      // (the push epilogue exists for the panel form without long-row kernels: the shards of a
      // general matrix whose next x slice every peer needs)
      if (sell_kernel_id && whole && csr_wants_sell(h) &&
          (epi_mode != EPI_PUSH || (h->segs[0].regular && g_knobs.sell != 1)) && csr_ensure_sell(h) == 0 &&
          (epi_mode != EPI_PUSH || (h->sell.chunk == 0 && h->sell.n_long == 0))) {
            const SellPlan &sp = h->sell;
            if (epi_mode == EPI_FUSED) {
                  if (sp.K > 1 || sp.n_long || sp.n_split_rows)
                        return fail(-ENOTSUP, "fused epilogue: not available on column panels or "
                                              "split rows");
                  if (want_dot) {
                        if (ensure_dot(&h->d_dot_partial, &h->dot_cap, sp.n_slices))
                              return -ENOMEM;
                        epi.dot_partial = h->d_dot_partial;
                        dot_slots = sp.n_slices;
                  }
            }
            sell_run(sp, wpb, d_x, d_y, epi_mode, epi, st);
            CsrArgs a{h, d_x, d_y, EPI_PLAIN, EpiArgs{}, st, 512};
            CsrArgs aw = a;
            aw.threads = 256;
            if (h->wide) {
                  launch_vec<long long>(aw, 5, 0, sp.long_warp.n, sp.long_warp.d_rows, -1);
                  launch_block_rows<long long>(a, 0, sp.long_block.n, sp.long_block.d_rows);
            } else {
                  launch_vec<int>(aw, 5, 0, sp.long_warp.n, sp.long_warp.d_rows, -1);
                  launch_block_rows<int>(a, 0, sp.long_block.n, sp.long_block.d_rows);
            }
            launch_split(a, sp.long_split);
      } else {
            if (want_dot) {
                  if (ensure_dot(&h->d_dot_partial, &h->dot_cap, kStreamDotSlots))
                        return -ENOMEM;
                  B200_CUDA(cudaMemsetAsync(h->d_dot_partial, 0, kStreamDotSlots * sizeof(double), st));
                  epi.dot_partial = h->d_dot_partial;
                  dot_slots = kStreamDotSlots;
            }
            // the requested range must be exactly a run of the segments declared at creation
            long long covered = 0;
            for (auto &sg : h->segs) {
                  if (sg.r0 < row0 || sg.r1 > row1 || sg.r1 == sg.r0)
                        continue;
                  covered += sg.r1 - sg.r0;
            }
            if (covered != row1 - row0 || row0 < 0 || row1 > h->M)
                  return fail(-EINVAL,
                              "rows [%lld,%lld) do not match the cut points given at creation", row0,
                              row1);
            for (auto &sg : h->segs) {
                  if (sg.r0 < row0 || sg.r1 > row1 || sg.r1 == sg.r0)
                        continue;
                  int rc = csr_run_segment(h, sg, kernel, wpb, d_x, d_y, epi_mode, epi, st);
                  if (rc)
                        return rc;
            }
      }
      if (want_dot) {
            dot_reduce_kernel<<<1, 1024, 0, st>>>(h->d_dot_partial, dot_slots, dot_out);
            ++g_counters.launches;
      }
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess)
            return fail(-EIO, "CSR kernel %d launch failed: %s", kernel, cudaGetErrorString(e));
      return 0;
}

// y = A x over the whole matrix, plain epilogue, with `done(r0, r1)` called as soon as rows
// [r0, r1) of y are final in stream order: in up to `blocks` pieces where the route allows it (the
// column-panel form of SELL-P: the last panel runs window range by window range), once at the end
// otherwise.  The multi-GPU all-gather hands finished pieces to the copy engines while the rest
// of the step still computes.
int csr_run_blocks(spmv_b200_csr *h, int kernel, int wpb, const double *d_x, double *d_y, void *stream,
                   int blocks, const std::function<void(long long, long long)> &done) {
      if (!h)
            return fail(-EINVAL, "null CSR handle");
      const bool sell_kernel_id = kernel == SPMV_B200_CSR_ADAPTIVE || kernel == SPMV_B200_CSR_STREAM;
      if (blocks > 1 && sell_kernel_id && csr_wants_sell(h) && csr_ensure_sell(h) == 0 &&
          h->sell.chunk == 0 && h->sell.n_long == 0) {
            int rc = sell_run(h->sell, clamp_wpb(wpb), d_x, d_y, EPI_PLAIN, EpiArgs{}, as_stream(stream), blocks, &done);
            cudaError_t e = cudaGetLastError();
            if (!rc && e != cudaSuccess)
                  rc = fail(-EIO, "SELL-P launch failed: %s", cudaGetErrorString(e));
            return rc;
      }
      int rc = csr_run(h, kernel, wpb, 0, h->M, d_x, d_y, EPI_PLAIN, EpiArgs{}, stream);
      if (!rc)
            done(0, h->M);
      return rc;
}

// Largest column referenced by entries [k0, k1): a device reduction (the host-buffer pipeline
// needs it for matrices that were generated on the device and have no host copy).
static __global__ void max_col_kernel(const int *__restrict__ ja, long long k0, long long k1,
                                      int *__restrict__ out) {
      int mx = -1;
      for (long long k = k0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; k < k1;
           k += (long long)gridDim.x * blockDim.x)
            mx = max(mx, ja[k]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
            mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if ((threadIdx.x & 31) == 0 && mx >= 0)
            atomicMax(out, mx);
}

// Smallest and largest stored (local) column index: a shard whose columns fall outside
// [0, n_local) would make every kernel gather out of bounds.
static __global__ void col_minmax_kernel(const int *__restrict__ ja, long long n,
                                         int *__restrict__ out) {
      int mn = 0x7fffffff, mx = -0x7fffffff - 1;
      for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n;
           k += (long long)gridDim.x * blockDim.x) {
            const int c = ja[k];
            mn = min(mn, c), mx = max(mx, c);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
            mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      }
      if ((threadIdx.x & 31) == 0) {
            atomicMin(out, mn);
            atomicMax(out + 1, mx);
      }
}

int csr_check_columns(const spmv_b200_csr *h) {
      if (h->NZ == 0)
            return 0;
      DeviceTemps tmp;
      int *d = nullptr;
      const int init[2] = {0x7fffffff, -0x7fffffff - 1};
      int got[2];
      if (tmp.alloc(&d, sizeof init, "column check"))
            return -ENOMEM;
      B200_CUDA(cudaMemcpy(d, init, sizeof init, cudaMemcpyHostToDevice));
      col_minmax_kernel<<<(int)std::min<long long>(1184, (h->NZ + 255) / 256), 256>>>(h->d_ja, h->NZ, d);
      cudaError_t e = cudaMemcpy(got, d, sizeof got, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess)
            return fail(-EIO, "column check failed: %s", cudaGetErrorString(e));
      if (got[0] < 0 || got[1] >= h->N)
            return fail(-ERANGE, "column indices span [%lld, %lld] but the x slice covers [%lld, %lld)",
                        (long long)got[0] + h->col_offset, (long long)got[1] + h->col_offset,
                        h->col_offset, h->col_offset + h->N);
      return 0;
}

static int max_col_range(const int *d_ja, long long k0, long long k1, int *out) {
      static int *d_out[kMaxDevices] = {nullptr};
      int dev = 0;
      cudaGetDevice(&dev);
      int *&slot = d_out[dev % kMaxDevices];
      if (!slot)
            B200_CUDA(cudaMalloc(&slot, sizeof(int)));
      const int init = -1;
      B200_CUDA(cudaMemcpy(slot, &init, sizeof(int), cudaMemcpyHostToDevice));
      if (k1 > k0) {
            const int grid = (int)std::min<long long>(1184, (k1 - k0 + 255) / 256);
            max_col_kernel<<<grid, 256>>>(d_ja, k0, k1, slot);
      }
      B200_CUDA(cudaMemcpy(out, slot, sizeof(int), cudaMemcpyDeviceToHost));
      return 0;
}

int csr_max_col(const spmv_b200_csr *h, long long k0, long long k1, int *out) {
      return max_col_range(h->d_ja, k0, k1, out);
}
int hll_max_col(const spmv_b200_hll *h, long long hack0, long long hack1, int *out) {
      return max_col_range(h->d_ja, h->h_hoff[hack0], h->h_hoff[hack1], out);
}

} // namespace b200

// --------------------------------------------------------------- creation --

static void csr_measure_span(spmv_b200_csr *h) {
      h->gather_span = with_offsets(h->wide, [&](auto t) {
            using OffT = typename decltype(t)::type;
            return measure_gather_span(CsrSrc<OffT>{(const OffT *)h->d_irp, h->d_ja, h->d_as}, h->M, h->N);
      });
}

// Planning needs the row offsets on the host: h_irp = the M + 1 offsets of d_irp (the device work
// that wrote them has finished).  64-bit offsets come down in place, 32-bit ones through a copy.
static int download_row_offsets(spmv_b200_csr *h, const char *what) {
      h->h_irp.resize((size_t)h->M + 1);
      std::vector<int> narrow(h->wide ? 0 : h->h_irp.size());
      void *dst = h->wide ? (void *)h->h_irp.data() : (void *)narrow.data();
      cudaError_t e = cudaMemcpy(dst, h->d_irp, h->h_irp.size() * (h->wide ? 8 : 4), cudaMemcpyDeviceToHost);
      if (e != cudaSuccess)
            return fail(-EIO, "%s: row offsets download failed: %s", what, cudaGetErrorString(e));
      std::copy(narrow.begin(), narrow.end(), h->h_irp.begin());
      return 0;
}

// Every constructor returns through here once its shell exists.  rc != 0: the fill failed (fail()
// has set the message), so the shell is destroyed.  Otherwise the row offsets come down to the host
// unless the constructor built them there (h_irp is empty until then), and the handle is planned.
static spmv_b200_csr *csr_finish(spmv_b200_csr *h, int rc, const int64_t *cuts, int n_cuts,
                                 const char *what) {
      if (!rc && h->h_irp.empty())
            rc = download_row_offsets(h, what);
      if (rc || finish_create(h, reinterpret_cast<const long long *>(cuts), n_cuts)) {
            spmv_b200_csr_destroy(h);
            return nullptr;
      }
      csr_measure_span(h);
      return h;
}

// A new handle whose row offsets and slack entries are zeroed on `st`, the stream its fill runs on,
// so the fill is ordered after the zeroing without a synchronisation.
static spmv_b200_csr *csr_alloc_shell(long long M, long long n_local, long long NZ,
                                      long long col_offset, cudaStream_t st) {
      if (ensure_device())
            return nullptr;
      if (M < 0 || n_local < 0 || NZ < 0 || M >= (1ll << 31) - 64) {
            fail(-EINVAL, "bad CSR shape M=%lld N=%lld NZ=%lld", M, n_local, NZ);
            return nullptr;
      }
      auto *h = new spmv_b200_csr();
      h->M = M, h->N = n_local, h->NZ = NZ, h->col_offset = col_offset;
      h->wide = g_knobs.force_wide || NZ >= (1ll << 31) - 64;
      cudaGetDevice(&h->device);
      // +8 entries of slack: the entry-split kernel bulk-copies row offsets in 16-byte units
      const size_t irp_bytes = (size_t)(M + 1 + 8) * (h->wide ? 8 : 4);
      // +16 entries of slack: bulk copies round the entry range out to x4
      if (cudaMalloc(&h->d_irp, irp_bytes) != cudaSuccess ||
          cudaMalloc(&h->d_ja, ((size_t)NZ + 16) * sizeof(int)) != cudaSuccess ||
          cudaMalloc(&h->d_as, ((size_t)NZ + 16) * sizeof(double)) != cudaSuccess) {
            fail(-ENOMEM, "cudaMalloc failed for CSR M=%lld NZ=%lld: %s", M, NZ,
                 cudaGetErrorString(cudaGetLastError()));
            spmv_b200_csr_destroy(h);
            return nullptr;
      }
      cudaError_t e = cudaMemsetAsync(h->d_irp, 0, irp_bytes, st);
      if (e == cudaSuccess)
            e = cudaMemsetAsync(h->d_ja + NZ, 0, 16 * sizeof(int), st);
      if (e == cudaSuccess)
            e = cudaMemsetAsync(h->d_as + NZ, 0, 16 * sizeof(double), st);
      if (e != cudaSuccess) {
            fail(-EIO, "zeroing a new CSR handle failed: %s", cudaGetErrorString(e));
            spmv_b200_csr_destroy(h);
            return nullptr;
      }
      return h;
}

extern "C" spmv_b200_csr *spmv_b200_csr_create_ex(int64_t M, int64_t n_local, int64_t NZ,
                                                  const void *irp, int irp_bytes, const int *JA,
                                                  const double *AS, int64_t col_offset,
                                                  const int64_t *cuts, int n_cuts) {
      if (!irp || (NZ > 0 && (!JA || !AS)) || (irp_bytes != 4 && irp_bytes != 8)) {
            fail(-EINVAL, "spmv_b200_csr_create_ex: bad arguments");
            return nullptr;
      }
      static const char *what = "create_ex";
      spmv_b200_csr *h = csr_alloc_shell(M, n_local, NZ, col_offset, 0);
      if (!h)
            return nullptr;

      h->h_irp.resize((size_t)M + 1);
      if (irp_bytes == 4) {
            const int *p = static_cast<const int *>(irp);
            for (long long r = 0; r <= M; ++r)
                  h->h_irp[r] = p[r];
      } else {
            const long long *p = static_cast<const long long *>(irp);
            for (long long r = 0; r <= M; ++r)
                  h->h_irp[r] = p[r];
      }
      bool ok = h->h_irp[0] == 0 && h->h_irp[M] == NZ;
      for (long long r = 0; r < M && ok; ++r)
            ok = h->h_irp[r + 1] >= h->h_irp[r];
      if (!ok)
            return csr_finish(h, fail(-EINVAL, "row offsets are not a monotone prefix ending at NZ"),
                              cuts, n_cuts, what);

      cudaError_t e;
      if (h->wide) {
            e = cudaMemcpy(h->d_irp, h->h_irp.data(), (size_t)(M + 1) * 8, cudaMemcpyHostToDevice);
      } else {
            std::vector<int> tmp(h->h_irp.begin(), h->h_irp.end());
            e = cudaMemcpy(h->d_irp, tmp.data(), (size_t)(M + 1) * 4, cudaMemcpyHostToDevice);
      }
      if (e == cudaSuccess && NZ > 0)
            e = cudaMemcpy(h->d_as, AS, (size_t)NZ * sizeof(double), cudaMemcpyHostToDevice);
      if (e == cudaSuccess && NZ > 0) {
            if (col_offset == 0) {
                  e = cudaMemcpy(h->d_ja, JA, (size_t)NZ * sizeof(int), cudaMemcpyHostToDevice);
            } else {
                  std::vector<int> rel((size_t)NZ);
#pragma omp parallel for schedule(static)
                  for (long long k = 0; k < NZ; ++k)
                        rel[k] = (int)((long long)JA[k] - col_offset);
                  e = cudaMemcpy(h->d_ja, rel.data(), (size_t)NZ * sizeof(int),
                                 cudaMemcpyHostToDevice);
            }
      }
      if (e != cudaSuccess)
            return csr_finish(h, fail(-EIO, "CSR upload failed: %s", cudaGetErrorString(e)), cuts, n_cuts,
                              what);
      g_counters.h2d += (long long)((M + 1) * (h->wide ? 8 : 4) + NZ * 12);
      return csr_finish(h, csr_check_columns(h), cuts, n_cuts, what);
}

extern "C" spmv_b200_csr *spmv_b200_csr_create(const sparse_csr *A) {
      if (!A) {
            fail(-EINVAL, "null sparse_csr");
            return nullptr;
      }
      return spmv_b200_csr_create_ex(A->M, A->N, A->NZ, A->IRP, 4, A->JA, A->AS, 0, nullptr, 0);
}

extern "C" spmv_b200_csr *spmv_b200_csr_gen_stencil27(int nx, int ny, int nz, int z0, int z1,
                                                      int64_t col_offset, int64_t n_local,
                                                      const int64_t *cuts, int n_cuts) {
      if (nx < 1 || ny < 1 || nz < 1 || z0 < 0 || z1 > nz || z0 > z1) {
            fail(-EINVAL, "bad stencil geometry");
            return nullptr;
      }
      const long long plane = (long long)nx * ny, rows = plane * (z1 - z0);
      auto prefix = [](long long c, long long n) {
            return c == 0 ? 0ll : (c >= n ? 3 * n - 2 : 3 * c - 1);
      };
      const long long nnz = (prefix(z1, nz) - prefix(z0, nz)) * (3ll * ny - 2) * (3ll * nx - 2);
      spmv_b200_csr *h = csr_alloc_shell(rows, n_local, nnz, col_offset, 0);
      if (!h)
            return nullptr;
      StencilGeom g{nx, ny, nz, z0, col_offset};
      with_offsets(h->wide, [&](auto t) {
            using OffT = typename decltype(t)::type;
            stencil27_fill_kernel<OffT><<<blocks_for(rows + 1, 256), 256>>>(g, rows, (OffT *)h->d_irp,
                                                                           h->d_ja, h->d_as);
      });
      ++g_counters.launches;
      const cudaError_t e = cudaDeviceSynchronize();
      const int rc = e == cudaSuccess ? 0 : fail(-EIO, "stencil generation failed: %s", cudaGetErrorString(e));
      return csr_finish(h, rc, cuts, n_cuts, "stencil generation");
}

// Bits that can be non-zero in an index below n (at least 1, at most 31): the end bit of a radix
// sort over such indices.
static int index_bits(long long n) {
      int b = 1;
      while (b < 31 && (1ll << b) < n)
            ++b;
      return b;
}

// Row offsets of h from entries per row: d_irp[0..M] = exclusive scan of count[0..M] (count[M] is 0,
// so d_irp[M] is the total).  d_scratch == nullptr only sets `bytes`.
static cudaError_t scan_row_offsets(void *d_scratch, size_t &bytes, const int *count, spmv_b200_csr *h,
                                    cudaStream_t st = 0) {
      return with_offsets(h->wide, [&](auto t) {
            using OffT = typename decltype(t)::type;
            return cub::DeviceScan::ExclusiveSum(d_scratch, bytes, count, (OffT *)h->d_irp, (int)(h->M + 1), st);
      });
}

// A^T on the current device.  Memory while the sort runs, besides A and the new handle:
//   sort keys   the two key buffers of the radix sort live in the new handle's value array
//               (8 bytes per entry = two int32 arrays), which the fill overwrites afterwards;
//   sort values one buffer is the new handle's column array, the other is temporary (4 B/entry);
//   row_of      row of every entry of A (temporary, 4 B/entry);
//   count       entries per column of A (temporary, 4 B per column + 4);
//   scratch     CUB's temporary storage (histograms and tile state, independent of the entry count
//               up to a few bytes per tile).
// Peak temporary memory is therefore 8 bytes per entry + 4 bytes per column + CUB's scratch.
static int csr_transpose_fill(const spmv_b200_csr *A, spmv_b200_csr *h) {
      static const char *what = "transpose";
      const long long NZ = A->NZ, NT = A->N; // NT: rows of A^T
      DeviceTemps tmp;
      int *d_count = nullptr, *d_row_of = nullptr, *d_idx = nullptr;
      void *d_scratch = nullptr;
      size_t scan_bytes = 0, sort_bytes = 0;
      int *key0 = reinterpret_cast<int *>(h->d_as);
      int *key1 = key0 + ((NZ + 3) & ~3ll); // 16-byte aligned second half of the value array
      cub::DoubleBuffer<int> keys(key0, key1), vals(nullptr, h->d_ja);
      const int end_bit = index_bits(NT); // column bits that can be non-zero
      cudaError_t e = scan_row_offsets(nullptr, scan_bytes, d_count, h);
      if (e == cudaSuccess && NZ > 0)
            e = cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys, vals, (int)NZ, 0, end_bit);
      if (e != cudaSuccess)
            return fail(-EIO, "transpose: CUB size query failed: %s", cudaGetErrorString(e));
      if (tmp.alloc(&d_count, (NT + 1) * sizeof(int), what) ||
          tmp.alloc(&d_scratch, std::max(scan_bytes, sort_bytes), what) ||
          (NZ > 0 && (tmp.alloc(&d_row_of, NZ * sizeof(int), what) || tmp.alloc(&d_idx, NZ * sizeof(int), what))))
            return -ENOMEM;
      e = cudaMemsetAsync(d_count, 0, (size_t)(NT + 1) * sizeof(int));
      if (e == cudaSuccess && NZ > 0) {
            const int grid = (int)std::min<long long>(blocks_for(A->M * 32, 256), 65535ll * 8);
            with_offsets(A->wide, [&](auto t) {
                  using OffT = typename decltype(t)::type;
                  transpose_prep_kernel<OffT><<<grid, 256>>>((const OffT *)A->d_irp, A->d_ja, A->M, d_row_of,
                                                             key0, d_idx, d_count);
            });
            ++g_counters.launches;
            e = cudaGetLastError();
      }
      if (e == cudaSuccess)
            e = scan_row_offsets(d_scratch, scan_bytes, d_count, h);
      if (e == cudaSuccess && NZ > 0) {
            vals = cub::DoubleBuffer<int>(d_idx, h->d_ja);
            e = cub::DeviceRadixSort::SortPairs(d_scratch, sort_bytes, keys, vals, (int)NZ, 0, end_bit);
      }
      if (e == cudaSuccess && NZ > 0) {
            const int grid = (int)std::min<long long>(blocks_for(NZ, 256), (long long)g_sm_count * 64);
            transpose_fill_kernel<<<grid, 256>>>(vals.Current(), d_row_of, A->d_as, NZ, h->d_ja, h->d_as);
            ++g_counters.launches;
            e = cudaGetLastError();
      }
      // the second key buffer may have reached into the 16 zero entries after the values
      if (e == cudaSuccess)
            e = cudaMemsetAsync(h->d_as + NZ, 0, 16 * sizeof(double));
      if (e == cudaSuccess)
            e = cudaDeviceSynchronize();
      if (e != cudaSuccess)
            return fail(-EIO, "transpose failed: %s", cudaGetErrorString(e));
      return 0;
}

extern "C" spmv_b200_csr *spmv_b200_csr_transpose(const spmv_b200_csr *A) {
      if (!A) {
            fail(-EINVAL, "null CSR handle");
            return nullptr;
      }
      if (A->NZ >= (1ll << 31) - 64) {
            fail(-ENOTSUP, "transpose of handles with 2^31 or more entries is not supported (NZ=%lld)",
                 A->NZ);
            return nullptr;
      }
      if (ensure_device())
            return nullptr;
      int prev = 0;
      if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(A->device) != cudaSuccess) {
            fail(-EIO, "transpose: cannot select device %d", A->device);
            return nullptr;
      }
      spmv_b200_csr *h = csr_alloc_shell(A->N, A->M, A->NZ, 0, 0);
      if (h)
            h = csr_finish(h, csr_transpose_fill(A, h), nullptr, 0, "transpose");
      cudaSetDevice(prev);
      return h;
}

// ------------------------------------------------------------- from COO --
// CSR from n COO entries on the current device, all device work on `st`.  Steps:
//   pack   bounds check, key = row << cb | col (rb row bits, cb column bits; 32-bit keys when
//          rb + cb <= 32, else 64-bit), and whether the keys are sorted or repeat; 16 bytes read back;
//   sort   only when some key is smaller than its predecessor: stable radix sort of (key, entry
//          index) over bits [0, rb + cb), so entries with equal (row, col) keep their input order;
//   heads  sum mode, when equal keys are possible: run starts, scanned in place into each run's
//          output position and the output entry count (read back, 4 bytes);
//   fill   one thread per output entry writes ja and as and counts its row; an exclusive scan of
//          the counts is the row offsets.  In sum mode the thread of a run adds its L values left to
//          right: L dependent loads on one thread, so one (row, col) repeated many times is slow.
// Temporary memory besides the new handle (KB = 4 or 8 bytes per key):
//   sort   two key buffers and two index buffers: 2*KB + 8 bytes per entry (16 or 24), plus CUB's
//          scratch (histograms and tile state: a small fraction of a byte per entry); the spare key
//          and index buffers and the scratch are freed when the sort is done;
//   fill   sorted keys, the permutation and, in sum mode, the output positions: KB + 8 bytes per entry
//          (12 or 16) + 4 bytes per row (+ 4) for the counts, plus CUB's scan scratch.
// Input that is already sorted skips the sort and the permutation: KB bytes per entry, + 4 in sum
// mode when keys repeat, + 4 per row.
template <typename IdxT, typename KeyT>
static spmv_b200_csr *csr_from_coo_here(long long M, long long N, long long n, const IdxT *d_row,
                                        const IdxT *d_col, const double *d_val, bool sum, cudaStream_t st) {
      static const char *what = "from_coo";
      const int rb = index_bits(M), cb = index_bits(N);
      const int grid = (int)std::max<long long>(
          1, std::min<long long>(blocks_for(n, 256), (long long)g_sm_count * 64));
      DeviceTemps tmp;
      KeyT *key = nullptr;
      CooStatus *d_st = nullptr, hs{0x7fffffff, 0, 0, 0};
      if (n > 0 && (tmp.alloc(&d_st, sizeof(CooStatus), what) || tmp.alloc(&key, n * sizeof(KeyT), what)))
            return nullptr;
      cudaError_t e = cudaSuccess;
      if (n > 0) {
            e = cudaMemcpyAsync(d_st, &hs, sizeof hs, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                  coo_pack_kernel<IdxT, KeyT><<<grid, 256, 0, st>>>(d_row, d_col, n, M, N, cb, key, d_st);
                  ++g_counters.launches;
                  e = cudaGetLastError();
            }
            if (e == cudaSuccess)
                  e = cudaMemcpyAsync(&hs, d_st, sizeof hs, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess)
                  e = cudaStreamSynchronize(st);
      }
      if (e == cudaSuccess && hs.bad != 0x7fffffff) {
            IdxT r = 0, c = 0;
            e = cudaMemcpy(&r, d_row + hs.bad, sizeof r, cudaMemcpyDeviceToHost);
            if (e == cudaSuccess)
                  e = cudaMemcpy(&c, d_col + hs.bad, sizeof c, cudaMemcpyDeviceToHost);
            if (e == cudaSuccess) {
                  fail(-EINVAL, "from_coo: entry %d has row %lld and column %lld, outside [0, %lld) x [0, %lld)",
                       hs.bad, (long long)r, (long long)c, M, N);
                  return nullptr;
            }
      }
      const int *perm = nullptr;
      if (e == cudaSuccess && hs.unsorted) {
            KeyT *key1 = nullptr;
            int *idx0 = nullptr, *idx1 = nullptr;
            void *scratch = nullptr;
            size_t bytes = 0;
            cub::DoubleBuffer<KeyT> keys(key, nullptr);
            cub::DoubleBuffer<int> vals(nullptr, nullptr);
            e = cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, vals, (int)n, 0, rb + cb, st);
            if (e != cudaSuccess) {
                  fail(-EIO, "from_coo: CUB size query failed: %s", cudaGetErrorString(e));
                  return nullptr;
            }
            if (tmp.alloc(&key1, n * sizeof(KeyT), what) || tmp.alloc(&idx0, n * sizeof(int), what) ||
                tmp.alloc(&idx1, n * sizeof(int), what) || tmp.alloc(&scratch, bytes, what))
                  return nullptr;
            coo_iota_kernel<<<grid, 256, 0, st>>>(idx0, n);
            ++g_counters.launches;
            e = cudaGetLastError();
            keys = cub::DoubleBuffer<KeyT>(key, key1);
            vals = cub::DoubleBuffer<int>(idx0, idx1);
            if (e == cudaSuccess) {
                  e = cub::DeviceRadixSort::SortPairs(scratch, bytes, keys, vals, (int)n, 0, rb + cb, st);
                  ++g_counters.launches; // one CUB call counts as one launch
            }
            if (e == cudaSuccess)
                  e = cudaStreamSynchronize(st);
            key = keys.Current();
            perm = vals.Current();
            tmp.release(keys.Alternate()), tmp.release(vals.Alternate()), tmp.release(scratch);
      }
      long long nz_out = n;
      int *pos = nullptr;
      if (e == cudaSuccess && sum && (hs.unsorted || hs.dup)) {
            void *scratch = nullptr;
            size_t bytes = 0;
            e = cub::DeviceScan::ExclusiveSum(nullptr, bytes, pos, (int)(n + 1), st);
            if (e != cudaSuccess) {
                  fail(-EIO, "from_coo: CUB size query failed: %s", cudaGetErrorString(e));
                  return nullptr;
            }
            if (tmp.alloc(&pos, (n + 1) * sizeof(int), what) || tmp.alloc(&scratch, bytes, what))
                  return nullptr;
            coo_heads_kernel<KeyT><<<grid, 256, 0, st>>>(key, n, pos);
            ++g_counters.launches;
            e = cudaGetLastError();
            if (e == cudaSuccess) {
                  e = cub::DeviceScan::ExclusiveSum(scratch, bytes, pos, (int)(n + 1), st);
                  ++g_counters.launches;
            }
            int total = 0;
            if (e == cudaSuccess)
                  e = cudaMemcpyAsync(&total, pos + n, sizeof total, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess)
                  e = cudaStreamSynchronize(st);
            nz_out = total;
            tmp.release(scratch);
      }
      if (e != cudaSuccess) {
            fail(-EIO, "from_coo failed: %s", cudaGetErrorString(e));
            return nullptr;
      }

      spmv_b200_csr *h = csr_alloc_shell(M, N, nz_out, 0, st);
      if (!h)
            return nullptr;
      int *count = nullptr;
      void *scratch = nullptr;
      size_t bytes = 0;
      e = scan_row_offsets(nullptr, bytes, count, h, st);
      int rc = e == cudaSuccess ? 0 : fail(-EIO, "from_coo: CUB size query failed: %s", cudaGetErrorString(e));
      if (!rc)
            rc = tmp.alloc(&count, (M + 1) * sizeof(int), what) || tmp.alloc(&scratch, bytes, what);
      if (!rc) {
            e = cudaMemsetAsync(count, 0, (M + 1) * sizeof(int), st);
            if (e == cudaSuccess && n > 0) {
                  if (pos)
                        coo_fill_kernel<KeyT, true><<<grid, 256, 0, st>>>(key, perm, pos, d_val, n, cb, h->d_ja,
                                                                          h->d_as, count);
                  else
                        coo_fill_kernel<KeyT, false><<<grid, 256, 0, st>>>(key, perm, pos, d_val, n, cb, h->d_ja,
                                                                           h->d_as, count);
                  ++g_counters.launches;
                  e = cudaGetLastError();
            }
            if (e == cudaSuccess) {
                  e = scan_row_offsets(scratch, bytes, count, h, st);
                  ++g_counters.launches;
            }
            if (e == cudaSuccess)
                  e = cudaStreamSynchronize(st);
            tmp.release_all();
            if (e != cudaSuccess)
                  rc = fail(-EIO, "from_coo failed: %s", cudaGetErrorString(e));
      }
      return csr_finish(h, rc, nullptr, 0, what);
}

template <typename IdxT>
static spmv_b200_csr *csr_from_coo_idx(long long M, long long N, long long n, const void *d_row,
                                       const void *d_col, const double *d_val, bool sum, cudaStream_t st) {
      const IdxT *r = static_cast<const IdxT *>(d_row), *c = static_cast<const IdxT *>(d_col);
      if (index_bits(M) + index_bits(N) <= 32)
            return csr_from_coo_here<IdxT, unsigned>(M, N, n, r, c, d_val, sum, st);
      return csr_from_coo_here<IdxT, unsigned long long>(M, N, n, r, c, d_val, sum, st);
}

extern "C" spmv_b200_csr *spmv_b200_csr_from_coo(int64_t M, int64_t N, int64_t n, const void *d_row,
                                                 const void *d_col, int idx_bytes, const double *d_val,
                                                 int flags, void *stream) {
      const long long lim = (1ll << 31) - 64;
      if (M < 0 || N < 0 || n < 0 || M >= lim || N >= lim) {
            fail(-EINVAL, "from_coo: bad shape M=%lld N=%lld n=%lld", (long long)M, (long long)N, (long long)n);
            return nullptr;
      }
      if (idx_bytes != 4 && idx_bytes != 8) {
            fail(-EINVAL, "from_coo: index width %d bytes (4 or 8)", idx_bytes);
            return nullptr;
      }
      if (flags & ~SPMV_B200_COO_SUM_DUPLICATES) {
            fail(-EINVAL, "from_coo: unknown flag bits 0x%x", flags);
            return nullptr;
      }
      if (n >= lim) {
            fail(-ENOTSUP, "from_coo: 2^31 or more entries are not supported (n=%lld)", (long long)n);
            return nullptr;
      }
      if (n > 0 && (!d_row || !d_col || !d_val)) {
            fail(-EINVAL, "from_coo: null array with n=%lld", (long long)n);
            return nullptr;
      }
      if (ensure_device())
            return nullptr;
      int dev = 0;
      if (cudaGetDevice(&dev) != cudaSuccess) {
            fail(-EIO, "from_coo: no current device");
            return nullptr;
      }
      const void *arrays[3] = {d_row, d_col, d_val};
      const char *names[3] = {"row", "col", "val"};
      for (int i = 0; i < 3 && n > 0; ++i) {
            cudaPointerAttributes a;
            if (cudaPointerGetAttributes(&a, arrays[i]) != cudaSuccess) {
                  cudaGetLastError(); // clear the error of the query
                  a.type = cudaMemoryTypeUnregistered;
            }
            if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != dev) {
                  fail(-EINVAL, "from_coo: %s array %p is not device or managed memory of device %d", names[i],
                       arrays[i], dev);
                  return nullptr;
            }
      }
      const bool sum = flags & SPMV_B200_COO_SUM_DUPLICATES;
      cudaStream_t st = static_cast<cudaStream_t>(stream);
      return idx_bytes == 4 ? csr_from_coo_idx<int>(M, N, n, d_row, d_col, d_val, sum, st)
                            : csr_from_coo_idx<long long>(M, N, n, d_row, d_col, d_val, sum, st);
}

// -------------------------------------------------------------- product --
namespace {
// Hash tables of the product (spgemm_kernels.cuh): a row's table has the least power of two slots
// that is >= 2 min(P_i, B.N) and >= kSpgemmMinSlots, at most 2^31.  Tables of up to
// kSpgemmSharedSlots slots are per warp in shared memory, one launch per size; larger ones are
// regions of one global table.
constexpr long long kSpgemmMinSlots = 32;
constexpr long long kSpgemmSharedSlots = 4096;
constexpr int kSpgemmSharedBins = 8; // 32, 64, ..., 4096 slots
constexpr int kSpgemmGlobalWarps = 4;

// Warps per block of a shared-table launch: 8192 slots per block (98 KB of keys, values and
// staging at 4096 slots in the numeric pass), at most 8 warps.
int spgemm_warps(long long slots) { return (int)std::min<long long>(8, std::max<long long>(1, 8192 / slots)); }

long long spgemm_slots(long long P, long long N) {
      const long long b = 2 * std::min(P, N);
      long long s = kSpgemmMinSlots;
      if (b > s)
            s = 1ll << (64 - __builtin_clzll((unsigned long long)(b - 1)));
      return std::min(s, 1ll << 31);
}
} // namespace

// C = A * B on the current device (A's).  Steps, all on the legacy default stream:
//   count     P_i for every row of A, read back (8 bytes per row) and binned on the host by table
//             size; rows with P_i = 0 are empty in C and run nowhere;
//   symbolic  entries per row of C and their 64-bit sum (read back, so that 2^31 - 64 or more
//             entries fail before C is allocated);
//   numeric   the rows of C, each in slot order, at C's row offsets (the scan of the counts) in two
//             temporary arrays;
//   sort      cub::DeviceSegmentedSort orders each row by column into C's arrays.
// Temporary memory besides the new handle: 8 bytes per row of A (P) + 4 per row (+ 4) for the
// counts + 4 per row with products (the binned rows) + 12 per global-table slot and 8 per row
// that has one + 12 per entry of C (the unsorted rows), plus CUB's scratch.
static spmv_b200_csr *csr_spgemm_here(const spmv_b200_csr *A, const spmv_b200_csr *B) {
      static const char *what = "spgemm";
      const long long M = A->M, lim = (1ll << 31) - 64;
      DeviceTemps tmp;
      long long *d_P = nullptr;
      if (tmp.alloc(&d_P, M * sizeof(long long), what))
            return nullptr;
      cudaError_t e = cudaSuccess;
      if (M > 0) {
            const int grid = (int)std::min<long long>(blocks_for(M * 32, 256), 65535ll * 8);
            with_offsets(A->wide, [&](auto ta) {
                  with_offsets(B->wide, [&](auto tb) {
                        using OffA = typename decltype(ta)::type;
                        using OffB = typename decltype(tb)::type;
                        spgemm_count_kernel<OffA, OffB>
                            <<<grid, 256>>>((const OffA *)A->d_irp, A->d_ja, M, (const OffB *)B->d_irp, d_P);
                  });
            });
            ++g_counters.launches;
            e = cudaGetLastError();
      }
      std::vector<long long> P((size_t)M);
      if (e == cudaSuccess)
            e = cudaMemcpy(P.data(), d_P, M * sizeof(long long), cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) {
            fail(-EIO, "spgemm: product count failed: %s", cudaGetErrorString(e));
            return nullptr;
      }
      g_counters.d2h += M * (long long)sizeof(long long);
      tmp.release(d_P);

      // bins: kSpgemmSharedBins shared-table sizes, then the global-table rows; a stable counting
      // sort of the rows by bin, and the global rows' table regions
      constexpr int kBins = kSpgemmSharedBins + 1;
      auto bin_of = [&](long long p) {
            const long long s = spgemm_slots(p, B->N);
            return s > kSpgemmSharedSlots ? kSpgemmSharedBins : 63 - __builtin_clzll((unsigned long long)s) - 5;
      };
      long long start[kBins + 1] = {0};
      for (long long r = 0; r < M; ++r)
            if (P[r] > 0)
                  ++start[bin_of(P[r]) + 1];
      for (int b = 0; b < kBins; ++b)
            start[b + 1] += start[b];
      std::vector<int> rows((size_t)start[kBins]);
      std::vector<long long> toff(1, 0);
      long long fill[kBins];
      std::copy(start, start + kBins, fill);
      for (long long r = 0; r < M; ++r) {
            if (P[r] <= 0)
                  continue;
            const int b = bin_of(P[r]);
            rows[fill[b]++] = (int)r;
            if (b == kSpgemmSharedBins)
                  toff.push_back(toff.back() + spgemm_slots(P[r], B->N));
      }
      std::vector<long long>().swap(P);

      int *d_rows = nullptr, *d_count = nullptr, *gkeys = nullptr;
      long long *d_toff = nullptr;
      double *gvals = nullptr;
      unsigned long long *d_total = nullptr;
      const long long gslots = toff.back();
      if (tmp.upload(&d_rows, rows, what) || tmp.upload(&d_toff, toff, what) ||
          tmp.alloc(&d_count, (M + 1) * sizeof(int), what) || tmp.alloc(&d_total, sizeof *d_total, what) ||
          tmp.alloc(&gkeys, gslots * sizeof(int), what) || tmp.alloc(&gvals, gslots * sizeof(double), what))
            return nullptr;
      e = cudaMemsetAsync(d_count, 0, (M + 1) * sizeof(int));
      if (e == cudaSuccess)
            e = cudaMemsetAsync(d_total, 0, sizeof *d_total);

      // one pass (symbolic or numeric) over every non-empty bin
      auto pass = [&](bool numeric, const void *irp_c, bool wide_c, int *t_ja, double *t_as) {
            cudaError_t pe = cudaSuccess;
            for (int b = 0; b < kBins && pe == cudaSuccess; ++b) {
                  const long long n = start[b + 1] - start[b];
                  if (n == 0)
                        continue;
                  const bool shared = b < kSpgemmSharedBins;
                  const long long slots = shared ? kSpgemmMinSlots << b : 0;
                  const int wpb = shared ? spgemm_warps(slots) : kSpgemmGlobalWarps;
                  const size_t smem = shared ? (size_t)wpb * (numeric ? slots * 12 + 256 : slots * 4)
                                             : (numeric ? (size_t)wpb * 256 : 0);
                  const int grid = (int)std::min<long long>(blocks_for(n * 32, wpb * 32), (long long)g_sm_count * 64);
                  const SpgemmRows rs{d_rows + start[b], n, slots, d_toff, gkeys, gvals};
                  with_offsets(A->wide, [&](auto ta) {
                        with_offsets(B->wide, [&](auto tb) {
                              using OffA = typename decltype(ta)::type;
                              using OffB = typename decltype(tb)::type;
                              auto go = [&](auto kernel, auto... args) {
                                    pe = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                              (int)smem);
                                    if (pe == cudaSuccess) {
                                          kernel<<<grid, wpb * 32, smem>>>(args...);
                                          pe = cudaGetLastError();
                                    }
                              };
                              const OffA *ia = (const OffA *)A->d_irp;
                              const OffB *ib = (const OffB *)B->d_irp;
                              if (numeric && shared)
                                    go(spgemm_numeric_kernel<SharedTable, OffA, OffB>, ia, A->d_ja, A->d_as, ib,
                                       B->d_ja, B->d_as, rs, irp_c, wide_c, t_ja, t_as);
                              else if (numeric)
                                    go(spgemm_numeric_kernel<GlobalTable, OffA, OffB>, ia, A->d_ja, A->d_as, ib,
                                       B->d_ja, B->d_as, rs, irp_c, wide_c, t_ja, t_as);
                              else if (shared)
                                    go(spgemm_symbolic_kernel<SharedTable, OffA, OffB>, ia, A->d_ja, ib, B->d_ja, rs,
                                       d_count, d_total);
                              else
                                    go(spgemm_symbolic_kernel<GlobalTable, OffA, OffB>, ia, A->d_ja, ib, B->d_ja, rs,
                                       d_count, d_total);
                        });
                  });
                  ++g_counters.launches;
            }
            return pe;
      };

      unsigned long long total = 0;
      if (e == cudaSuccess)
            e = pass(false, nullptr, false, nullptr, nullptr);
      if (e == cudaSuccess)
            e = cudaMemcpy(&total, d_total, sizeof total, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) {
            fail(-EIO, "spgemm: symbolic pass failed: %s", cudaGetErrorString(e));
            return nullptr;
      }
      if ((long long)total >= lim) {
            fail(-ENOTSUP, "spgemm: products with 2^31 - 64 or more entries are not supported (%llu entries)",
                 total);
            return nullptr;
      }
      const long long nz = (long long)total;

      spmv_b200_csr *h = csr_alloc_shell(M, B->N, nz, 0, 0);
      if (!h)
            return nullptr;
      int *t_ja = nullptr;
      double *t_as = nullptr;
      void *scratch = nullptr;
      size_t scan_bytes = 0, sort_bytes = 0;
      auto segsort = [&](void *s, size_t &bytes) {
            return with_offsets(h->wide, [&](auto t) {
                  using OffT = typename decltype(t)::type;
                  const OffT *irp = (const OffT *)h->d_irp;
                  return cub::DeviceSegmentedSort::SortPairs(s, bytes, t_ja, h->d_ja, t_as, h->d_as, (int)nz, (int)M,
                                                             irp, irp + 1);
            });
      };
      e = scan_row_offsets(nullptr, scan_bytes, d_count, h);
      if (e == cudaSuccess && nz > 0)
            e = segsort(nullptr, sort_bytes);
      int rc = e == cudaSuccess ? 0 : fail(-EIO, "spgemm: CUB size query failed: %s", cudaGetErrorString(e));
      if (!rc)
            rc = tmp.alloc(&scratch, std::max(scan_bytes, sort_bytes), what) ||
                 tmp.alloc(&t_ja, nz * sizeof(int), what) || tmp.alloc(&t_as, nz * sizeof(double), what);
      if (!rc) {
            e = scan_row_offsets(scratch, scan_bytes, d_count, h);
            ++g_counters.launches;
            if (e == cudaSuccess)
                  e = pass(true, h->d_irp, h->wide, t_ja, t_as);
            if (e == cudaSuccess && nz > 0) {
                  e = segsort(scratch, sort_bytes);
                  ++g_counters.launches;
            }
            if (e == cudaSuccess)
                  e = cudaDeviceSynchronize();
            tmp.release_all();
            if (e != cudaSuccess)
                  rc = fail(-EIO, "spgemm failed: %s", cudaGetErrorString(e));
      }
      return csr_finish(h, rc, nullptr, 0, what);
}

extern "C" spmv_b200_csr *spmv_b200_csr_spgemm(const spmv_b200_csr *A, const spmv_b200_csr *B) {
      if (!A || !B) {
            fail(-EINVAL, "spgemm: null CSR handle");
            return nullptr;
      }
      if (A->N != B->M) {
            fail(-EINVAL, "spgemm: A has %lld columns but B has %lld rows", A->N, B->M);
            return nullptr;
      }
      if (A->device != B->device) {
            fail(-EINVAL, "spgemm: A is on device %d, B on device %d", A->device, B->device);
            return nullptr;
      }
      if (ensure_device())
            return nullptr;
      int prev = 0;
      if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(A->device) != cudaSuccess) {
            fail(-EIO, "spgemm: cannot select device %d", A->device);
            return nullptr;
      }
      spmv_b200_csr *h = csr_spgemm_here(A, B);
      cudaSetDevice(prev);
      return h;
}

extern "C" void spmv_b200_csr_destroy(spmv_b200_csr *h) {
      if (!h)
            return;
      for (auto &sg : h->segs)
            free_segment(sg);
      for (auto &sg : h->pipe_segs)
            free_segment(sg);
      free_sell(h->sell), free_sell(h->sell_mm2), free_sell(h->sell_mm4);
      cudaFree(h->d_dot_partial);
      cudaFree(h->d_irp);
      cudaFree(h->d_ja);
      cudaFree(h->d_as);
      delete h;
}

extern "C" int64_t spmv_b200_csr_rows(const spmv_b200_csr *h) { return h ? h->M : -1; }
extern "C" int64_t spmv_b200_csr_cols(const spmv_b200_csr *h) { return h ? h->N : -1; }
extern "C" int64_t spmv_b200_csr_nnz(const spmv_b200_csr *h) { return h ? h->NZ : -1; }

extern "C" int spmv_b200_csr_download(const spmv_b200_csr *h, int64_t *irp64, int *JA,
                                      double *AS) {
      if (!h)
            return fail(-EINVAL, "null CSR handle");
      if (irp64)
            std::copy(h->h_irp.begin(), h->h_irp.end(), irp64);
      if (JA && h->NZ)
            B200_CUDA(cudaMemcpy(JA, h->d_ja, (size_t)h->NZ * sizeof(int), cudaMemcpyDeviceToHost));
      if (AS && h->NZ)
            B200_CUDA(
                cudaMemcpy(AS, h->d_as, (size_t)h->NZ * sizeof(double), cudaMemcpyDeviceToHost));
      return 0;
}

extern "C" int spmv_b200_csr_plan_info(const spmv_b200_csr *h, int64_t *out, int n_out) {
      if (!h || !out)
            return fail(-EINVAL, "null argument");
      for (int i = 0; i < n_out; ++i)
            out[i] = 0;
      for (auto &sg : h->segs) {
            for (int k = 0; k < kNumKinds && k < n_out; ++k)
                  out[k] += sg.kind_rows[k];
            if (n_out > kNumKinds)
                  out[kNumKinds] += sg.regular ? 1 : 0;
            if (n_out > kNumKinds + 1)
                  out[kNumKinds + 1] = sg.base_kind;
      }
      return 0;
}

extern "C" int spmv_b200_csr_codes_info(const spmv_b200_csr *h, int64_t *out, int n_out) {
      if (!h || !out)
            return fail(-EINVAL, "null argument");
      int64_t v[4] = {0, 0, 0, 0}; // state, tiles, largest dictionary, block bytes
      for (const auto &sg : h->segs)
            for (const auto &kv : sg.stream) {
                  const StreamPlan &sp = kv.second;
                  if (sp.codes_state == -1)
                        v[0] = -1;
                  else if (sp.codes_state == 1 && v[0] == 0)
                        v[0] = 1;
                  if (sp.codes_state == 1) {
                        v[1] += sp.n_tiles;
                        v[2] = std::max<int64_t>(v[2], sp.max_dict);
                        v[3] += sp.code_bytes;
                  }
            }
      for (int i = 0; i < n_out && i < 4; ++i)
            out[i] = v[i];
      return 0;
}

extern "C" int spmv_b200_csr_sell_info(spmv_b200_csr *h, int build, int64_t *out, int n_out) {
      if (!h || !out)
            return fail(-EINVAL, "null argument");
      if (build && h->sell.state == 0 && h->segs.size() == 1)
            csr_ensure_sell(h);
      const SellPlan &sp = h->sell;
      const int64_t v[11] = {sp.state, sp.K, sp.sigma, sp.n_slices, sp.slots, sp.nnz_in_slices,
                             sp.n_long, (int64_t)(h->gather_span * 1e6), sp.chunk, sp.n_split_rows,
                             sp.n_partials};
      for (int i = 0; i < n_out && i < 11; ++i)
            out[i] = v[i];
      return 0;
}

// Host half of the SELL-P build on caller-supplied per-panel row counts (no GPU involved):
// exposed so the ordering / slice-offset rule can be checked without a device.
extern "C" int spmv_b200_sell_plan(const int *counts, int64_t M, int K, int sigma, int *perm,
                                   int64_t *soff) {
      if (!counts || !perm || !soff || M < 0 || K < 1 || K > 64 || sigma < 32 || sigma % 32)
            return fail(-EINVAL, "sell_plan: bad arguments");
      std::vector<int> c(counts, counts + (size_t)K * M), pv;
      std::vector<long long> sv;
      long long nnz = 0;
      sell_plan_host(c, M, K, sigma, pv, sv, &nnz, nullptr);
      std::copy(pv.begin(), pv.end(), perm);
      std::copy(sv.begin(), sv.end(), soff);
      return 0;
}

// Same for the virtual-row form: sizes[4] = {virtual rows, slices, split rows, pieces}; dest
// (slices*32) and soff (slices+1) may be NULL on a first call that only asks for the sizes.
extern "C" int spmv_b200_sell_plan_vrows(const int64_t *irp, int64_t M, int chunk, int sigma,
                                         int64_t *sizes, int *dest_out, int64_t *soff_out) {
      if (!irp || !sizes || M < 0 || chunk < 1 || sigma < 32 || sigma % 32)
            return fail(-EINVAL, "sell_plan_vrows: bad arguments");
      std::vector<long long> h_irp(irp, irp + M + 1);
      std::vector<int> vr_row, vr_j0, vr_len, dest, split_row, split_first, perm_v;
      std::vector<long long> soff;
      sell_virtual_rows(h_irp, M, chunk, vr_row, vr_j0, vr_len, dest, split_row, split_first);
      long long nnz = 0;
      const long long V = (long long)vr_row.size();
      sell_plan_host(vr_len, V, 1, sigma, perm_v, soff, &nnz, nullptr);
      sizes[0] = V, sizes[1] = (V + 31) / 32, sizes[2] = (int64_t)split_row.size(), sizes[3] = split_first.back();
      if (dest_out)
            for (size_t i = 0; i < perm_v.size(); ++i)
                  dest_out[i] = perm_v[i] >= 0 ? dest[perm_v[i]] : -1;
      if (soff_out)
            std::copy(soff.begin(), soff.end(), soff_out);
      return 0;
}

extern "C" int spmv_b200_csr_sell_download(const spmv_b200_csr *h, int64_t *soff, int *perm, int *JA,
                                           double *AS) {
      if (!h || h->sell.state != 1)
            return fail(-EINVAL, "no SELL-P plan on this handle");
      const SellPlan &sp = h->sell;
      if (soff)
            B200_CUDA(cudaMemcpy(soff, sp.d_soff, (size_t)sp.K * (sp.n_slices + 1) * 8,
                                 cudaMemcpyDeviceToHost));
      if (perm)
            B200_CUDA(cudaMemcpy(perm, sp.d_perm, (size_t)sp.K * sp.n_slices * 32 * 4,
                                 cudaMemcpyDeviceToHost));
      if (JA && sp.slots)
            B200_CUDA(cudaMemcpy(JA, sp.d_ja, (size_t)sp.slots * 4, cudaMemcpyDeviceToHost));
      if (AS && sp.slots)
            B200_CUDA(cudaMemcpy(AS, sp.d_as, (size_t)sp.slots * 8, cudaMemcpyDeviceToHost));
      return 0;
}

extern "C" int spmv_b200_csr_spmv(spmv_b200_csr *h, int kernel, int wpb, const double *d_x,
                                  double *d_y, void *stream) {
      return csr_run(h, kernel, wpb, 0, h ? h->M : 0, d_x, d_y, EPI_PLAIN, EpiArgs{}, stream);
}

extern "C" int spmv_b200_csr_spmv_rows(spmv_b200_csr *h, int kernel, int wpb, int64_t row0,
                                       int64_t row1, const double *d_x, double *d_y,
                                       void *stream) {
      return csr_run(h, kernel, wpb, row0, row1, d_x, d_y, EPI_PLAIN, EpiArgs{}, stream);
}

extern "C" int spmv_b200_csr_spmv_rows_push(spmv_b200_csr *h, int kernel, int wpb, int64_t row0,
                                            int64_t row1, const double *d_x, double *d_y,
                                            int n_push, const int64_t *push_row0,
                                            const int64_t *push_row1, double *const *d_push_dst,
                                            void *stream) {
      if (n_push < 0 || n_push > kMaxPush)
            return fail(-EINVAL, "n_push must be 0..%d", kMaxPush);
      EpiArgs p{};
      p.n_push = n_push;
      for (int i = 0; i < n_push; ++i) {
            p.row0[i] = push_row0[i];
            p.row1[i] = push_row1[i];
            p.dst[i] = d_push_dst[i];
      }
      return csr_run(h, kernel, wpb, row0, row1, d_x, d_y, n_push ? EPI_PUSH : EPI_PLAIN, p, stream);
}

extern "C" int spmv_b200_csr_spmv_fused(spmv_b200_csr *h, int kernel, int wpb, const double *d_x,
                                        double *d_y, double alpha, double beta, const double *d_z,
                                        const double *d_w, double *d_dot, void *stream) {
      EpiArgs e{};
      e.alpha = alpha, e.beta = beta;
      e.z = d_z;
      e.w = d_dot ? d_w : nullptr;
      e.dot_partial = d_dot; // csr_run swaps in the per-warp scratch and reduces into d_dot
      return csr_run(h, kernel, wpb, 0, h ? h->M : 0, d_x, d_y, EPI_FUSED, e, stream);
}

// ------------------------------------------------------------------- SpMM
namespace {

template <int K, typename OffT>
void launch_mm_rows(const spmv_b200_csr *h, int lpr_log2, long long row0, long long nrows, const int *rowlist,
                    const double *X, double *Y, cudaStream_t st) {
      if (nrows <= 0)
            return;
      const OffT *irp = (const OffT *)h->d_irp;
      constexpr int T = 256;
#define MM_CASE(L)                                                                                 \
      csr_mm_kernel<K, L, OffT><<<blocks_for(nrows * L, T), T, 0, st>>>(irp, h->d_ja, h->d_as, row0, nrows, \
                                                                         rowlist, X, Y)
      switch (lpr_log2) {
      case 0: MM_CASE(1); break;
      case 1: MM_CASE(2); break;
      case 2: MM_CASE(4); break;
      case 3: MM_CASE(8); break;
      case 4: MM_CASE(16); break;
      default: MM_CASE(32); break;
      }
#undef MM_CASE
      ++g_counters.launches;
}

template <int K>
int csr_spmm_k(spmv_b200_csr *h, const double *X, double *Y, cudaStream_t st) {
      if (csr_wants_sell(h) && csr_ensure_sell(h) == 0) {
            // column panels are sized for the x they must keep in the L2: K right-hand sides need K
            // times as many, i.e. a plan of their own (virtual-row plans have one panel: shared)
            SellPlan *plan = &h->sell;
            if (h->sell.chunk == 0 && sell_panels_for(h->N * K, h->gather_span) != h->sell.K) {
                  plan = K == 2 ? &h->sell_mm2 : &h->sell_mm4;
                  if (csr_build_sell(h, *plan, K))
                        return fail(-ENOMEM, "SpMM: could not build the %d-vector slice plan", K);
            }
            SellPlan &sp = *plan;
            const int threads = 128;
            const int grid = blocks_for(sp.n_slices * 32, threads);
            if (sp.chunk > 0) { // virtual rows: one panel, pieces of split rows combined in order
                  if (sp.n_partials && !sp.d_partial_mm &&
                      cudaMalloc(&sp.d_partial_mm, (size_t)sp.n_partials * 4 * sizeof(double)) != cudaSuccess)
                        return fail(-ENOMEM, "SpMM partial sums: out of device memory");
                  sell_mm_kernel<K, EPI_PLAIN, true><<<grid, threads, 0, st>>>(
                      sp.d_soff, sp.d_perm, sp.d_ja, sp.d_as, sp.n_slices, X, Y, sp.d_partial_mm);
                  ++g_counters.launches;
                  if (sp.n_split_rows) {
                        csr_combine_mm_kernel<K><<<blocks_for(sp.n_split_rows, 128), 128, 0, st>>>(
                            sp.d_split_row, sp.d_split_first, (int)sp.n_split_rows, sp.d_partial_mm, Y);
                        ++g_counters.launches;
                  }
                  return 0;
            }
            for (int p = 0; p < sp.K; ++p) {
                  const long long *soff = sp.d_soff + (size_t)p * (sp.n_slices + 1);
                  const int *perm = sp.d_perm + (size_t)p * sp.n_slices * 32;
                  if (p == 0)
                        sell_mm_kernel<K, EPI_PLAIN, false><<<grid, threads, 0, st>>>(soff, perm, sp.d_ja, sp.d_as,
                                                                                      sp.n_slices, X, Y, nullptr);
                  else
                        sell_mm_kernel<K, EPI_ACC, false><<<grid, threads, 0, st>>>(soff, perm, sp.d_ja, sp.d_as,
                                                                                    sp.n_slices, X, Y, nullptr);
                  ++g_counters.launches;
            }
            // rows too long for a slice: a warp per row
            const RowList lists[2] = {sp.long_warp, sp.long_block};
            for (const RowList &l : lists) {
                  if (h->wide)
                        launch_mm_rows<K, long long>(h, 5, 0, l.n, l.d_rows, X, Y, st);
                  else
                        launch_mm_rows<K, int>(h, 5, 0, l.n, l.d_rows, X, Y, st);
            }
            if (sp.long_split.n_rows) {
                  if (h->wide)
                        launch_mm_rows<K, long long>(h, 5, 0, sp.long_split.n_rows, sp.long_split.d_row, X, Y, st);
                  else
                        launch_mm_rows<K, int>(h, 5, 0, sp.long_split.n_rows, sp.long_split.d_row, X, Y, st);
            }
            return 0;
      }
      // no sorted slices for this matrix: lanes per row from the mean row length
      const double mean = h->M ? (double)h->NZ / (double)h->M : 0.0;
      const int lg = mean <= 6 ? 1 : (mean <= 12 ? 2 : (mean <= 48 ? 3 : (mean <= 96 ? 4 : 5)));
      if (h->wide)
            launch_mm_rows<K, long long>(h, lg, 0, h->M, nullptr, X, Y, st);
      else
            launch_mm_rows<K, int>(h, lg, 0, h->M, nullptr, X, Y, st);
      return 0;
}

} // namespace

extern "C" int spmv_b200_csr_spmm(spmv_b200_csr *h, int k, const double *d_X, double *d_Y, void *stream) {
      if (!h || !d_X || !d_Y)
            return fail(-EINVAL, "csr_spmm: null argument");
      if (k != 2 && k != 4)
            return fail(-EINVAL, "csr_spmm: 2 or 4 right-hand sides (got %d)", k);
      if (((uintptr_t)d_X & 15) || ((uintptr_t)d_Y & 7))
            return fail(-EINVAL, "csr_spmm: X must be 16-byte aligned");
      cudaStream_t st = as_stream(stream);
      int rc = k == 2 ? csr_spmm_k<2>(h, d_X, d_Y, st) : csr_spmm_k<4>(h, d_X, d_Y, st);
      if (rc)
            return rc;
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess)
            return fail(-EIO, "SpMM launch failed: %s", cudaGetErrorString(e));
      return 0;
}

extern "C" int spmv_b200_csr_launches(const spmv_b200_csr *h, int kernel) {
      if (!h)
            return -EINVAL;
      const bool sell_id = kernel == SPMV_B200_CSR_ADAPTIVE || kernel == SPMV_B200_CSR_STREAM;
      if (sell_id && h->sell.state == 1 && csr_wants_sell(const_cast<spmv_b200_csr *>(h)))
            return h->sell.K + (h->sell.n_split_rows > 0) + (h->sell.long_warp.n > 0) +
                   (h->sell.long_block.n > 0) + (h->sell.long_split.n_rows ? 2 : 0);
      int n = 0;
      for (auto &sg : h->segs) {
            if (sg.r1 == sg.r0)
                  continue;
            const bool streamed = kernel == SPMV_B200_CSR_STREAM ||
                                  (kernel == SPMV_B200_CSR_ADAPTIVE && sg.regular);
            if (streamed) {
                  n += 1;
                  for (auto &kv : sg.stream) {
                        for (int k = 5; k < 7; ++k)
                              n += kv.second.long_lists[k].n > 0;
                        n += kv.second.split.n_rows ? 2 : 0;
                        break;
                  }
            } else if (kernel == SPMV_B200_CSR_ADAPTIVE) {
                  n += sg.regular ? 1 : 0;
                  for (int k = 0; k < 7; ++k)
                        if (!(sg.regular && k <= sg.base_kind))
                              n += sg.lists[k].n > 0;
                  n += sg.split.n_rows ? 2 : 0;
            } else {
                  n += 1;
            }
      }
      return n;
}

// ------------------------------------------------------------------ timing --

namespace {

template <typename F>
int time_launches(F &&run, int warmup, int reps, int flush_l2, double *ms_out, void *stream) {
      if (reps < 1 || !ms_out)
            return fail(-EINVAL, "reps must be >= 1 and ms_out non-null");
      cudaStream_t st = as_stream(stream);
      std::vector<cudaEvent_t> ev(2 * (size_t)reps);
      for (auto &e : ev)
            B200_CUDA(cudaEventCreate(&e));
      int rc = 0;
      for (int i = 0; i < warmup && !rc; ++i)
            rc = run();
      for (int i = 0; i < reps && !rc; ++i) {
            if (flush_l2)
                  rc = spmv_b200_flush_l2(stream);
            if (rc)
                  break;
            cudaEventRecord(ev[2 * i], st);
            rc = run();
            cudaEventRecord(ev[2 * i + 1], st);
      }
      cudaError_t e = cudaStreamSynchronize(st);
      if (!rc && e != cudaSuccess)
            rc = fail(-EIO, "kernel execution failed: %s", cudaGetErrorString(e));
      for (int i = 0; i < reps && !rc; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]) != cudaSuccess)
                  rc = fail(-EIO, "cudaEventElapsedTime failed");
            ms_out[i] = ms;
      }
      for (auto &e2 : ev)
            cudaEventDestroy(e2);
      return rc;
}

} // namespace

namespace b200 {
double median_of(std::vector<double> v) {
      std::sort(v.begin(), v.end());
      return v[v.size() / 2];
}
} // namespace b200

extern "C" int spmv_b200_csr_time(spmv_b200_csr *h, int kernel, int wpb, const double *d_x,
                                  double *d_y, int warmup, int reps, int flush_l2, double *ms_out,
                                  void *stream) {
      return time_launches([&] { return spmv_b200_csr_spmv(h, kernel, wpb, d_x, d_y, stream); },
                           warmup, reps, flush_l2, ms_out, stream);
}


// ================================================================ HLL handle

namespace {

#define HLL_STREAM_CONFIGS(X)                                                                      \
      X(0, 4, 2, 4096)                                                                             \
      X(1, 2, 3, 2048)                                                                             \
      X(2, 8, 2, 8192)
constexpr int kNumHllStreamCfg = 3;
struct HllStreamShape {
      int warps, stages, cap;
};
constexpr HllStreamShape kHllStreamShapes[kNumHllStreamCfg] = {
#define X(id, w, s, c) {w, s, c},
    HLL_STREAM_CONFIGS(X)
#undef X
};

int hll_stream_cfg_for(int wpb) {
      if (g_knobs.hll_stream_cfg >= 0 && g_knobs.hll_stream_cfg < kNumHllStreamCfg)
            return g_knobs.hll_stream_cfg;
      return wpb <= 2 ? 1 : (wpb <= 4 ? 0 : 2);
}

int hll_build_tiles(spmv_b200_hll *h, int warps, int cap, spmv_b200_hll::Tiles &t) {
      std::vector<int> tile_h;
      long long b = 0;
      while (b < h->n_hacks) {
            long long e = b;
            while (e < h->n_hacks && e - b < warps && h->h_hoff[e + 1] - h->h_hoff[b] <= cap)
                  ++e;
            if (e == b)
                  e = b + 1; // oversized hack: its own tile
            tile_h.push_back((int)b);
            b = e;
      }
      tile_h.push_back((int)h->n_hacks);
      t.n_tiles = (int)tile_h.size() - 1;
      int rc = upload(&t.d_tile_h, tile_h);
      t.built = rc == 0;
      return rc;
}

int hll_alloc(spmv_b200_hll *h, const std::vector<int> &width) {
      h->h_hoff.resize((size_t)h->n_hacks + 1);
      h->h_hoff[0] = 0;
      for (long long b = 0; b < h->n_hacks; ++b)
            h->h_hoff[b + 1] = h->h_hoff[b] + 32ll * width[b], h->max_width = std::max(h->max_width, (int)width[b]);
      h->slots = h->h_hoff[h->n_hacks];
      B200_CUDA(cudaMalloc(&h->d_hoff, ((size_t)h->n_hacks + 1) * sizeof(long long)));
      B200_CUDA(cudaMemcpy(h->d_hoff, h->h_hoff.data(), ((size_t)h->n_hacks + 1) * sizeof(long long),
                           cudaMemcpyHostToDevice));
      B200_CUDA(cudaMalloc(&h->d_ja, ((size_t)h->slots + 32) * sizeof(int)));
      B200_CUDA(cudaMalloc(&h->d_as, ((size_t)h->slots + 32) * sizeof(double)));
      B200_CUDA(cudaMalloc(&h->d_rowlen, ((size_t)h->n_hacks * 32 + 32) * sizeof(int)));
      return 0;
}

HllSrc hll_src(const spmv_b200_hll *h) { return HllSrc{h->d_hoff, h->d_ja, h->d_as, h->d_rowlen}; }

bool hll_wants_sell(spmv_b200_hll *h) {
      if (g_knobs.sell == 0 || h->M < 64)
            return false;
      if (g_knobs.sell == 1)
            return true;
      return sell_panels_for(h->N, h->gather_span) > 1;
}

int hll_ensure_sell(spmv_b200_hll *h) {
      if (h->sell.state != 0)
            return h->sell.state == 1 ? 0 : -1;
      const int K = sell_panels_for(h->N, h->gather_span);
      int rc = sell_build(hll_src(h), h->M, h->N, K, 0x7fffffff, h->sell, nullptr);
      return rc || h->sell.state != 1 ? sell_not_built(h->sell) : 0;
}

} // namespace

namespace b200 {

// Hacks [hack0, hack1) (the stream kernel and the SELL-P route only take the whole matrix).
int hll_run_range(spmv_b200_hll *h, int kernel, int wpb, long long hack0, long long hack1,
                  const double *d_x, double *d_y, int epi_mode, const EpiArgs &epi_in,
                  void *stream) {
      if (!h)
            return fail(-EINVAL, "null HLL handle");
      if (h->n_hacks == 0 || hack1 <= hack0)
            return 0;
      if (hack0 < 0 || hack1 > h->n_hacks)
            return fail(-EINVAL, "hack range [%lld,%lld) out of bounds", hack0, hack1);
      wpb = clamp_wpb(wpb);
      cudaStream_t st = as_stream(stream);
      const int threads = 32 * wpb;
      const long long n = hack1 - hack0;
      const int grid = blocks_for(n * 32, threads);
      const bool whole = hack0 == 0 && hack1 == h->n_hacks;
      EpiArgs epi = epi_in;
      const bool want_dot = epi_mode == EPI_FUSED && epi.w && epi.dot_partial;
      double *dot_out = epi.dot_partial;
      long long dot_slots = 0;
      if (epi_mode == EPI_FUSED) {
            if (kernel != SPMV_B200_HLL_WARP_HACK || !whole)
                  return fail(-ENOTSUP, "the fused epilogue exists for HLL kernel 2, whole matrix");
            epi.dot_partial = nullptr;
            if (want_dot) {
                  if (ensure_dot(&h->d_dot_partial, &h->dot_cap, h->n_hacks))
                        return -ENOMEM;
                  epi.dot_partial = h->d_dot_partial;
                  dot_slots = h->n_hacks;
            }
      }
      switch (kernel) {
      case SPMV_B200_HLL_THREAD_ROW_RM:
      case SPMV_B200_HLL_THREAD_ROW:
            hll_warp_kernel<EPI_PLAIN><<<grid, threads, 0, st>>>(h->d_hoff, h->d_ja, h->d_as, hack0,
                                                                 hack1, h->M, d_x, d_y, epi);
            break;
      case SPMV_B200_HLL_WARP_HACK: {
            // x larger than the L2 and scattered columns: column panels (sell_kernels.cuh); the
            // slices are built on the GPU from this very HLL
            if (whole && hll_wants_sell(h) && hll_ensure_sell(h) == 0 &&
                (epi_mode != EPI_FUSED || h->sell.K == 1)) {
                  sell_run(h->sell, wpb, d_x, d_y, epi_mode, epi, st);
                  --g_counters.launches; // counted again below
                  break;
            }
            // Measured (profiles/r1_kbench_c2_sweep.txt): lane = row with 64/32-bit loads wins
            // whenever the gather is cache friendly (C2: 99 % vs 97 % / 88 % for 256/128-bit and
            // 128/64-bit loads, whose lanes share rows and split their gathers).
            // narrow hacks: persistent warps, each with its own ring of bulk-copied hacks (hll_pipe_kernel)
            if (g_knobs.hll_pipe != 0 && h->max_width > 0 && h->max_width <= kHllPipeMaxWidth &&
                (g_knobs.hll_pipe > 0 || n >= 4ll * g_sm_count * 8)) {
                  constexpr int kStages = 2, kWarps = 8;
                  const int capw = 32 * h->max_width; // 3.8 KB per warp for width 5: 48 warps per SM
                  const size_t smem = (size_t)kWarps * kStages * capw * 12 + (size_t)kWarps * kStages * 8;
                  const int fu = epi_mode == EPI_FUSED;
                  static int occ_by_dev[2][kHllPipeMaxWidth + 1][kMaxDevices] = {{{0}}};
                  int &occ = occ_by_dev[fu][h->max_width][h->device % kMaxDevices];
                  if (!occ) {
                        if (fu) {
                              B200_CUDA(cudaFuncSetAttribute(hll_pipe_kernel<kStages, EPI_FUSED>,
                                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 100 << 10));
                              B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                                  &occ, hll_pipe_kernel<kStages, EPI_FUSED>, kWarps * 32, smem));
                        } else {
                              B200_CUDA(cudaFuncSetAttribute(hll_pipe_kernel<kStages, EPI_PLAIN>,
                                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 100 << 10));
                              B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                                  &occ, hll_pipe_kernel<kStages, EPI_PLAIN>, kWarps * 32, smem));
                        }
                        if (occ < 1)
                              return fail(-EINVAL, "hll_pipe_kernel does not fit on an SM");
                  }
                  const int g = (int)std::min<long long>((n + kWarps - 1) / kWarps, (long long)occ * g_sm_count);
                  if (fu)
                        hll_pipe_kernel<kStages, EPI_FUSED><<<g, kWarps * 32, smem, st>>>(
                            h->d_hoff, h->d_ja, h->d_as, hack0, hack1, capw, h->M, d_x, d_y, epi);
                  else
                        hll_pipe_kernel<kStages, EPI_PLAIN><<<g, kWarps * 32, smem, st>>>(
                            h->d_hoff, h->d_ja, h->d_as, hack0, hack1, capw, h->M, d_x, d_y, epi);
                  break;
            }
            if (epi_mode == EPI_FUSED)
                  hll_warp_kernel<EPI_FUSED><<<grid, threads, 0, st>>>(
                      h->d_hoff, h->d_ja, h->d_as, hack0, hack1, h->M, d_x, d_y, epi);
            else
                  hll_warp_kernel<EPI_PLAIN><<<grid, threads, 0, st>>>(
                      h->d_hoff, h->d_ja, h->d_as, hack0, hack1, h->M, d_x, d_y, epi);
            break;
      }
      case SPMV_B200_HLL_STREAM: {
            if (!whole)
                  return fail(-ENOTSUP, "the staged HLL kernel runs on the whole matrix only");
            const int cfg = hll_stream_cfg_for(wpb);
            auto &t = h->stream[cfg];
            if (!t.built) {
                  int rc = hll_build_tiles(h, kHllStreamShapes[cfg].warps,
                                           kHllStreamShapes[cfg].cap, t);
                  if (rc)
                        return rc;
            }
            switch (cfg) {
#define X(id, W, S, C)                                                                             \
      case id: {                                                                                   \
            auto kern = hll_stream_kernel<W, S, C>;                                                \
            constexpr size_t smem = (size_t)S * C * 12 + S * 8 + 16;                               \
            static int occ_by_dev[kMaxDevices] = {0};                                              \
            int rc = stream_occupancy(kern, W * 32, smem, h->device, occ_by_dev);                  \
            if (rc)                                                                                \
                  return rc;                                                                       \
            const int g = std::min(t.n_tiles, occ_by_dev[h->device % kMaxDevices] * g_sm_count);   \
            kern<<<g, W * 32, smem, st>>>(h->d_hoff, h->d_ja, h->d_as, t.d_tile_h, t.n_tiles,      \
                                          h->M, d_x, d_y);                                         \
            break;                                                                                 \
      }
                  HLL_STREAM_CONFIGS(X)
#undef X
            }
            break;
      }
      default:
            return fail(-EINVAL, "unknown HLL kernel id %d", kernel);
      }
      ++g_counters.launches;
      if (want_dot) {
            dot_reduce_kernel<<<1, 1024, 0, st>>>(h->d_dot_partial, dot_slots, dot_out);
            ++g_counters.launches;
      }
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess)
            return fail(-EIO, "HLL kernel %d launch failed: %s", kernel, cudaGetErrorString(e));
      return 0;
}

} // namespace b200

static spmv_b200_hll *hll_alloc_shell(long long M, long long N, long long NZ, long long n_hacks, int device) {
      auto *h = new spmv_b200_hll();
      h->M = M, h->N = N, h->NZ = NZ, h->n_hacks = n_hacks, h->device = device;
      return h;
}

// Both HLL constructors return through here once the shell exists.  rc != 0: a step failed (fail()
// has set the message), so the shell is destroyed.  Otherwise the fill is waited for (`what` names
// it if it failed) and the handle takes `span` as its gather span, or measures it when `span` < 0.
static spmv_b200_hll *hll_finish(spmv_b200_hll *h, int rc, double span, const char *what) {
      const cudaError_t e = rc ? cudaSuccess : cudaDeviceSynchronize();
      if (e != cudaSuccess)
            rc = fail(-EIO, "%s failed: %s", what, cudaGetErrorString(e));
      if (rc) {
            spmv_b200_hll_destroy(h);
            return nullptr;
      }
      h->gather_span = span >= 0 ? span : measure_gather_span(hll_src(h), h->M, h->N);
      return h;
}

// Gather the per-hack host arrays into one staging copy (hack b from slot src_off[b]), ship it, and
// let the GPU transpose / re-stride / patch the pads.
static int hll_fill_from_host(spmv_b200_hll *h, const sparse_hll *H, const std::vector<long long> &src_off,
                              int is_col_major) {
      static const char *what = "HLL upload";
      const long long src_slots = src_off.back();
      // not std::vector: its zero fill would be one more pass over the matrix
      std::unique_ptr<int[]> st_ja(new (std::nothrow) int[src_slots]);
      std::unique_ptr<double[]> st_as(new (std::nothrow) double[src_slots]);
      if (!st_ja || !st_as)
            return fail(-ENOMEM, "host staging allocation failed (%lld slots)", src_slots);
#pragma omp parallel for schedule(static, 256)
      for (long long b = 0; b < h->n_hacks; ++b) {
            const size_t n = (size_t)(src_off[b + 1] - src_off[b]);
            memcpy(st_ja.get() + src_off[b], H->blocks[b].JA, n * sizeof(int));
            memcpy(st_as.get() + src_off[b], H->blocks[b].AS, n * sizeof(double));
      }
      DeviceTemps tmp;
      int *d_sja = nullptr;
      double *d_sas = nullptr;
      long long *d_soff = nullptr;
      if (tmp.alloc(&d_sja, (size_t)src_slots * sizeof(int), what) ||
          tmp.alloc(&d_sas, (size_t)src_slots * sizeof(double), what) ||
          tmp.alloc(&d_soff, src_off.size() * sizeof(long long), what))
            return -ENOMEM;
      cudaError_t e = cudaMemcpy(d_sja, st_ja.get(), (size_t)src_slots * sizeof(int), cudaMemcpyHostToDevice);
      if (e == cudaSuccess)
            e = cudaMemcpy(d_sas, st_as.get(), (size_t)src_slots * sizeof(double), cudaMemcpyHostToDevice);
      if (e == cudaSuccess)
            e = cudaMemcpy(d_soff, src_off.data(), src_off.size() * sizeof(long long), cudaMemcpyHostToDevice);
      if (e != cudaSuccess)
            return fail(-EIO, "HLL upload failed: %s", cudaGetErrorString(e));
      g_counters.h2d += src_slots * 12;
      hll_fill_from_host_layout_kernel<<<blocks_for(h->n_hacks * 32, 256), 256>>>(
          d_soff, d_sja, d_sas, is_col_major, h->M, h->n_hacks, h->d_hoff, h->d_ja, h->d_as, h->d_rowlen);
      ++g_counters.launches;
      return 0;
}

extern "C" spmv_b200_hll *spmv_b200_hll_create(const sparse_hll *H, int is_col_major) {
      if (ensure_device())
            return nullptr;
      if (!H || (H->num_blocks > 0 && !H->blocks)) {
            fail(-EINVAL, "null sparse_hll");
            return nullptr;
      }
      if (H->hack_size != kHack) {
            fail(-EINVAL, "hack_size %d unsupported (library is built for 32)", H->hack_size);
            return nullptr;
      }
      int device = 0;
      cudaGetDevice(&device);
      spmv_b200_hll *h = hll_alloc_shell(H->M, H->N, H->NZ, H->num_blocks, device);
      std::vector<int> width((size_t)h->n_hacks);
      std::vector<long long> src_off((size_t)h->n_hacks + 1, 0);
      for (long long b = 0; b < h->n_hacks; ++b) {
            width[b] = H->blocks[b].max_NZ;
            src_off[b + 1] = src_off[b] + (long long)H->blocks[b].M * H->blocks[b].max_NZ;
      }
      int rc = hll_alloc(h, width);
      if (!rc && h->n_hacks > 0)
            rc = hll_fill_from_host(h, H, src_off, is_col_major);
      return hll_finish(h, rc, -1.0, "HLL layout kernel");
}

extern "C" spmv_b200_hll *spmv_b200_hll_from_csr(const spmv_b200_csr *A) {
      if (ensure_device())
            return nullptr;
      if (!A) {
            fail(-EINVAL, "null CSR handle");
            return nullptr;
      }
      spmv_b200_hll *h = hll_alloc_shell(A->M, A->N, A->NZ, (A->M + kHack - 1) / kHack, A->device);
      // hack widths (longest row of each hack) on the GPU; the host only needs them for the
      // prefix sum that sizes the buffers
      std::vector<int> width((size_t)h->n_hacks, 0);
      int rc = 0;
      if (h->n_hacks > 0) {
            DeviceTemps tmp;
            int *d_width = nullptr;
            rc = tmp.alloc(&d_width, width.size() * sizeof(int), "hack widths");
            if (!rc) {
                  with_offsets(A->wide, [&](auto t) {
                        using OffT = typename decltype(t)::type;
                        hll_width_kernel<OffT><<<blocks_for(h->n_hacks * 32, 256), 256>>>(
                            (const OffT *)A->d_irp, A->M, h->n_hacks, d_width);
                  });
                  ++g_counters.launches;
                  const cudaError_t e =
                      cudaMemcpy(width.data(), d_width, width.size() * sizeof(int), cudaMemcpyDeviceToHost);
                  if (e != cudaSuccess)
                        rc = fail(-EIO, "hack width kernel failed: %s", cudaGetErrorString(e));
            }
      }
      rc = rc ? rc : hll_alloc(h, width);
      if (!rc && h->n_hacks > 0) {
            with_offsets(A->wide, [&](auto t) {
                  using OffT = typename decltype(t)::type;
                  hll_fill_from_csr_kernel<OffT><<<blocks_for(h->n_hacks * 32, 256), 256>>>(
                      (const OffT *)A->d_irp, A->d_ja, A->d_as, A->M, h->n_hacks, h->d_hoff, h->d_ja,
                      h->d_as, h->d_rowlen);
            });
            ++g_counters.launches;
      }
      return hll_finish(h, rc, A->gather_span, "CSR->HLL kernel");
}

extern "C" void spmv_b200_hll_destroy(spmv_b200_hll *h) {
      if (!h)
            return;
      for (auto &kv : h->stream)
            cudaFree(kv.second.d_tile_h);
      free_sell(h->sell);
      cudaFree(h->d_dot_partial);
      cudaFree(h->d_hoff);
      cudaFree(h->d_ja);
      cudaFree(h->d_as);
      cudaFree(h->d_rowlen);
      delete h;
}

extern "C" int64_t spmv_b200_hll_rows(const spmv_b200_hll *h) { return h ? h->M : -1; }
extern "C" int64_t spmv_b200_hll_cols(const spmv_b200_hll *h) { return h ? h->N : -1; }
extern "C" int64_t spmv_b200_hll_nnz(const spmv_b200_hll *h) { return h ? h->NZ : -1; }
extern "C" int64_t spmv_b200_hll_num_hacks(const spmv_b200_hll *h) { return h ? h->n_hacks : -1; }
extern "C" int64_t spmv_b200_hll_slots(const spmv_b200_hll *h) { return h ? h->slots : -1; }

extern "C" int spmv_b200_hll_download(const spmv_b200_hll *h, int64_t *hoff, int *JA,
                                      double *AS) {
      if (!h)
            return fail(-EINVAL, "null HLL handle");
      if (hoff)
            std::copy(h->h_hoff.begin(), h->h_hoff.end(), hoff);
      if (JA && h->slots)
            B200_CUDA(
                cudaMemcpy(JA, h->d_ja, (size_t)h->slots * sizeof(int), cudaMemcpyDeviceToHost));
      if (AS && h->slots)
            B200_CUDA(cudaMemcpy(AS, h->d_as, (size_t)h->slots * sizeof(double),
                                 cudaMemcpyDeviceToHost));
      return 0;
}

extern "C" int spmv_b200_hll_sell_info(spmv_b200_hll *h, int build, int64_t *out, int n_out) {
      if (!h || !out)
            return fail(-EINVAL, "null argument");
      if (build && h->sell.state == 0)
            hll_ensure_sell(h);
      const SellPlan &sp = h->sell;
      const int64_t v[8] = {sp.state, sp.K, sp.sigma, sp.n_slices, sp.slots, sp.nnz_in_slices,
                            sp.n_long, (int64_t)(h->gather_span * 1e6)};
      for (int i = 0; i < n_out && i < 8; ++i)
            out[i] = v[i];
      return 0;
}

extern "C" int spmv_b200_hll_spmv(spmv_b200_hll *h, int kernel, int wpb, const double *d_x,
                                  double *d_y, void *stream) {
      return hll_run_range(h, kernel, wpb, 0, h ? h->n_hacks : 0, d_x, d_y, EPI_PLAIN, EpiArgs{},
                           stream);
}

extern "C" int spmv_b200_hll_spmv_fused(spmv_b200_hll *h, int kernel, int wpb, const double *d_x,
                                        double *d_y, double alpha, double beta, const double *d_z,
                                        const double *d_w, double *d_dot, void *stream) {
      EpiArgs e{};
      e.alpha = alpha, e.beta = beta;
      e.z = d_z;
      e.w = d_dot ? d_w : nullptr;
      e.dot_partial = d_dot;
      return hll_run_range(h, kernel, wpb, 0, h ? h->n_hacks : 0, d_x, d_y, EPI_FUSED, e, stream);
}

extern "C" int spmv_b200_hll_launches(const spmv_b200_hll *h, int kernel) {
      if (!h || h->n_hacks <= 0)
            return 0;
      if (kernel == SPMV_B200_HLL_WARP_HACK && h->sell.state == 1 &&
          hll_wants_sell(const_cast<spmv_b200_hll *>(h)))
            return h->sell.K;
      return 1;
}

extern "C" int spmv_b200_hll_time(spmv_b200_hll *h, int kernel, int wpb, const double *d_x,
                                  double *d_y, int warmup, int reps, int flush_l2, double *ms_out,
                                  void *stream) {
      return time_launches([&] { return spmv_b200_hll_spmv(h, kernel, wpb, d_x, d_y, stream); },
                           warmup, reps, flush_l2, ms_out, stream);
}

// ===================================================== library / device / mem

extern "C" const char *spmv_b200_last_error(void) { return tls_error(); }
extern "C" const char *spmv_b200_version(void) { return "spmv-b200 0.2 (sm_100a)"; }

extern "C" int spmv_b200_device_count(void) {
      int n = 0;
      return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

extern "C" int spmv_b200_set_device(int ordinal) {
      B200_CUDA(cudaSetDevice(ordinal));
      g_sm_count = 0; // re-query
      return ensure_device();
}

extern "C" int spmv_b200_device_info(spmv_b200_devinfo *out) {
      if (!out)
            return fail(-EINVAL, "null argument");
      int rc = ensure_device();
      if (rc)
            return rc;
      int dev = 0;
      cudaDeviceProp p;
      B200_CUDA(cudaGetDevice(&dev));
      B200_CUDA(cudaGetDeviceProperties(&p, dev));
      memset(out, 0, sizeof *out);
      snprintf(out->name, sizeof out->name, "%.127s", p.name);
      out->cc_major = p.major, out->cc_minor = p.minor;
      out->sm_count = p.multiProcessorCount;
      out->l2_bytes_mb = (int)(p.l2CacheSize >> 20);
      out->hbm_bytes = (int64_t)p.totalGlobalMem;
      out->max_smem_per_block = (int)p.sharedMemPerBlockOptin;
      return 0;
}

extern "C" void *spmv_b200_dmalloc(size_t bytes) {
      if (ensure_device())
            return nullptr;
      void *p = nullptr;
      B200_CUDA_PTR(cudaMalloc(&p, bytes ? bytes : 1));
      return p;
}
extern "C" int spmv_b200_dfree(void *d_ptr) {
      B200_CUDA(cudaFree(d_ptr));
      return 0;
}
extern "C" int spmv_b200_h2d(void *d_dst, const void *src, size_t bytes, void *stream) {
      B200_CUDA(cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, as_stream(stream)));
      g_counters.h2d += (long long)bytes;
      return 0;
}
extern "C" int spmv_b200_d2h(void *dst, const void *d_src, size_t bytes, void *stream) {
      B200_CUDA(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, as_stream(stream)));
      g_counters.d2h += (long long)bytes;
      return 0;
}
extern "C" int spmv_b200_dmemset(void *d_dst, int byte, size_t bytes, void *stream) {
      B200_CUDA(cudaMemsetAsync(d_dst, byte, bytes, as_stream(stream)));
      return 0;
}
extern "C" int spmv_b200_stream_sync(void *stream) {
      B200_CUDA(cudaStreamSynchronize(as_stream(stream)));
      return 0;
}
extern "C" void *spmv_b200_host_alloc(size_t bytes) {
      if (ensure_device())
            return nullptr;
      void *p = nullptr;
      B200_CUDA_PTR(cudaMallocHost(&p, bytes ? bytes : 1));
      return p;
}
extern "C" int spmv_b200_host_free(void *ptr) {
      B200_CUDA(cudaFreeHost(ptr));
      return 0;
}
// Reads `n` 16-byte words; the sum goes to a sink nobody reads (keeps the loads alive).
static __global__ void l2_read_kernel(const int4 *__restrict__ p, long long n, int *__restrict__ sink) {
      int acc = 0;
      for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
           i += (long long)gridDim.x * blockDim.x) {
            const int4 v = p[i];
            acc ^= v.x ^ v.y ^ v.z ^ v.w;
      }
      if (acc == 0x5a5a5a5b)
            *sink = acc;
}

// Evict the L2: overwrite a buffer four times its size, then READ the first half of it again.
// The write alone would leave the L2 full of DIRTY lines, and the kernel timed next would pay for
// their write-back (126 MB of extra DRAM traffic charged to an 80 MB SpMV); after the read pass
// the L2 holds clean lines of the scratch buffer only.
extern "C" int spmv_b200_flush_l2(void *stream) {
      int rc = ensure_device();
      if (rc)
            return rc;
      int dev = 0;
      B200_CUDA(cudaGetDevice(&dev));
      void *&buf = g_flush_buf[dev % kMaxDevices];
      if (!buf)
            B200_CUDA(cudaMalloc(&buf, kFlushBytes + 256));
      static int toggle = 0;
      B200_CUDA(cudaMemsetAsync(buf, ++toggle & 0xff, kFlushBytes, as_stream(stream)));
      l2_read_kernel<<<1184, 256, 0, as_stream(stream)>>>(static_cast<const int4 *>(buf),
                                                          (long long)(kFlushBytes / 2 / sizeof(int4)),
                                                          reinterpret_cast<int *>(static_cast<char *>(buf) + kFlushBytes));
      B200_CUDA(cudaGetLastError());
      return 0;
}

extern "C" void spmv_b200_set_timing(int warmup, int reps) {
      g_knobs.warmup = std::max(0, warmup);
      g_knobs.reps = std::max(0, reps); // 0: no separately timed launches (pipelined entry only)
}

extern "C" void spmv_b200_counters(int64_t *launches, int64_t *h2d_bytes, int64_t *d2h_bytes) {
      if (launches)
            *launches = g_counters.launches;
      if (h2d_bytes)
            *h2d_bytes = g_counters.h2d;
      if (d2h_bytes)
            *d2h_bytes = g_counters.d2h;
}

// Experiment knobs (kbench sweeps, tests).  Unknown keys return -EINVAL.
extern "C" int spmv_b200_set_knob(const char *key, int value) {
      if (!key)
            return -EINVAL;
      struct {
            const char *name;
            int *slot;
      } table[] = {{"csr_stream_cfg", &g_knobs.csr_stream_cfg},
                   {"hll_pipe", &g_knobs.hll_pipe},
                   {"csr_pipe", &g_knobs.csr_pipe},
                   {"csr_codes", &g_knobs.csr_codes},
                   {"hll_stream_cfg", &g_knobs.hll_stream_cfg},
                   {"force_wide", &g_knobs.force_wide},
                   {"pipeline", &g_knobs.pipeline},
                   {"pipe_chunks", &g_knobs.pipe_chunks},
                   {"sell", &g_knobs.sell},
                   {"sell_panels", &g_knobs.sell_panels},
                   {"sell_sigma", &g_knobs.sell_sigma},
                   {"sell_panel_mb", &g_knobs.sell_panel_mb},
                   {"sell_chunk", &g_knobs.sell_chunk},
                   {"sell_max_row", &g_knobs.sell_max_row},
                   {"cache", &g_knobs.cache}};
      for (auto &t : table)
            if (!strcmp(key, t.name)) {
                  *t.slot = value;
                  return 0;
            }
      return fail(-EINVAL, "unknown knob %s", key);
}
