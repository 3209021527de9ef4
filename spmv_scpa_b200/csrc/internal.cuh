// internal.cuh -- host-side state shared by the translation units of libspmv_b200
// (spmv_b200.cu: handles, plans, launchers; entry.cu: the reference-style entry points and the
// host-buffer pipelines; dist.cu: the multi-GPU iterated SpMV).  Not installed, not part of the
// C ABI.
#pragma once

#include <algorithm>
#include <cerrno>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <numeric>
#include <vector>

#include "common.cuh"

extern "C" {
#include "cuda_csr.h"
#include "cuda_hll.h"
#include "cuda_timer.h"
#include "spmv_b200.h"
}

namespace b200 {

struct Counters {
      long long launches = 0, h2d = 0, d2h = 0;
};
extern Counters g_counters;

struct Knobs {
      int csr_stream_cfg = -1; // -1: pick from warps_per_block and the row-length profile
      int csr_pipe = -1;       // short regular CSR rows through per-warp bulk-copy rings: -1 auto, 0 off, 1 whenever they fit
      int csr_codes = 1;       // row-tile stream plans stream column codes where they apply; 0: int32 columns
      int hll_pipe = -1;       // narrow hacks through per-warp bulk-copy rings: -1 auto, 0 off, 1 whenever they fit
      int hll_stream_cfg = -1;
      int force_wide = 0;      // use 64-bit row offsets even when NZ < 2^31 (tests)
      int pipeline = 1;        // host-buffer pipeline in the host-pointer entry points
      int pipe_chunks = 0;     // 0: by size
      int sell = -1;           // -1 auto, 0 never, 1 always route ids 2/4 (CSR) and 2 (HLL) to SELL-P
      int sell_panels = 0;     // 0: by size of x
      int sell_sigma = 16384;  // rows per sorting window
      int sell_panel_mb = 64;  // target size of a panel's x slice (C3 sweep: 64 MB beats 43 / 32 MB)
      int sell_max_row = 4096; // longer rows go to the CSR long-row kernels (panel mode)
      int sell_chunk = 256;    // ragged matrices: rows are cut into virtual rows of this many entries
                               // (C4 sweep: 32/64/128/256/512/1024 -> 34/42/45/46/44/39 %); 0 = off
      int cache = 1;           // entry-point matrix cache: 0 off, 1 full content hash, 2 trust pointers
      int warmup = 1, reps = 3;
};
extern Knobs g_knobs;

extern int g_sm_count;
constexpr int kMaxDevices = 64;
// hll_pipe_kernel: matrices whose widest hack has at most this many slot columns
constexpr int kHllPipeMaxWidth = 8;
// csr_pipe_kernel: segments whose longest row has at most this many entries
constexpr int kCsrPipeMaxRow = 8;

int ensure_device();

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
int upload(T **d, const std::vector<T> &h) {
      *d = nullptr;
      if (h.empty())
            return 0;
      B200_CUDA(cudaMalloc(d, h.size() * sizeof(T)));
      B200_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
      g_counters.h2d += (long long)(h.size() * sizeof(T));
      return 0;
}

inline int blocks_for(long long threads, int block) {
      return (int)((threads + block - 1) / block);
}
inline int clamp_wpb(int wpb) { return wpb < 1 ? 1 : (wpb > 32 ? 32 : wpb); }

// adaptive bins by row length
constexpr int kNumKinds = 8; // 0..5: 2^k lanes per row, 6: CTA per row, 7: split
constexpr long long kKindMax[kNumKinds] = {4, 8, 16, 32, 64, 2048, 65536, -1};
constexpr long long kSplitChunk = 32768;

inline int kind_of(long long len) {
      for (int k = 0; k < kNumKinds - 1; ++k)
            if (len <= kKindMax[k])
                  return k;
      return kNumKinds - 1;
}

struct RowList {
      int *d_rows = nullptr;
      long long n = 0;
};

struct SplitPlan {
      long long *d_k0 = nullptr, *d_k1 = nullptr;
      int *d_row = nullptr, *d_first = nullptr;
      double *d_partial = nullptr;
      int n_rows = 0, n_chunks = 0;
};

struct StreamPlan {
      int *d_tile_row = nullptr;
      long long *d_tile_k = nullptr;
      int n_tiles = 0;
      RowList long_lists[kNumKinds]; // rows that do not fit a stage, by kind (5..7)
      SplitPlan split;
      bool built = false;
      // column codes of the row-tile configurations (csr_kernels.cuh, stream_codes_kernel):
      // tile t's block is d_codes[d_code_off[t], d_code_off[t+1])
      int codes_state = 0; // 0 not tried, 1 built, -1 not applicable (a tile has too many offsets)
      long long *d_code_off = nullptr;
      unsigned char *d_codes = nullptr;
      long long code_bytes = 0;
      int max_dict = 0; // largest dictionary of a tile
};

struct Segment {
      long long r0 = 0, r1 = 0;
      // adaptive plan
      bool regular = false;
      bool lists_built = false;
      int base_kind = 0;
      RowList lists[kNumKinds];
      SplitPlan split;
      long long kind_rows[kNumKinds] = {0};
      long long max_len = 0; // longest row of the segment
      // stream plans, one per kernel configuration
      std::map<int, StreamPlan> stream;
};

// Column-panelled, window-sorted sliced ELLPACK built from a resident CSR or HLL (sell_kernels.cuh)
struct SellPlan {
      int state = 0; // 0 not tried, 1 built, -1 not applicable / failed
      int K = 0, sigma = 0;
      long long M = 0, n_slices = 0, slots = 0, nnz_in_slices = 0;
      std::vector<int> pc;      // K+1 panel bounds
      long long *d_soff = nullptr;
      int *d_perm = nullptr;
      int *d_ja = nullptr;
      double *d_as = nullptr;
      // virtual rows (ragged CSR, one panel): rows longer than `chunk` are cut into pieces whose
      // partial sums are combined per row; M then counts virtual rows
      int chunk = 0;
      long long n_rows = 0, n_split_rows = 0, n_partials = 0;
      int *d_split_row = nullptr, *d_split_first = nullptr;
      double *d_partial = nullptr;
      double *d_partial_mm = nullptr; // 4 partial sums per piece (SpMM), allocated on first use
      // rows too long for a slice (CSR source only): warp-per-row, CTA-per-row and split lists
      RowList long_warp;
      RowList long_block;
      SplitPlan long_split;
      long long n_long = 0;
};
void free_sell(SellPlan &sp);

} // namespace b200

struct spmv_b200_csr {
      long long M = 0, N = 0, NZ = 0, col_offset = 0;
      bool wide = false; // 64-bit row offsets
      void *d_irp = nullptr;
      int *d_ja = nullptr;
      double *d_as = nullptr;
      std::vector<long long> h_irp; // host copy of the row offsets (planning)
      std::vector<b200::Segment> segs;
      int device = 0;
      // gather locality of the matrix (col_extent_kernel sample): share of x one block of 256
      // consecutive rows spans, median over the sample; -1 = not measured yet
      double gather_span = -1.0;
      b200::SellPlan sell;
      b200::SellPlan sell_mm2, sell_mm4; // SpMM with 2 / 4 right-hand sides when it needs more column panels
      // host-buffer pipeline (banded matrices): row chunks with their own launch plans, and how
      // much of x each chunk needs to have arrived
      std::vector<b200::Segment> pipe_segs;
      std::vector<long long> pipe_x_hi; // x[0, pipe_x_hi[c]) must be on the device before chunk c
      int pipe_state = 0;               // 0 not tried, 1 usable, -1 not worth it
      // scratch for the fused epilogue (per-warp partial dot products)
      double *d_dot_partial = nullptr;
      long long dot_cap = 0;
};

struct spmv_b200_hll {
      long long M = 0, N = 0, NZ = 0, n_hacks = 0, slots = 0;
      int device = 0;
      long long *d_hoff = nullptr;
      int *d_ja = nullptr;
      double *d_as = nullptr;
      int *d_rowlen = nullptr; // entries per row (n_hacks * 32), pads excluded
      std::vector<long long> h_hoff;
      int max_width = 0; // widest hack
      struct Tiles {
            int *d_tile_h = nullptr;
            int n_tiles = 0;
            bool built = false;
      };
      std::map<int, Tiles> stream;
      double gather_span = -1.0;
      b200::SellPlan sell;
      // host-buffer pipeline: hack ranges and the x prefix each needs
      std::vector<long long> pipe_hack; // chunk c = hacks [pipe_hack[c], pipe_hack[c+1])
      std::vector<long long> pipe_x_hi;
      int pipe_state = 0;
      double *d_dot_partial = nullptr;
      long long dot_cap = 0;
};

namespace b200 {

// ---- spmv_b200.cu ----
int build_adaptive(spmv_b200_csr *h, Segment &sg);
void free_segment(Segment &sg);
int csr_run_segment(spmv_b200_csr *h, Segment &sg, int kernel, int wpb, const double *d_x,
                    double *d_y, int epi_mode, const EpiArgs &epi, cudaStream_t st);
int csr_run(spmv_b200_csr *h, int kernel, int wpb, long long row0, long long row1,
            const double *d_x, double *d_y, int epi_mode, const EpiArgs &epi, void *stream);
int csr_run_blocks(spmv_b200_csr *h, int kernel, int wpb, const double *d_x, double *d_y, void *stream,
                   int blocks, const std::function<void(long long, long long)> &done);
int hll_run_range(spmv_b200_hll *h, int kernel, int wpb, long long hack0, long long hack1,
                  const double *d_x, double *d_y, int epi_mode, const EpiArgs &epi, void *stream);
double median_of(std::vector<double> v);
// largest column index referenced by entries [k0, k1) of a resident CSR (device reduction)
int csr_max_col(const spmv_b200_csr *h, long long k0, long long k1, int *out);
int hll_max_col(const spmv_b200_hll *h, long long hack0, long long hack1, int *out);
int csr_check_columns(const spmv_b200_csr *h);

} // namespace b200
