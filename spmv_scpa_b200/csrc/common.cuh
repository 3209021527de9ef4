// common.cuh -- error plumbing and sm_100a PTX wrappers shared by the kernels.
//
// New code (no reference counterpart: the reference checks no CUDA call and
// uses plain LDG / __ldg only, src/cuda_csr.cu, src/cuda_hll.cu).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libspmv_b200 is written for sm_100a (B200) only"
#endif

namespace b200 {

// ---------------------------------------------------------------- errors --
inline char *tls_error() {
      static thread_local char buf[512];
      return buf;
}

inline int fail(int code, const char *fmt, ...) {
      va_list ap;
      va_start(ap, fmt);
      vsnprintf(tls_error(), 512, fmt, ap);
      va_end(ap);
      fprintf(stderr, "[ERROR] libspmv_b200: %s\n", tls_error());
      return code;
}

#define B200_CUDA(call)                                                        \
      do {                                                                     \
            cudaError_t e_ = (call);                                           \
            if (e_ != cudaSuccess)                                             \
                  return ::b200::fail(-5 /*EIO*/, "%s failed: %s (%s:%d)",     \
                                      #call, cudaGetErrorString(e_), __FILE__, \
                                      __LINE__);                               \
      } while (0)

#define B200_CUDA_PTR(call)                                                    \
      do {                                                                     \
            cudaError_t e_ = (call);                                           \
            if (e_ != cudaSuccess) {                                           \
                  ::b200::fail(-5, "%s failed: %s (%s:%d)", #call,             \
                               cudaGetErrorString(e_), __FILE__, __LINE__);    \
                  return nullptr;                                              \
            }                                                                  \
      } while (0)

constexpr int kWarp = 32;
constexpr int kHack = 32;

// --------------------------------------------------------- cache policies --
// L2 eviction priorities are attached per access through a 64-bit policy
// operand (on sm_100 the bare .L2::evict_* qualifiers are only accepted on
// 256-bit loads).
__device__ __forceinline__ uint64_t policy_evict_first() {
      uint64_t p;
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
      return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
      uint64_t p;
      asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
      return p;
}

// ------------------------------------------------------- streaming loads --
// Matrix values / indices are read exactly once per SpMV: keep them out of
// L1 (no_allocate) and first in line for L2 eviction.  The asm statements are
// deliberately NOT volatile: everything they read is constant for the whole
// launch, and ptxas must be free to issue a batch of them back to back (a
// volatile load pins program order and serialises load -> use -> load).
__device__ __forceinline__ double ld_stream_f64(const double *p, uint64_t pol) {
      double v;
      asm("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;"
                   : "=d"(v)
                   : "l"(p), "l"(pol));
      return v;
}
__device__ __forceinline__ int ld_stream_s32(const int *p, uint64_t pol) {
      int v;
      asm("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;"
                   : "=r"(v)
                   : "l"(p), "l"(pol));
      return v;
}
// Same L2 priority but allowed to live in L1: sub-warp row groups re-touch the
// tail of a 32-byte sector on their next step.
__device__ __forceinline__ double ld_stream_l1_f64(const double *p, uint64_t pol) {
      double v;
      asm("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
      return v;
}
__device__ __forceinline__ int ld_stream_l1_s32(const int *p, uint64_t pol) {
      int v;
      asm("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
      return v;
}

// ------------------------------------------------------------- x gathers --
// The irregular gather of x goes through the read-only path, is allowed to
// live in L1, and is marked evict_last in L2 so the streamed matrix does not
// push it out.
__device__ __forceinline__ double ld_x(const double *p, uint64_t pol) {
      double v;
      asm("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;"
                   : "=d"(v)
                   : "l"(p), "l"(pol));
      return v;
}

// K consecutive values X[c*K .. c*K + K) of a row-major block of K right-hand sides (SpMM): one
// or two 16-byte loads out of the SAME 32-byte sector a single-vector gather would fetch for 8
// useful bytes.
template <int K>
__device__ __forceinline__ void ld_xk(const double *X, int c, uint64_t pol, double (&v)[K]) {
      static_assert(K == 2 || K == 4, "2 or 4 right-hand sides");
      // c < 0: no entry -> zeros, no load.  Predicated, not branched: the gathers of a batch must
      // all be in flight together.
      const double *p = X + (long long)(c < 0 ? 0 : c) * K;
#pragma unroll
      for (int j = 0; j < K; j += 2)
            asm("{\n\t"
                ".reg .pred q;\n\t"
                "setp.ge.s32 q, %4, 0;\n\t"
                "mov.f64 %0, 0d0000000000000000;\n\t"
                "mov.f64 %1, 0d0000000000000000;\n\t"
                "@q ld.global.nc.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;\n\t"
                "}"
                : "=d"(v[j]), "=d"(v[j + 1])
                : "l"(p + j), "l"(pol), "r"(c));
}

// --------------------------------------------------- mbarrier + bulk copy --
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
      return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                   "r"(bytes)
                   : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "WAIT_%=:\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
          "@p bra DONE_%=;\n"
          "bra WAIT_%=;\n"
          "DONE_%=:\n"
          "}\n" ::"r"(smem_u32(bar)),
          "r"(parity)
          : "memory");
}
// 1-D bulk copy global -> shared, completion counted in bytes on `bar`.
// Requirements: src, dst 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src, uint32_t bytes,
                                         uint64_t *bar, uint64_t pol) {
      asm volatile(
          "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
          "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
          "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
          : "memory");
}

// ------------------------------------------------------------ reductions --
template <int WIDTH>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
      for (int o = WIDTH / 2; o > 0; o >>= 1)
            v += __shfl_xor_sync(0xffffffffu, v, o, WIDTH);
      return v;
}

// ------------------------------------------------------------- epilogues --
// What happens to a finished row sum is a compile-time choice (template flag
// EPI of every kernel), so the single-GPU kernels carry none of the compares
// the multi-GPU or fused variants need.
//   EPI_PLAIN  y[row] = v
//   EPI_PUSH   ... and rows a neighbouring rank needs are also stored straight
//              into that rank's halo buffer (peer HBM mapped through CUDA IPC
//              or peer access, reached over NVLink): the multi-GPU halo
//              exchange fused into the SpMV epilogue
//   EPI_ACC    y[row] += v  (column panels after the first one)
//   EPI_ACC_PUSH  y[row] += v, and the finished sum goes to the peers like EPI_PUSH (last column
//              panel of a shard whose next x slice every peer needs: the all-gather of a general
//              matrix fused into the SpMV epilogue)
//   EPI_FUSED  y[row] = alpha*v + beta*z[row], and sum_i y[i]*w[i] is
//              accumulated per warp (iterated solvers: SpMV + axpby + dot in
//              one pass over the matrix)
constexpr int EPI_PLAIN = 0;
constexpr int EPI_PUSH = 1;
constexpr int EPI_ACC = 2;
constexpr int EPI_FUSED = 3;
constexpr int EPI_ACC_PUSH = 4;
constexpr int kMaxPush = 8; // peers one launch can store to (7 = every other GPU of an 8-GPU box)

struct EpiArgs {
      // EPI_PUSH
      int n_push;
      long long row0[kMaxPush], row1[kMaxPush];
      double *dst[kMaxPush];
      // EPI_FUSED (z, w, dot_partial may be null)
      double alpha, beta;
      const double *z, *w;
      double *dot_partial; // one slot per warp of the launch
};

template <int EPI>
__device__ __forceinline__ void store_y(double *y, long long row, double v, const EpiArgs &e,
                                        double &dot_acc) {
      if (EPI == EPI_ACC) {
            y[row] += v;
      } else if (EPI == EPI_FUSED) {
            double r = e.alpha * v;
            if (e.z)
                  r = fma(e.beta, e.z[row], r);
            y[row] = r;
            if (e.w)
                  dot_acc = fma(r, e.w[row], dot_acc);
      } else {
            if (EPI == EPI_ACC_PUSH)
                  v += y[row];
            y[row] = v;
            if (EPI == EPI_PUSH || EPI == EPI_ACC_PUSH) {
                  for (int i = 0; i < e.n_push; ++i)
                        if (row >= e.row0[i] && row < e.row1[i])
                              e.dst[i][row - e.row0[i]] = v;
            }
      }
}

// End of a warp's work in an EPI_FUSED kernel: lane 0 publishes the warp's
// partial dot product in slot `warp_slot` (deterministic: a fixed launch shape
// gives a fixed summation tree; dot_reduce_kernel adds the slots in order).
template <int EPI>
__device__ __forceinline__ void epi_finish_warp(const EpiArgs &e, double dot_acc,
                                                long long warp_slot) {
      if (EPI == EPI_FUSED) {
            if (e.dot_partial) {
                  dot_acc = group_sum<32>(dot_acc);
                  if ((threadIdx.x & 31) == 0)
                        e.dot_partial[warp_slot] = dot_acc;
            }
      }
}

// out[0] = sum of partial[0..n), fixed order (one CTA, strided then tree).
static __global__ void __launch_bounds__(1024)
    dot_reduce_kernel(const double *__restrict__ partial, long long n, double *__restrict__ out) {
      __shared__ double part[32];
      double acc = 0.0;
      for (long long i = threadIdx.x; i < n; i += blockDim.x)
            acc += partial[i];
      acc = group_sum<32>(acc);
      if ((threadIdx.x & 31) == 0)
            part[threadIdx.x >> 5] = acc;
      __syncthreads();
      if (threadIdx.x < 32) {
            double v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.0;
            v = group_sum<32>(v);
            if (threadIdx.x == 0)
                  out[0] = v;
      }
}

} // namespace b200
