// Shared helpers for libfemb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/femb200.h"

namespace femb {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const std::string& msg);

#define FEMB_CUDA(call)                                                                         \
  do {                                                                                          \
    cudaError_t _e = (call);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      femb::set_error(std::string(#call) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ +   \
                      ":" + std::to_string(__LINE__) + ")");                                    \
      return FEMB_ERR_CUDA;                                                                     \
    }                                                                                           \
  } while (0)

#define FEMB_CHECK_ARG(cond, msg)                                                               \
  do {                                                                                          \
    if (!(cond)) {                                                                              \
      femb::set_error(std::string("invalid argument: ") + msg);                                 \
      return FEMB_ERR_ARG;                                                                      \
    }                                                                                           \
  } while (0)

#define FEMB_LAUNCH_CHECK() FEMB_CUDA(cudaGetLastError())

inline cudaStream_t as_stream(femb_stream s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- stream-ordered scratch memory ----------------------------------------------------------
// The C ABI never allocates user-visible memory; scratch comes from the CUDA stream-ordered pool.
struct Scratch {
  cudaStream_t stream;
  void* ptrs[32];
  int n = 0;
  explicit Scratch(cudaStream_t s) : stream(s) { keep_pool_warm(); }
  // The default pool hands memory back to the driver at every synchronisation unless a release threshold is set;
  // re-acquiring hundreds of MB per call costs milliseconds.
  static void keep_pool_warm() {
    static thread_local int done_for = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done_for = dev;
  }
  template <typename T>
  cudaError_t alloc(T** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMallocAsync(&q, (count ? count : 1) * sizeof(T), stream);
    if (e == cudaSuccess && n < 32) ptrs[n++] = q;
    *p = static_cast<T*>(q);
    return e;
  }
  ~Scratch() {
    for (int i = n - 1; i >= 0; --i) cudaFreeAsync(ptrs[i], stream);
  }
};

int num_sms();

// ---- per-(thread, device) solver context --------------------------------------------------------
// Stream capture is illegal on the legacy default stream (torch's default current stream), so the graph-captured solves run
// on a private non-blocking stream ordered after the caller's stream by an event.  Streams, events and the pinned status
// buffer belong to ONE device: they are kept in a table indexed by the current device (a solve on cuda:1 after one on
// cuda:0 in the same thread must not reuse device 0's stream).
struct SolveCtx {
  cudaStream_t stream = nullptr;
  cudaEvent_t order_ev = nullptr;
  cudaEvent_t poll_ev[2] = {nullptr, nullptr}, time_ev[2] = {nullptr, nullptr};
  void* pinned = nullptr;  // SOLVE_PINNED_BYTES of page-locked host memory (two status structs)
  // iteration-graph cache of the single-GPU CG (krylov.cu): the scalars / per-CTA partials live in a persistent device buffer so
  // that a repeated solve with the same operator, vectors and parameters finds every address baked into the graph unchanged and
  // re-launches the instantiated graph instead of capturing + instantiating again (~1 ms per solve: most of a small solve)
  void* dev_scratch = nullptr;
  size_t dev_scratch_bytes = 0;
  // 16-bit delta-encoded column index of the merged CG loop (krylov.cu, idx16_encode_kernel): failed-tile counter, one flag
  // byte per 128-row tile, then col16 (2 bytes per nonzero), re-encoded by every solve that uses it
  void* idx16 = nullptr;
  size_t idx16_bytes = 0;
  cudaGraphExec_t graph_exec = nullptr;
  unsigned char graph_key[512];
  size_t graph_key_bytes = 0;
};
constexpr size_t SOLVE_PINNED_BYTES = 1024;
// context of the CURRENT device with its stream ordered after `user`; nullptr (and set_error) on any CUDA failure
SolveCtx* solve_ctx(cudaStream_t user);

// ---- device helpers --------------------------------------------------------------------------
constexpr int SMS = 148;  // B200

template <typename I>
__device__ __forceinline__ long long ldidx(const I* p) { return static_cast<long long>(__ldg(p)); }

__device__ __forceinline__ void st256(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
__device__ __forceinline__ void st128(double* p, double a, double b) {
  asm volatile("st.global.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(a), "d"(b) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Fixed-order block reduction (deterministic): warp shuffles, then warp 0 sums the warp partials.
template <int THREADS>
__device__ __forceinline__ double block_sum(double v) {
  __shared__ double sh[THREADS / 32];
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double t = 0.0;
  if (w == 0) {
    t = lane < THREADS / 32 ? sh[lane] : 0.0;
    t = warp_sum(t);
  }
  __syncthreads();
  return t;  // valid in warp 0
}

// closed-form 3x3 inverse / determinant (row-major m[9])
template <typename T>
__device__ __forceinline__ T det3(const T* m) {
  return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}
template <typename T>
__device__ __forceinline__ T inv3(const T* m, T* r) {
  const T c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
  const T det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  const T id = T(1) / det;
  r[0] = c00 * id;
  r[1] = (m[2] * m[7] - m[1] * m[8]) * id;
  r[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  r[3] = c01 * id;
  r[4] = (m[0] * m[8] - m[2] * m[6]) * id;
  r[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  r[6] = c02 * id;
  r[7] = (m[1] * m[6] - m[0] * m[7]) * id;
  r[8] = (m[0] * m[4] - m[1] * m[3]) * id;
  return det;
}

inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
inline int grid_for(long long work_items, int per_block, int max_waves = 64) {
  long long b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  const long long cap = static_cast<long long>(SMS) * max_waves;
  return static_cast<int>(b < cap ? b : cap);
}

}  // namespace femb
