// Device-side building blocks shared by the single-GPU solver (krylov.cu) and the multi-GPU solver (dist.cu).
#pragma once
#include <cstdlib>

#include "common.cuh"

namespace femb {

constexpr int SPMV_THREADS = 256;
constexpr int STREAM_CAP = 5632;  // products per CTA (44 KB of static shared memory)

__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ int ld_stream(const int* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
// x gathers: read-only path when x is immutable during the kernel, plain (coherent at L2, L1-cached) loads when peers
// write the ghost part of x before this kernel's flag wait (multi-GPU)
template <bool NC>
__device__ __forceinline__ double ld_x(const double* p) {
  if (NC) return __ldg(p);
  return *p;
}

// CSR-stream SpMV over the rows [0,n): a CTA owns R = 256/LR consecutive rows.  Their nonzeros form one contiguous slice
// of val/col, which the whole CTA streams with fully coalesced loads, multiplies by the gathered x and parks in shared
// memory; then LR lanes per row add up that row's products (index order within a lane, fixed shuffle tree across lanes).
// Short FEM rows (~15 nonzeros for P1) therefore cost no idle lanes and no per-row pointer chasing while streaming.
// Returns this thread's partial of sum_r y_r * x_r (only when `fused`), with masked rows forced to zero.
struct NoHaloWait {
  __device__ __forceinline__ void operator()() const {}
};

// `halo_row`: rows >= halo_row may read entries of x that another GPU is still writing; `wait` (block-uniform, may
// __syncthreads) is called once, right before this CTA touches its first such tile, so interior tiles overlap the exchange.
template <int LR, bool NC, typename Wait = NoHaloWait>
__device__ __forceinline__ double spmv_stream_rows(long long n, const int* __restrict__ crow, const int* __restrict__ col,
                                                   const double* __restrict__ val, const double* __restrict__ x, double* __restrict__ y,
                                                   const unsigned char* __restrict__ mask, bool accumulate, bool fused,
                                                   long long halo_row = 0x7fffffffffffffffll, Wait wait = Wait()) {
  constexpr int R = SPMV_THREADS / LR;
  __shared__ double prod[STREAM_CAP];
  __shared__ int rp[R + 1];
  const int tid = threadIdx.x, sub = tid % LR, lr = tid / LR;
  double dot = 0.0;
  bool waited = false;
  for (long long r0 = (long long)blockIdx.x * R; r0 < n; r0 += (long long)gridDim.x * R) {
    const int nr = (int)min((long long)R, n - r0);
    if (!waited && r0 + nr > halo_row) {
      wait();
      waited = true;
    }
    // the row's own x entry, mask byte and previous y are requested now so their latency hides behind the streaming phase
    // instead of sitting between the row sum and the tile's closing barrier
    double x_own = 0.0, y_prev = 0.0;
    bool keep = true;
    if (lr < nr && sub == 0) {
      if (fused) {
        x_own = ld_x<NC>(x + r0 + lr);
        if (mask) keep = mask[r0 + lr] != 0;
      }
      if (accumulate) y_prev = y[r0 + lr];
    }
    for (int t = tid; t <= nr; t += SPMV_THREADS) rp[t] = __ldg(crow + r0 + t);
    __syncthreads();
    const int s = rp[0], e = rp[nr];
    const bool fits = (e - s) <= STREAM_CAP;
    if (fits) {
      int j = s + tid;
      for (; j + 3 * SPMV_THREADS < e; j += 4 * SPMV_THREADS) {
        int c[4];
        double v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) c[q] = ld_stream(col + j + q * SPMV_THREADS), v[q] = ld_stream(val + j + q * SPMV_THREADS);
#pragma unroll
        for (int q = 0; q < 4; ++q) prod[j - s + q * SPMV_THREADS] = v[q] * ld_x<NC>(x + c[q]);
      }
      for (; j < e; j += SPMV_THREADS) prod[j - s] = ld_stream(val + j) * ld_x<NC>(x + ld_stream(col + j));
    }
    __syncthreads();
    double sum = 0.0;
    if (lr < nr) {
      const int a = rp[lr], b = rp[lr + 1];
      if (fits) {
        for (int j = a - s + sub; j < b - s; j += LR) sum += prod[j];
      } else {  // oversized slice (very long rows): read straight from global memory
        for (int j = a + sub; j < b; j += LR) sum += ld_stream(val + j) * ld_x<NC>(x + ld_stream(col + j));
      }
    }
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lr < nr && sub == 0) {
      const long long r = r0 + lr;
      if (accumulate) sum += y_prev;
      if (fused) {
        if (!keep) sum = 0.0;
        dot += sum * x_own;
      }
      y[r] = sum;
    }
    __syncthreads();
  }
  return dot;
}

// ---- TMA-pipelined CSR SpMV ------------------------------------------------------------------------------------------------
// Persistent CTAs; the val/col slice of each row tile is brought into shared memory by the TMA engine
// (cp.async.bulk, 1-D, completion on an mbarrier) STAGES-1 tiles ahead of the arithmetic, so the matrix stream -- 90 % of
// the bytes -- is always in flight, independent of how many warps are stalled on the x gathers.  Each row is then owned
// by LR lanes that walk their slice of the staged tile (odd row lengths => conflict-free LDS), gather x through L1/L2
// eight at a time and accumulate in registers: no product buffer, no second pass.  Slices are aligned down to 4 entries so
// both copies are 16-byte aligned; tiles that do not fit a stage, and the last tile of the matrix (the aligned copy could
// run past the end of val/col), take the direct global-load path.
// Measured on B200, 64 M-tet Poisson operator (2.145 GB algorithmic): 0.38 ms = 5.7 TB/s with (128 threads, 2 stages,
// 2304 entries) x 4 CTAs/SM or (64, 2, 1152) x 8; 0.66 ms with only 2 CTAs/SM; the LDG-streaming kernel above: 0.52 ms.
__device__ __forceinline__ unsigned smem_u32(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Same copy with an L2 evict-first policy: the matrix stream is read once per SpMV, so it should not displace the CG vectors
// (x gathers, and u/r/p/Ap of the vector kernels), which fit in the 126 MB L2 once the operator is split over several GPUs.
__device__ __forceinline__ unsigned long long l2_evict_first_policy() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, unsigned bytes, unsigned long long* bar, unsigned long long pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}
// L2 residency of the matrix head: when the operator is only a few times larger than the 126 MB L2 (the per-rank block of a
// strong-scaled solve), the first `pin` bytes of val/col are staged with an evict_last policy and so survive from one SpMV
// to the next, while the rest keeps streaming evict_first; those tiles then cost no HBM traffic.  At 1 GPU on the 64 M-tet
// operator (1.9 GB) the pinned share is 3 % and changes nothing; at 8 GPUs (241 MB per rank) it is a quarter of the stream.
__device__ __forceinline__ unsigned long long l2_evict_last_policy() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
static __device__ int g_spmv_l2_hint = 1;  // per translation unit; FEMB_SPMV_L2HINT=0 switches the hint off (A/B runs)
static inline void spmv_apply_env_once() {  // call outside stream capture, before the first launch
  static thread_local int done_for = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
  done_for = dev;
  if (const char* e = getenv("FEMB_SPMV_L2HINT")) {
    const int v = atoi(e);
    cudaMemcpyToSymbol(g_spmv_l2_hint, &v, sizeof(int));
  }
}
// nonzeros (from the start of val/col) to keep L2-resident across SpMVs of one solve: FEMB_SPMV_PIN_MB overrides the rule
inline long long spmv_pin_entries(long long nnz) {
  static const double env_mb = getenv("FEMB_SPMV_PIN_MB") ? atof(getenv("FEMB_SPMV_PIN_MB")) : -1.0;
  const double bytes = 12.0 * (double)nnz;
  double pin_mb = env_mb;
  if (pin_mb < 0.0) pin_mb = 0.0;  // measured on the 8-GPU per-rank problem (243 MB operator): 0 / 24 / 48 / 72 / 96 MB pinned ->
                                   // 57.9 / 58.8 / 59.8 / 62.7 / 63.2 us per CG iteration -- the pinned lines displace the vectors; off
  return (long long)std::min(bytes, pin_mb * 1e6) / 12;
}

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------------
// Both kernels of a CG iteration are launched with cudaLaunchAttributeProgrammaticStreamSerialization inside the graph:
// a kernel signals `launch_dependents` as soon as it starts, so the next kernel's CTAs become resident while this one
// drains, run their prologue (barrier init, first TMA stages of the read-only matrix) and park in `griddepcontrol.wait`
// until this grid has completed and flushed.  Without the launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
struct PdlWait {
  __device__ __forceinline__ void operator()() const { pdl_wait(); }
};
struct NoDep {
  __device__ __forceinline__ void operator()() const {}
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid), cfg.blockDim = dim3((unsigned)block), cfg.dynamicSmemBytes = smem, cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at, cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// bit 0: the vector kernel is launched programmatically behind the SpMV, bit 1: the SpMV behind the vector kernel.
// Measured (1 GPU, us per CG iteration, 64 M-tet operator / the 8-GPU per-rank operator): mode 0 507.1 / 57.5, mode 1
// 533.1 / 57.6 (vector CTAs parked beside the running SpMV slow it down), mode 2 503.4 / 57.3, mode 3 648.9 / 57.7.
// Graph launch gaps are already ~1-2 us, so only mode 2 (the SpMV's barrier init and first TMA stages overlap the vector
// kernel's tail) is kept as the default.
inline int pdl_mode() {
  static const int m = getenv("FEMB_NO_PDL") ? 0 : (getenv("FEMB_PDL_MODE") ? atoi(getenv("FEMB_PDL_MODE")) : 2);
  return m;
}
inline bool pdl_enabled() { return pdl_mode() != 0; }

constexpr int TMA_THREADS = 128, TMA_STAGES = 2, TMA_CAP = 2304, TMA_CTAS_PER_SM = 4;
constexpr size_t TMA_SMEM = (size_t)TMA_STAGES * TMA_CAP * 12;

// Needs TMA_SMEM bytes of dynamic shared memory and blockDim.x == THREADS.  Returns this thread's partial of y.x (fused).
// `dep` runs once after the first stages are in flight and before anything but the (read-only) matrix is touched: the PDL
// wait of graph-captured loops.  `stop` (read after dep) aborts the tile loop: the staged copies are drained first, a CTA must
// not exit with bulk copies still landing in its shared memory.  `pin` = leading nonzeros staged evict_last (see above).
template <int LR, bool NC, int THREADS = TMA_THREADS, int STAGES = TMA_STAGES, int CAP = TMA_CAP, typename Wait = NoHaloWait,
          typename Dep = NoDep>
__device__ __forceinline__ double spmv_tma_rows(long long n, long long nnz, const int* __restrict__ crow, const int* __restrict__ col,
                                                const double* __restrict__ val, const double* __restrict__ x, double* __restrict__ y,
                                                const unsigned char* __restrict__ mask, bool accumulate, bool fused,
                                                long long halo_row = 0x7fffffffffffffffll, Wait wait = Wait(),
                                                const double* __restrict__ rvec = nullptr, double* extra = nullptr, Dep dep = Dep(),
                                                const int* stop = nullptr, long long pin = 0, const double* __restrict__ wvec = nullptr) {
  // wvec (merged-reduction Jacobi-PCG): the two extra sums carry the preconditioner's diagonal, extra[0] += y_r w_r rvec_r,
  // extra[1] += y_r^2 w_r
  // rvec/extra (merged-reduction CG): extra[0] += y_r * rvec_r, extra[1] += y_r * y_r for the rows this thread finishes
  constexpr int R = THREADS / LR;
  extern __shared__ __align__(128) unsigned char tma_smem[];
  double* vbuf = reinterpret_cast<double*>(tma_smem);                           // [STAGES][CAP]
  int* cbuf = reinterpret_cast<int*>(tma_smem + sizeof(double) * STAGES * CAP);  // [STAGES][CAP]
  __shared__ unsigned long long full[STAGES];
  __shared__ int base[STAGES];  // first staged entry of the tile (aligned down), -1 = not staged (direct path)
  const int tid = threadIdx.x, sub = tid % LR, lr = tid / LR;
  const long long ntiles = (n + R - 1) / R;
  const bool use_hint = g_spmv_l2_hint != 0;
  const unsigned long long pol = l2_evict_first_policy(), pol_keep = l2_evict_last_policy();
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // producer (thread 0): the row-pointer pair of the tile it will stage next is requested one iteration early, so issuing
  // the copies never waits on a global load while the other threads sit at the barrier
  auto bounds = [&](long long k, int& a, int& b) {
    const long long t = blockIdx.x + k * gridDim.x;
    a = b = 0;
    if (t < ntiles) a = __ldg(crow + t * R), b = __ldg(crow + min(n, t * R + R));
  };
  auto stage_tile = [&](long long k, int a, int b) {
    if (blockIdx.x + k * gridDim.x >= ntiles) return;
    const int s = (int)(k % STAGES);
    const int a0 = a & ~3, cnt = (b - a0 + 3) & ~3;
    if (cnt > CAP || (long long)a0 + cnt > nnz || cnt == 0) {
      base[s] = -1;
      return;
    }
    base[s] = a0;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&full[s], (unsigned)cnt * 12u);
    if (use_hint) {
      const unsigned long long pl = (long long)a0 + cnt <= pin ? pol_keep : pol;
      bulk_g2s_hint(vbuf + (size_t)s * CAP, val + a0, (unsigned)cnt * 8u, &full[s], pl);
      bulk_g2s_hint(cbuf + (size_t)s * CAP, col + a0, (unsigned)cnt * 4u, &full[s], pl);
    } else {
      bulk_g2s(vbuf + (size_t)s * CAP, val + a0, (unsigned)cnt * 8u, &full[s]);
      bulk_g2s(cbuf + (size_t)s * CAP, col + a0, (unsigned)cnt * 4u, &full[s]);
    }
  };
  int na = 0, nb = 0;  // bounds of the next tile to stage (thread 0 only)
  if (tid == 0) {
    for (int k = 0; k < STAGES - 1; ++k) {
      bounds(k, na, nb);
      stage_tile(k, na, nb);
    }
    bounds(STAGES - 1, na, nb);
  }
  double dot = 0.0;
  unsigned phase_bits = 0;  // parity per stage
  bool waited = false;
  dep();  // everything above touched only crow/col/val; x, y, rvec, mask-independent state below may come from the previous kernel
  if (stop) {  // sticky stop flag (block-uniform through shared memory): drain what was staged, then leave
    __shared__ int stop_sh;
    if (tid == 0) stop_sh = *(volatile const int*)stop;
    __syncthreads();
    if (stop_sh) {
      for (int k = 0; k < STAGES - 1; ++k)
        if (blockIdx.x + (long long)k * gridDim.x < ntiles && base[k % STAGES] >= 0) mbar_wait(&full[k % STAGES], 0u);
      return 0.0;
    }
  }
  for (long long k = 0;; ++k) {
    const long long t = blockIdx.x + k * gridDim.x;
    if (t >= ntiles) break;
    const int s = (int)(k % STAGES);
    if (!waited && min(n, t * R + R) > halo_row) {  // first tile of this CTA that may read ghost entries of x
      wait();
      waited = true;
    }
    if (tid == 0) {  // refill the stage that was drained in iteration k-1, then request the bounds of the tile after it
      stage_tile(k + STAGES - 1, na, nb);
      bounds(k + STAGES, na, nb);
    }
    const long long r = t * R + lr;
    int ra = 0, rb = 0;
    double x_own = 0.0, y_prev = 0.0, r_own = 0.0, w_own = 1.0;
    bool keep = true;
    if (r < n) {
      ra = __ldg(crow + r), rb = __ldg(crow + r + 1);
      if (sub == 0) {
        if (fused) {
          x_own = ld_x<NC>(x + r);
          if (mask) keep = mask[r] != 0;
          if (rvec) r_own = rvec[r];
          if (wvec) w_own = wvec[r];
        }
        if (accumulate) y_prev = y[r];
      }
    }
    __syncthreads();  // base[s] written by thread 0 (this or an earlier iteration) is visible
    const int a0 = base[s];
    double sum = 0.0;
    if (a0 >= 0) {
      mbar_wait(&full[s], (phase_bits >> s) & 1u);
      phase_bits ^= 1u << s;
      const double* vs = vbuf + (size_t)s * CAP - a0;
      const int* cs = cbuf + (size_t)s * CAP - a0;
      int j = ra + sub;
      for (; j + 7 * LR < rb; j += 8 * LR) {  // eight independent x gathers in flight per lane
        double xv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) xv[q] = ld_x<NC>(x + cs[j + q * LR]);
#pragma unroll
        for (int q = 0; q < 8; ++q) sum += vs[j + q * LR] * xv[q];
      }
      {  // tail: up to seven more, still issued together
        double xv[7];
#pragma unroll
        for (int q = 0; q < 7; ++q) xv[q] = (j + q * LR < rb) ? ld_x<NC>(x + cs[j + q * LR]) : 0.0;
#pragma unroll
        for (int q = 0; q < 7; ++q)
          if (j + q * LR < rb) sum += vs[j + q * LR] * xv[q];
      }
    } else {
      for (int j = ra + sub; j < rb; j += LR) sum += ld_stream(val + j) * ld_x<NC>(x + ld_stream(col + j));
    }
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (r < n && sub == 0) {
      if (accumulate) sum += y_prev;
      if (fused) {
        if (!keep) sum = 0.0;
        dot += sum * x_own;
        if (extra) extra[0] += sum * (w_own * r_own), extra[1] += sum * (sum * w_own);
      }
      y[r] = sum;
    }
    __syncthreads();  // the stage is drained: thread 0 may refill it in the next iteration
  }
  return dot;
}

// lanes per row for the TMA kernel: the smallest LR whose R = THREADS/LR rows keep a tile within one stage
inline int tma_pick_lr(long long n, long long nnz) {
  const double avg = n > 0 ? (double)nnz / (double)n : 1.0;
  for (int lr = 1; lr <= 32; lr *= 2)
    if ((TMA_THREADS / lr) * avg * 1.15 <= TMA_CAP) return lr;
  return 32;
}
inline int tma_grid(long long n, int lr) {
  const long long tiles = (n + TMA_THREADS / lr - 1) / (TMA_THREADS / lr);
  return (int)std::max<long long>(1, std::min<long long>(tiles, (long long)SMS * TMA_CTAS_PER_SM));
}

// IDX16 variant (LR = 1): 10 bytes per staged entry.  A full 128-row tile of the P1 Kuhn-cube operator (15 nonzeros per row)
// needs 1927 entries with the 8-entry alignment.  The -D overrides exist for the stage / CTA sweep (DESIGN 3.4).
#ifndef FEMB_TMA16_STAGES
#define FEMB_TMA16_STAGES 2
#endif
#ifndef FEMB_TMA16_CAP
#define FEMB_TMA16_CAP 2176
#endif
#ifndef FEMB_TMA16_CTAS
#define FEMB_TMA16_CTAS 5
#endif
constexpr int TMA16_STAGES = FEMB_TMA16_STAGES, TMA16_CAP = FEMB_TMA16_CAP, TMA16_CTAS_PER_SM = FEMB_TMA16_CTAS;
constexpr size_t TMA16_SMEM = (size_t)TMA16_STAGES * TMA16_CAP * 10;
inline int tma16_grid(long long n) {
  const long long tiles = (n + TMA_THREADS - 1) / TMA_THREADS;
  return (int)std::max<long long>(1, std::min<long long>(tiles, (long long)SMS * TMA16_CTAS_PER_SM));
}

// 16-bit-index twin of spmv_tma_rows<1, true, ..., NoHaloWait, PdlWait> for the merged CG loop (a sibling, so the int32 kernels
// of krylov.cu and dist.cu compile exactly as before).  The staged index stream is col16 (idx16_encode_kernel, krylov.cu):
// col16[a] = r - col[a] for the first entry a of row r, col16[j] = col[j] - col[j-1] after it, i.e. 10 instead of 12 bytes per
// staged nonzero.  One lane owns a row and rebuilds its columns with one running add per entry; the products are summed in the
// int32 kernel's order, so y is bit-identical.  A tile whose tile_ok byte is 0, that does not fit a stage, or whose val copy
// would run past nnz (col16 itself is padded) takes the direct path from the int32 col.  Slices start at a multiple of 8
// entries (16-byte aligned 2-byte copy); val is copied in pairs of entries.
template <int STAGES, int CAP>
__device__ __forceinline__ double spmv_tma16_rows(long long n, long long nnz, const int* __restrict__ crow, const int* __restrict__ col,
                                                  const unsigned short* __restrict__ col16, const unsigned char* __restrict__ tile_ok,
                                                  const double* __restrict__ val, const double* __restrict__ x, double* __restrict__ y,
                                                  const unsigned char* __restrict__ mask, bool accumulate, bool fused,
                                                  const double* __restrict__ rvec, double* extra, const int* stop, long long pin,
                                                  const double* __restrict__ wvec) {
  static_assert(CAP % 8 == 0, "16-byte aligned stages");
  constexpr int R = TMA_THREADS;
  extern __shared__ __align__(128) unsigned char tma_smem[];
  double* vbuf = reinterpret_cast<double*>(tma_smem);                                                 // [STAGES][CAP]
  unsigned short* dbuf = reinterpret_cast<unsigned short*>(tma_smem + sizeof(double) * STAGES * CAP);  // [STAGES][CAP]
  __shared__ unsigned long long full[STAGES];
  __shared__ int base[STAGES];  // first staged entry of the tile (aligned down), -1 = not staged (direct path)
  const int tid = threadIdx.x;
  const long long ntiles = (n + R - 1) / R;
  const bool use_hint = g_spmv_l2_hint != 0;
  const unsigned long long pol = l2_evict_first_policy(), pol_keep = l2_evict_last_policy();
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // producer (thread 0): row-pointer pair and flag of the tile it stages next are requested one iteration early
  auto bounds = [&](long long k, int& a, int& b, int& ok) {
    const long long t = blockIdx.x + k * gridDim.x;
    a = b = ok = 0;
    if (t < ntiles) a = __ldg(crow + t * R), b = __ldg(crow + min(n, t * R + R)), ok = __ldg(tile_ok + t);
  };
  auto stage_tile = [&](long long k, int a, int b, int ok) {
    if (blockIdx.x + k * gridDim.x >= ntiles) return;
    const int s = (int)(k % STAGES);
    const int a0 = a & ~7, cnt = (b - a0 + 7) & ~7, cntv = (b - a0 + 1) & ~1;
    if (!ok || cnt > CAP || (long long)a0 + cntv > nnz || b == a) {
      base[s] = -1;
      return;
    }
    base[s] = a0;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&full[s], (unsigned)cntv * 8u + (unsigned)cnt * 2u);
    if (use_hint) {
      const unsigned long long pl = (long long)a0 + cntv <= pin ? pol_keep : pol;
      bulk_g2s_hint(vbuf + (size_t)s * CAP, val + a0, (unsigned)cntv * 8u, &full[s], pl);
      bulk_g2s_hint(dbuf + (size_t)s * CAP, col16 + a0, (unsigned)cnt * 2u, &full[s], pl);
    } else {
      bulk_g2s(vbuf + (size_t)s * CAP, val + a0, (unsigned)cntv * 8u, &full[s]);
      bulk_g2s(dbuf + (size_t)s * CAP, col16 + a0, (unsigned)cnt * 2u, &full[s]);
    }
  };
  int na = 0, nb = 0, nok = 0;
  if (tid == 0) {
    for (int k = 0; k < STAGES - 1; ++k) {
      bounds(k, na, nb, nok);
      stage_tile(k, na, nb, nok);
    }
    bounds(STAGES - 1, na, nb, nok);
  }
  double dot = 0.0;
  unsigned phase_bits = 0;
  pdl_wait();  // everything above touched only the matrix; x, y, rvec may come from the previous kernel
  if (stop) {  // sticky stop flag: drain what was staged, then leave
    __shared__ int stop_sh;
    if (tid == 0) stop_sh = *(volatile const int*)stop;
    __syncthreads();
    if (stop_sh) {
      for (int k = 0; k < STAGES - 1; ++k)
        if (blockIdx.x + (long long)k * gridDim.x < ntiles && base[k % STAGES] >= 0) mbar_wait(&full[k % STAGES], 0u);
      return 0.0;
    }
  }
  for (long long k = 0;; ++k) {
    const long long t = blockIdx.x + k * gridDim.x;
    if (t >= ntiles) break;
    const int s = (int)(k % STAGES);
    if (tid == 0) {
      stage_tile(k + STAGES - 1, na, nb, nok);
      bounds(k + STAGES, na, nb, nok);
    }
    const long long r = t * R + tid;
    int ra = 0, rb = 0;
    double x_own = 0.0, y_prev = 0.0, r_own = 0.0, w_own = 1.0;
    bool keep = true;
    if (r < n) {
      ra = __ldg(crow + r), rb = __ldg(crow + r + 1);
      if (fused) {
        x_own = __ldg(x + r);
        if (mask) keep = mask[r] != 0;
        if (rvec) r_own = rvec[r];
        if (wvec) w_own = wvec[r];
      }
      if (accumulate) y_prev = y[r];
    }
    __syncthreads();  // base[s] written by thread 0 is visible
    const int a0 = base[s];
    double sum = 0.0;
    if (a0 >= 0) {
      mbar_wait(&full[s], (phase_bits >> s) & 1u);
      phase_bits ^= 1u << s;
      const double* vs = vbuf + (size_t)s * CAP - a0;
      const unsigned short* ds = dbuf + (size_t)s * CAP - a0;
      int c = ra < rb ? (int)r - 2 * (int)ds[ra] : 0;  // + ds[ra] = the first column
      int j = ra;
      for (; j + 7 < rb; j += 8) {  // eight independent x gathers in flight
        double xv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) c += ds[j + q], xv[q] = __ldg(x + c);
#pragma unroll
        for (int q = 0; q < 8; ++q) sum += vs[j + q] * xv[q];
      }
      {  // tail: up to seven more, still issued together
        double xv[7];
#pragma unroll
        for (int q = 0; q < 7; ++q) {
          if (j + q < rb) c += ds[j + q];
          xv[q] = (j + q < rb) ? __ldg(x + c) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 7; ++q)
          if (j + q < rb) sum += vs[j + q] * xv[q];
      }
    } else {
      for (int j = ra; j < rb; ++j) sum += ld_stream(val + j) * __ldg(x + ld_stream(col + j));
    }
    if (r < n) {
      if (accumulate) sum += y_prev;
      if (fused) {
        if (!keep) sum = 0.0;
        dot += sum * x_own;
        if (extra) extra[0] += sum * (w_own * r_own), extra[1] += sum * (sum * w_own);
      }
      y[r] = sum;
    }
    __syncthreads();  // the stage is drained: thread 0 may refill it in the next iteration
  }
  return dot;
}

// ---- TMA-pipelined block-CSR SpMV, 3x3 blocks (elasticity: 3 dofs per node) ---------------------------------------------------
// The node-level pattern (brow/bcol) with one 72-byte row-major block per entry cuts the index stream 9x against scalar CSR
// (12 -> 8.44 bytes per scalar nonzero) and fetches x[3c..3c+2] once per block instead of once per scalar row, i.e. a third
// of the gathers.  Same pipeline as spmv_tma_rows: persistent CTAs, thread 0 stages the block and column slices of the next
// row tile with cp.async.bulk while the CTA multiplies the current one; LR lanes share a block row, each lane walks its
// blocks (stride 9 doubles between lanes => conflict-free LDS) and the three partial sums are reduced with shuffles.
// Slices start at a multiple of 4 blocks so both copies are 16-byte aligned (4*72 and 4*4 bytes).
constexpr int BSR_CAP = 352;  // blocks per stage: 2 stages x 352 x 76 B = 53.5 KB per CTA, 4 CTAs per SM
constexpr size_t BSR_SMEM = (size_t)TMA_STAGES * BSR_CAP * 76;

template <int LR, bool NC, int THREADS = TMA_THREADS, int STAGES = TMA_STAGES, int CAP = BSR_CAP>
__device__ __forceinline__ double spmv_bsr3_tma_rows(long long nb, long long nnzb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                     const double* __restrict__ bval, const double* __restrict__ x, double* __restrict__ y,
                                                     const unsigned char* __restrict__ mask, bool accumulate, bool fused) {
  constexpr int R = THREADS / LR;
  extern __shared__ __align__(128) unsigned char tma_smem[];
  double* vbuf = reinterpret_cast<double*>(tma_smem);                                // [STAGES][CAP][9]
  int* cbuf = reinterpret_cast<int*>(tma_smem + sizeof(double) * 9 * STAGES * CAP);  // [STAGES][CAP]
  __shared__ unsigned long long full[STAGES];
  __shared__ int base[STAGES];
  const int tid = threadIdx.x, sub = tid % LR, lr = tid / LR;
  const long long ntiles = (nb + R - 1) / R;
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  auto bounds = [&](long long k, int& a, int& b) {
    const long long t = blockIdx.x + k * gridDim.x;
    a = b = 0;
    if (t < ntiles) a = __ldg(brow + t * R), b = __ldg(brow + min(nb, t * R + R));
  };
  auto stage_tile = [&](long long k, int a, int b) {
    if (blockIdx.x + k * gridDim.x >= ntiles) return;
    const int s = (int)(k % STAGES);
    const int a0 = a & ~3, cnt = (b - a0 + 3) & ~3;
    if (cnt > CAP || (long long)a0 + cnt > nnzb || cnt == 0) {
      base[s] = -1;
      return;
    }
    base[s] = a0;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&full[s], (unsigned)cnt * 76u);
    bulk_g2s(vbuf + (size_t)s * CAP * 9, bval + (size_t)a0 * 9, (unsigned)cnt * 72u, &full[s]);
    bulk_g2s(cbuf + (size_t)s * CAP, bcol + a0, (unsigned)cnt * 4u, &full[s]);
  };
  int na = 0, nbnd = 0;
  if (tid == 0) {
    for (int k = 0; k < STAGES - 1; ++k) {
      bounds(k, na, nbnd);
      stage_tile(k, na, nbnd);
    }
    bounds(STAGES - 1, na, nbnd);
  }
  double dot = 0.0;
  unsigned phase_bits = 0;
  for (long long k = 0;; ++k) {
    const long long t = blockIdx.x + k * gridDim.x;
    if (t >= ntiles) break;
    const int s = (int)(k % STAGES);
    if (tid == 0) {
      stage_tile(k + STAGES - 1, na, nbnd);
      bounds(k + STAGES, na, nbnd);
    }
    const long long r = t * R + lr;
    int ra = 0, rb = 0;
    double xo[3] = {0, 0, 0}, yp[3] = {0, 0, 0};
    bool keep[3] = {true, true, true};
    if (r < nb) {
      ra = __ldg(brow + r), rb = __ldg(brow + r + 1);
      if (sub == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          if (fused) {
            xo[i] = ld_x<NC>(x + 3 * r + i);
            if (mask) keep[i] = mask[3 * r + i] != 0;
          }
          if (accumulate) yp[i] = y[3 * r + i];
        }
      }
    }
    __syncthreads();
    const int a0 = base[s];
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    if (a0 >= 0) {
      mbar_wait(&full[s], (phase_bits >> s) & 1u);
      phase_bits ^= 1u << s;
      const double* vs = vbuf + (size_t)s * CAP * 9 - (size_t)a0 * 9;
      const int* cs = cbuf + (size_t)s * CAP - a0;
      int j = ra + sub;
      for (; j + 3 * LR < rb; j += 4 * LR) {  // four blocks = twelve independent x gathers in flight per lane
        double xv[4][3];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double* xp = x + 3ll * cs[j + q * LR];
          xv[q][0] = ld_x<NC>(xp), xv[q][1] = ld_x<NC>(xp + 1), xv[q][2] = ld_x<NC>(xp + 2);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double* b = vs + (size_t)(j + q * LR) * 9;
          s0 += b[0] * xv[q][0] + b[1] * xv[q][1] + b[2] * xv[q][2];
          s1 += b[3] * xv[q][0] + b[4] * xv[q][1] + b[5] * xv[q][2];
          s2 += b[6] * xv[q][0] + b[7] * xv[q][1] + b[8] * xv[q][2];
        }
      }
      {
        double xv[3][3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const bool in = j + q * LR < rb;
          const double* xp = x + 3ll * (in ? cs[j + q * LR] : 0);
          xv[q][0] = in ? ld_x<NC>(xp) : 0.0, xv[q][1] = in ? ld_x<NC>(xp + 1) : 0.0, xv[q][2] = in ? ld_x<NC>(xp + 2) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 3; ++q)
          if (j + q * LR < rb) {
            const double* b = vs + (size_t)(j + q * LR) * 9;
            s0 += b[0] * xv[q][0] + b[1] * xv[q][1] + b[2] * xv[q][2];
            s1 += b[3] * xv[q][0] + b[4] * xv[q][1] + b[5] * xv[q][2];
            s2 += b[6] * xv[q][0] + b[7] * xv[q][1] + b[8] * xv[q][2];
          }
      }
    } else {
      for (int j = ra + sub; j < rb; j += LR) {
        const double* b = bval + (size_t)j * 9;
        const double* xp = x + 3ll * ld_stream(bcol + j);
        const double x0 = ld_x<NC>(xp), x1 = ld_x<NC>(xp + 1), x2 = ld_x<NC>(xp + 2);
        s0 += ld_stream(b) * x0 + ld_stream(b + 1) * x1 + ld_stream(b + 2) * x2;
        s1 += ld_stream(b + 3) * x0 + ld_stream(b + 4) * x1 + ld_stream(b + 5) * x2;
        s2 += ld_stream(b + 6) * x0 + ld_stream(b + 7) * x1 + ld_stream(b + 8) * x2;
      }
    }
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (r < nb && sub == 0) {
      double sv[3] = {s0, s1, s2};
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (accumulate) sv[i] += yp[i];
        if (fused) {
          if (!keep[i]) sv[i] = 0.0;
          dot += sv[i] * xo[i];
        }
        y[3 * r + i] = sv[i];
      }
    }
    __syncthreads();
  }
  return dot;
}

inline int bsr_pick_lr(long long nb, long long nnzb) {
  const double avg = nb > 0 ? (double)nnzb / (double)nb : 1.0;
  for (int lr = 1; lr <= 32; lr *= 2)
    if ((TMA_THREADS / lr) * avg * 1.15 <= BSR_CAP) return lr;
  return 32;
}

}  // namespace femb
