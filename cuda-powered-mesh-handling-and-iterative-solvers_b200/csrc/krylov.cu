// CSR SpMV and the conjugate-gradient loops of the reference (solver/solver.py:144-229 projected CG,
// :766-812 Jacobi-PCG) on the assembled operator.
//
// One CG iteration = three kernels, captured `check_every` at a time in a CUDA graph:
//   k1  Ap = mask .* (A p), per-CTA partial of p.Ap, last CTA reduces the partials in index order -> pAp, guards, alpha
//   k2  u += alpha p, r -= alpha Ap, partial of r.r (or r.Minv r), last CTA -> rs_new, convergence test, beta, rs_old
//   k3  p = r + beta p            (or Minv r + beta p)
// All scalars stay on the device.  Once the sticky stop flag is set the remaining kernels of the graph are no-ops, so the
// state returned is exactly the state at the reference's `break`.
#include <cstdlib>

#include "spmv_dev.cuh"

namespace femb {

struct CGState {
  double rs_old, rs_new, pAp, alpha, beta;
  int it, stop, status, iterations;
  unsigned int ticket1, ticket2;
  int fin, fin_status;  // merged loop: this iteration ends the solve after the u/r update (converged / bad beta)
};

// Last-CTA-done epilogue of CG step k1: per-CTA partial of p.Ap, then the last CTA to arrive sums the partials in index
// order (deterministic), applies the reference's guards (solver.py:187-198) and publishes alpha.
template <int THREADS>
__device__ __forceinline__ void cg_k1_epilogue_n(double dot, double* __restrict__ partial, CGState* __restrict__ st, double eps, int guards) {
  const double t = block_sum<THREADS>(dot);
  __shared__ bool last;
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = t;
    __threadfence();
    last = atomicAdd(&st->ticket1, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double a = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket1 = 0;
      st->pAp = a;
      if (guards && (fabs(a) < eps || a < 0.0)) {  // solver.py:187-192
        st->stop = 1, st->status = 1, st->iterations = st->it + 1;
      } else {
        const double alpha = st->rs_old / (a + eps);
        st->alpha = alpha;
        if (guards && !isfinite(alpha)) st->stop = 1, st->status = 1, st->iterations = st->it + 1;  // solver.py:196-198
      }
    }
  }
}

__device__ __forceinline__ void cg_k1_epilogue(double dot, double* __restrict__ partial, CGState* __restrict__ st, double eps, int guards) {
  cg_k1_epilogue_n<SPMV_THREADS>(dot, partial, st, eps, guards);
}

// Merged-reduction loop (default for CG without a preconditioner): the SpMV also sums r.Ap and Ap.Ap, so its last CTA knows
// alpha AND  rs_new = rs - 2 alpha r.Ap + alpha^2 Ap.Ap = |r - alpha Ap|^2  and with it the convergence verdict and beta:
// every scalar of the iteration is decided here, and ONE vector kernel (cg_merged_kernel) applies u += alpha p,
// r -= alpha Ap, p = r + beta p in a single pass (7 vector passes instead of 9, 2 kernels instead of 3).  That pass also
// accumulates the true r.r of the new residual, which becomes the `rs` of the next iteration, so the recurrence never runs
// more than one step away from an exactly summed value (relative error ~ eps * rs/rs_new).
template <int THREADS>
__device__ __forceinline__ void cg_k1_epilogue3_n(double dot, double e0, double e1, double* __restrict__ partial, CGState* __restrict__ st,
                                                  double eps, int guards, double tol) {
  const double t0 = block_sum<THREADS>(dot), t1 = block_sum<THREADS>(e0), t2 = block_sum<THREADS>(e1);
  const int G = gridDim.x;
  __shared__ bool last;
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = t0, partial[G + blockIdx.x] = t1, partial[2 * G + blockIdx.x] = t2;
    __threadfence();
    last = atomicAdd(&st->ticket1, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double a = 0.0, b = 0.0, c = 0.0;
    for (int k = threadIdx.x; k < G; k += THREADS)
      a += ((volatile double*)partial)[k], b += ((volatile double*)partial)[G + k], c += ((volatile double*)partial)[2 * G + k];
    a = block_sum<THREADS>(a), b = block_sum<THREADS>(b), c = block_sum<THREADS>(c);
    if (threadIdx.x == 0) {
      st->ticket1 = 0;
      st->pAp = a;
      const double rs = st->rs_old, alpha = rs / (a + eps);
      if (guards && (fabs(a) < eps || a < 0.0 || !isfinite(alpha))) {  // solver.py:187-198: break before any update
        st->stop = 1, st->status = 1, st->iterations = st->it + 1;
      } else {
        double rs_new = rs - 2.0 * alpha * b + alpha * alpha * c;
        if (!(rs_new > 0.0)) rs_new = 0.0;  // cancellation at machine-precision convergence
        const double beta = rs_new / (rs + eps);
        // The recurrence value only feeds beta.  Convergence is decided by cg_merged_kernel on the exactly summed r.r of the
        // updated residual (the reference's test, solver.py:208-212): the estimate carries an absolute error ~ eps_mach * rs
        // and can be <= tol^2 (or clip to 0) one step before the true norm is, e.g. at the finite-termination step of a
        // small system.  A clipped estimate gives beta = 0, i.e. a steepest-descent restart, never a false "converged".
        st->alpha = alpha, st->beta = beta, st->rs_new = rs_new;
        st->fin = 0;
        if (guards && !isfinite(beta)) st->fin = 1, st->fin_status = 1;  // solver.py:216-218
      }
    }
  }
}

// L lanes cooperate on one row.  FUSED adds the row mask, the p.Ap partial and the last-CTA scalar epilogue.
template <int L, bool FUSED>
__global__ void __launch_bounds__(SPMV_THREADS) spmv_kernel(long long n, const int* __restrict__ crow, const int* __restrict__ col,
                                                            const double* __restrict__ val, const double* __restrict__ x,
                                                            double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                            double* __restrict__ partial, CGState* __restrict__ st, double eps, int guards,
                                                            const double* __restrict__ rvec, double tol, const double* __restrict__ wvec) {
  if (st && st->stop) return;
  const bool accumulate = (guards & 2) != 0;  // y += A x (operator given as a sum of matrices)
  guards &= 1;
  double e0 = 0.0, e1 = 0.0;
  const int sub = threadIdx.x % L;
  const long long group = (blockIdx.x * (long long)blockDim.x + threadIdx.x) / L;
  const long long ngroups = ((long long)gridDim.x * blockDim.x) / L;
  double dot = 0.0;
  for (long long r0 = 0; r0 < n; r0 += ngroups) {  // warp-uniform trip count (shuffles below use the full mask)
    const long long r = r0 + group;
    double sum = 0.0;
    if (r < n) {
      const int s = __ldg(crow + r), e = __ldg(crow + r + 1);
      int j = s + sub;
      for (; j + L < e; j += 2 * L) {
        const int c0 = ld_stream(col + j), c1 = ld_stream(col + j + L);
        const double v0 = ld_stream(val + j), v1 = ld_stream(val + j + L);
        sum += v0 * __ldg(x + c0);
        sum += v1 * __ldg(x + c1);
      }
      if (j < e) sum += ld_stream(val + j) * __ldg(x + ld_stream(col + j));
    }
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (r < n && sub == 0) {
      if (accumulate) sum += y[r];
      if (FUSED) {
        if (mask && !mask[r]) sum = 0.0;
        dot += sum * __ldg(x + r);
        if (rvec) {  // merged-reduction sums; wvec = the Jacobi diagonal of PCG (z = wvec .* r)
          const double w = wvec ? wvec[r] : 1.0;
          e0 += sum * (w * rvec[r]), e1 += sum * (sum * w);
        }
      }
      y[r] = sum;
    }
  }
  if (FUSED) {
    if (rvec) cg_k1_epilogue3_n<SPMV_THREADS>(dot, e0, e1, partial, st, eps, guards, tol);
    else cg_k1_epilogue(dot, partial, st, eps, guards);
  }
}

template <int LR, bool FUSED>
__global__ void __launch_bounds__(SPMV_THREADS) spmv_stream_kernel(long long n, const int* __restrict__ crow, const int* __restrict__ col,
                                                                   const double* __restrict__ val, const double* __restrict__ x,
                                                                   double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                                   double* __restrict__ partial, CGState* __restrict__ st, double eps,
                                                                   int guards, const double* __restrict__ rvec, double tol,
                                                                   const double* __restrict__ wvec) {
  if (st && st->stop) return;
  const double dot = spmv_stream_rows<LR, true>(n, crow, col, val, x, y, mask, (guards & 2) != 0, FUSED);
  if (FUSED) cg_k1_epilogue(dot, partial, st, eps, guards & 1);
}

// default SpMV: TMA-pipelined row tiles (spmv_dev.cuh)
template <int LR, bool FUSED>
__global__ void __launch_bounds__(TMA_THREADS) spmv_tma_kernel(long long n, long long nnz, const int* __restrict__ crow, const int* __restrict__ col,
                                                               const double* __restrict__ val, const double* __restrict__ x,
                                                               double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                               double* __restrict__ partial, CGState* __restrict__ st, double eps, int guards,
                                                               const double* __restrict__ rvec, double tol, long long pin,
                                                               const double* __restrict__ wvec) {
  pdl_launch_dependents();
  double extra[2] = {0.0, 0.0};
  const double dot = spmv_tma_rows<LR, true, TMA_THREADS, TMA_STAGES, TMA_CAP, NoHaloWait, PdlWait>(
      n, nnz, crow, col, val, x, y, mask, (guards & 2) != 0, FUSED, 0x7fffffffffffffffll, NoHaloWait(), rvec, rvec ? extra : nullptr, PdlWait(),
      st ? &st->stop : nullptr, pin, wvec);
  if (st && st->stop) return;  // block-uniform: the flag is only written by the previous kernel's last CTA
  if (FUSED) {
    if (rvec) cg_k1_epilogue3_n<TMA_THREADS>(dot, extra[0], extra[1], partial, st, eps, guards & 1, tol);
    else cg_k1_epilogue_n<TMA_THREADS>(dot, partial, st, eps, guards & 1);
  }
}

// same with the 16-bit delta-encoded column stream (LR = 1, merged CG loop): col16 / tile_ok from idx16_encode_kernel
template <bool FUSED>
__global__ void __launch_bounds__(TMA_THREADS) spmv_tma16_kernel(long long n, long long nnz, const int* __restrict__ crow, const int* __restrict__ col,
                                                                 const double* __restrict__ val, const double* __restrict__ x,
                                                                 double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                                 double* __restrict__ partial, CGState* __restrict__ st, double eps, int guards,
                                                                 const double* __restrict__ rvec, double tol, long long pin,
                                                                 const double* __restrict__ wvec, const unsigned short* __restrict__ col16,
                                                                 const unsigned char* __restrict__ tile_ok) {
  pdl_launch_dependents();
  double extra[2] = {0.0, 0.0};
  const double dot = spmv_tma16_rows<TMA16_STAGES, TMA16_CAP>(n, nnz, crow, col, col16, tile_ok, val, x, y, mask, (guards & 2) != 0, FUSED, rvec,
                                                             rvec ? extra : nullptr, st ? &st->stop : nullptr, pin, wvec);
  if (st && st->stop) return;
  if (FUSED) {
    if (rvec) cg_k1_epilogue3_n<TMA_THREADS>(dot, extra[0], extra[1], partial, st, eps, guards & 1, tol);
    else cg_k1_epilogue_n<TMA_THREADS>(dot, partial, st, eps, guards & 1);
  }
}

// 16-bit column index: col16[a] = row - col[a] for the first entry a of a row, col16[j] = col[j] - col[j-1] after it.  One CTA
// per 128-row tile (the tile of spmv_tma16_kernel); tile_ok[t] = 1 when every row of the tile encodes losslessly (first column
// 0..65535 below the row, strictly increasing columns with gaps <= 65535), and *bad counts the tiles that do not.
__global__ void __launch_bounds__(TMA_THREADS) idx16_encode_kernel(long long n, const int* __restrict__ crow, const int* __restrict__ col,
                                                                   unsigned short* __restrict__ col16, unsigned char* __restrict__ tile_ok,
                                                                   int* __restrict__ bad) {
  const long long ntiles = (n + TMA_THREADS - 1) / TMA_THREADS;
  for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const long long r = t * TMA_THREADS + threadIdx.x;
    bool ok = true;
    if (r < n) {
      const int a = __ldg(crow + r), b = __ldg(crow + r + 1);
      long long prev = r;
      for (int j = a; j < b; ++j) {
        const long long c = __ldg(col + j), d = j == a ? prev - c : c - prev;
        ok = ok && d >= (j == a ? 0 : 1) && d <= 65535;
        col16[j] = (unsigned short)d;
        prev = c;
      }
    }
    ok = __syncthreads_and(ok);
    if (threadIdx.x == 0) {
      tile_ok[t] = ok ? 1 : 0;
      if (!ok) atomicAdd(bad, 1);
    }
  }
}

// block-CSR (3x3) variant for 3-dof operators: n = 3 nb scalar rows, crow/col are the node-level pattern, val the blocks
template <int LR, bool FUSED>
__global__ void __launch_bounds__(TMA_THREADS) spmv_bsr3_tma_kernel(long long nb, long long nnzb, const int* __restrict__ brow,
                                                                    const int* __restrict__ bcol, const double* __restrict__ bval,
                                                                    const double* __restrict__ x, double* __restrict__ y,
                                                                    const unsigned char* __restrict__ mask, double* __restrict__ partial,
                                                                    CGState* __restrict__ st, double eps, int guards,
                                                                    const double* __restrict__ rvec, double tol, const double* __restrict__ wvec) {
  if (st && st->stop) return;
  const double dot = spmv_bsr3_tma_rows<LR, true>(nb, nnzb, brow, bcol, bval, x, y, mask, (guards & 2) != 0, FUSED);
  if (FUSED) cg_k1_epilogue_n<TMA_THREADS>(dot, partial, st, eps, guards & 1);
}

// Warp-per-block-row variant (default for 3x3 blocks).  ncu on the 2 M-tet P2 operator showed the TMA row-tile kernels
// (scalar and block) latency-bound at 16 resident warps per SM (long-scoreboard 15 per issue, 32-35 % of DRAM peak): with
// ~28 blocks per row a tile holds only 8 rows, so the x gathers of one tile are all that is in flight between two CTA
// barriers, while the plain lanes-per-row kernel at 64 warps per SM reached 64 %.  Here every warp is independent and lean:
// lanes 0..26 cover three consecutive blocks per step (lane = 9*block + position, fixed for the whole kernel, so no index
// arithmetic in the loop), the 216 bytes of a step are one contiguous coalesced read, every lane keeps ONE accumulator
// (its position's row of the block), the three x gathers of a block land in one sector, and four shuffles finish a row.
// MERGED (the two extra dot products of the merged-reduction loop) is a template parameter: compiled into the plain and the
// classic-fused kernels it costs them 8 registers, i.e. 48 instead of 64 resident warps per SM (measured: 1.30 -> 1.52 ms on
// the 2 M-tet P2 operator).
constexpr int BSRV_THREADS = 256;
template <bool FUSED, int U, bool MERGED>
__global__ void __launch_bounds__(BSRV_THREADS) spmv_bsr3_vec_kernel(long long nb, long long nnzb, const int* __restrict__ brow,
                                                                     const int* __restrict__ bcol, const double* __restrict__ bval,
                                                                     const double* __restrict__ x, double* __restrict__ y,
                                                                     const unsigned char* __restrict__ mask, double* __restrict__ partial,
                                                                     CGState* __restrict__ st, double eps, int guards,
                                                                     const double* __restrict__ rvec, double tol, const double* __restrict__ wvec) {
  if (st && st->stop) return;
  const bool accumulate = (guards & 2) != 0;
  guards &= 1;
  double e0 = 0.0, e1 = 0.0;
  const int lane = threadIdx.x & 31;
  const int boff = lane / 9, pos = lane - 9 * boff, cx = pos % 3;  // lanes 27..31: boff = 3 -> idle
  const bool active = lane < 27;
  const long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  double dot = 0.0;
  const bool owner = lane == 0 || lane == 3 || lane == 6;  // these lanes finish row 3r + lane/3
  for (long long r = gw; r < nb; r += nw) {
    const int a = __ldg(brow + r), e = __ldg(brow + r + 1);
    // the row's own vector entries are requested before the block loop: r and minv stream from DRAM, and loading them after
    // the shuffles put a full memory latency at the end of every row (merged Jacobi-PCG: 2.06 ms instead of 1.46 per iteration)
    double r_own = 0.0, w_own = 1.0;
    if (MERGED && owner) {
      r_own = rvec[3 * r + lane / 3];
      if (wvec) w_own = wvec[3 * r + lane / 3];
    }
    double acc = 0.0;
    if (active) {
      int b = a + boff;
      for (; b + 3 * (U - 1) < e; b += 3 * U) {
        double v[U], xv[U];
#pragma unroll
        for (int q = 0; q < U; ++q) {
          v[q] = ld_stream(bval + (size_t)(b + 3 * q) * 9 + pos);
          xv[q] = __ldg(x + 3ll * ld_stream(bcol + b + 3 * q) + cx);
        }
#pragma unroll
        for (int q = 0; q < U; ++q) acc += v[q] * xv[q];
      }
      for (; b < e; b += 3) acc += ld_stream(bval + (size_t)b * 9 + pos) * __ldg(x + 3ll * ld_stream(bcol + b) + cx);
    }
    // lanes p, p+9, p+18 hold the same position; then positions 3i..3i+2 form row i of the block
    acc += __shfl_down_sync(0xffffffffu, acc, 9) + __shfl_down_sync(0xffffffffu, acc, 18);
    acc += __shfl_down_sync(0xffffffffu, acc, 1) + __shfl_down_sync(0xffffffffu, acc, 2);
    if (lane == 0 || lane == 3 || lane == 6) {
      const long long i = 3 * r + lane / 3;
      double sv = acc;
      if (accumulate) sv += y[i];
      if (FUSED) {
        if (mask && !mask[i]) sv = 0.0;
        dot += sv * __ldg(x + i);
        if (MERGED) e0 += sv * (w_own * r_own), e1 += sv * (sv * w_own);
      }
      y[i] = sv;
    }
  }
  if (FUSED) {
    if (MERGED) cg_k1_epilogue3_n<BSRV_THREADS>(dot, e0, e1, partial, st, eps, guards, tol);
    else cg_k1_epilogue_n<BSRV_THREADS>(dot, partial, st, eps, guards);
  }
}

// CSR values of a 3-dof operator (rows 3i..3i+2 of node i stored one after the other) <-> 3x3 blocks: a permutation inside
// each node's 9*len segment.  One warp per node row.
template <bool TO_BSR>
__global__ void csr_bsr3_permute_kernel(long long nb, const int* __restrict__ brow, const double* __restrict__ in, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long w0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = w0; i < nb; i += nw) {
    const long long a = brow[i];
    const int len = brow[i + 1] - (int)a, row = 3 * len;
    for (int t = lane; t < 9 * len; t += 32) {
      const int al = t / row, rem = t - al * row, slot = rem / 3, be = rem - 3 * slot;
      const long long ci = 9 * a + t, bi = 9 * (a + slot) + 3 * al + be;
      if (TO_BSR) out[bi] = in[ci];
      else out[ci] = in[bi];
    }
  }
}

__global__ void bsr3_jacobi_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol, const double* __restrict__ bval,
                                   const unsigned char* __restrict__ mask, double* __restrict__ minv) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < nb; r += (long long)gridDim.x * blockDim.x) {
    int lo = brow[r], hi = brow[r + 1];
    const int end = hi;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (bcol[mid] < r) lo = mid + 1;
      else hi = mid;
    }
    const bool found = lo < end && bcol[lo] == r;
    for (int i = 0; i < 3; ++i) {
      const double d = found ? bval[(size_t)lo * 9 + 4 * i] : 0.0;
      minv[3 * r + i] = (d != 0.0 && (!mask || mask[3 * r + i])) ? 1.0 / d : 0.0;
    }
  }
}

constexpr int VEC_THREADS = 256;

// k2: u += alpha p ; r -= alpha Ap ; partial r.r or r.(minv r) ; last CTA: convergence / beta / bookkeeping
__global__ void __launch_bounds__(VEC_THREADS) cg_update_kernel(long long n, double* __restrict__ u, double* __restrict__ r,
                                                                const double* __restrict__ p, const double* __restrict__ Ap,
                                                                const double* __restrict__ minv, double* __restrict__ partial,
                                                                CGState* __restrict__ st, double tol, double eps, int guards, int max_iter) {
  if (st->stop) return;
  const double alpha = st->alpha;
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double pi = p[i], ri = r[i] - alpha * Ap[i];
    u[i] += alpha * pi;
    r[i] = ri;
    dot += minv ? ri * (minv[i] * ri) : ri * ri;
  }
  const double t = block_sum<VEC_THREADS>(dot);
  __shared__ bool last;
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = t;
    __threadfence();
    last = atomicAdd(&st->ticket2, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double a = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += VEC_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<VEC_THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket2 = 0;
      st->rs_new = a;
      if (sqrt(a) < tol) {  // solver.py:210-212 / :804-806
        st->stop = 1, st->status = 0, st->iterations = st->it + 1;
      } else {
        const double beta = a / (st->rs_old + eps);
        st->beta = beta;
        if (guards && !isfinite(beta)) {  // solver.py:216-218
          st->stop = 1, st->status = 1, st->iterations = st->it + 1;
        } else {
          st->rs_old = a;
          st->it += 1;
          if (st->it >= max_iter) st->stop = 2, st->status = 2, st->iterations = max_iter;
        }
      }
    }
  }
}

// k3: p = z + beta p with z = r or minv*r.  stop==1 means the reference broke out before this update; stop==2 (max_iter) did not.
__global__ void __launch_bounds__(VEC_THREADS) cg_direction_kernel(long long n, const double* __restrict__ r, double* __restrict__ p,
                                                                   const double* __restrict__ minv, const CGState* __restrict__ st) {
  if (st->stop == 1) return;
  const double beta = st->beta;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double z = minv ? minv[i] * r[i] : r[i];
    p[i] = z + beta * p[i];
  }
}

// merged loop, second kernel: all scalars were fixed by the SpMV's last CTA (cg_k1_epilogue3_n)
__global__ void __launch_bounds__(VEC_THREADS) cg_merged_kernel(long long n, double* __restrict__ u, double* __restrict__ r, double* __restrict__ p,
                                                                const double* __restrict__ Ap, const double* __restrict__ minv,
                                                                double* __restrict__ partial, CGState* __restrict__ st, int max_iter, double tol) {
  // minv != nullptr: Jacobi-PCG (solver.py:766-812): z = minv .* r, the exact sum is r.z, p = z + beta p
  pdl_launch_dependents();
  pdl_wait();
  if (st->stop) return;
  const double alpha = st->alpha, beta = st->beta;
  const bool move_p = st->fin == 0;
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double pi = p[i], ri = r[i] - alpha * Ap[i];
    const double zi = minv ? minv[i] * ri : ri;
    u[i] += alpha * pi;
    r[i] = ri;
    dot += ri * zi;
    if (move_p) p[i] = zi + beta * pi;
  }
  const double t = block_sum<VEC_THREADS>(dot);
  __shared__ bool last;
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = t;
    __threadfence();
    last = atomicAdd(&st->ticket2, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double a = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += VEC_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<VEC_THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket2 = 0;
      st->rs_new = a;  // the reported residual is the exactly summed one
      if (sqrt(a) < tol) {  // solver.py:210-212: break after the u / r update (p is not part of the result)
        st->stop = 1, st->status = 0, st->iterations = st->it + 1;
      } else if (!move_p) {
        st->stop = 1, st->status = st->fin_status, st->iterations = st->it + 1;
      } else {
        st->rs_old = a;  // exactly summed r.r of the new residual: the next recurrence starts from it
        st->it += 1;
        if (st->it >= max_iter) st->stop = 2, st->status = 2, st->iterations = max_iter;
      }
    }
  }
}

// setup: u <- mask.*u ; (after Ap = A u) r = mask.*(F - Ap), p = z, partial r.z -> rs_old
__global__ void cg_mask_kernel(long long n, double* __restrict__ u, const unsigned char* __restrict__ mask) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!mask[i]) u[i] = 0.0;
}

__global__ void __launch_bounds__(VEC_THREADS) cg_init_kernel(long long n, const double* __restrict__ F, const double* __restrict__ Au,
                                                              const unsigned char* __restrict__ mask, const double* __restrict__ minv,
                                                              double* __restrict__ r, double* __restrict__ p, double* __restrict__ partial) {
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double ri = F[i] - Au[i];
    if (mask && !mask[i]) ri = 0.0;
    const double z = minv ? minv[i] * ri : ri;
    r[i] = ri;
    p[i] = z;
    dot += ri * z;
  }
  const double t = block_sum<VEC_THREADS>(dot);
  if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

__global__ void __launch_bounds__(VEC_THREADS) cg_init_finish(int nparts, const double* __restrict__ partial, CGState* __restrict__ st,
                                                              int max_iter) {
  double a = 0.0;
  for (int k = threadIdx.x; k < nparts; k += VEC_THREADS) a += partial[k];
  a = block_sum<VEC_THREADS>(a);
  if (threadIdx.x == 0) {
    CGState s;
    memset(&s, 0, sizeof(s));
    s.rs_old = a;
    s.rs_new = a;
    if (max_iter <= 0) s.stop = 2, s.status = 2;
    *st = s;
  }
}

__global__ void jacobi_kernel(long long n, const int* __restrict__ crow, const int* __restrict__ col, const double* __restrict__ val,
                              const unsigned char* __restrict__ mask, double* __restrict__ minv) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x) {
    double d = 0.0;
    int lo = crow[r], hi = crow[r + 1];
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (col[mid] < r) lo = mid + 1;
      else hi = mid;
    }
    if (lo < crow[r + 1] && col[lo] == r) d = val[lo];
    minv[r] = (d != 0.0 && (!mask || mask[r])) ? 1.0 / d : 0.0;
  }
}

// Kernel selection, encoded in one int: 100+LR = TMA-pipelined (default), LR = LDG-streaming (FEMB_SPMV_STREAM=1),
// -L = legacy L-lanes-per-row vector kernel (FEMB_SPMV_VECTOR=1).  The env switches exist for A/B profiling.
static int pick_lanes(long long n, long long nnz, int block = 1) {
  static const bool bsr_tma = getenv("FEMB_BSR_TMA") != nullptr;
  static const int bsrv_unroll = getenv("FEMB_BSRV_UNROLL") ? atoi(getenv("FEMB_BSRV_UNROLL")) : 4;
  if (block == 3) return bsr_tma ? 200 + bsr_pick_lr(n / 3, nnz) : (bsrv_unroll == 2 ? 301 : 300);
  const double avg = n > 0 ? (double)nnz / (double)n : 1.0;
  static const bool force_vector = getenv("FEMB_SPMV_VECTOR") != nullptr, force_stream = getenv("FEMB_SPMV_STREAM") != nullptr;
  if (force_vector) return -(avg <= 3 ? 2 : avg <= 6 ? 4 : avg <= 24 ? 8 : avg <= 48 ? 16 : 32);
  // long rows (P2 / quadratic-hex elasticity kept in scalar CSR, 6-dof shell operators): a warp per row keeps 64 warps per
  // SM busy on independent gathers and measured 0.64 of the HBM peak on the 2 M-tet P2 operator against 0.47 for row tiles
  static const bool force_tma = getenv("FEMB_SPMV_TMA") != nullptr;
  if (!force_stream && !force_tma && avg >= 64.0) return -32;
  if (!force_stream) return 100 + tma_pick_lr(n, nnz);
  for (int lr = 1; lr <= 32; lr *= 2)
    if ((SPMV_THREADS / lr) * avg * 1.25 <= STREAM_CAP) return lr;
  return 32;
}

static thread_local long long nnz_hint = 0;  // set by the callers right before launch_spmv (the TMA kernel clamps its copies to nnz)
static thread_local bool pdl_hint = false;   // launch the next TMA SpMV with the programmatic-serialization attribute (graph loop only)
static thread_local long long pin_hint = 0;  // leading nonzeros staged evict_last (spmv_pin_entries), 0 outside solves
// set: lanes == 101 launches spmv_tma16_kernel on this encoded index (cg_solve_impl only)
static thread_local const unsigned short* col16_hint = nullptr;
static thread_local const unsigned char* tile_ok_hint = nullptr;

template <bool FUSED>
static void launch_spmv(int lanes, int grid, cudaStream_t s, long long n, const int* crow, const int* col, const double* val, const double* x,
                        double* y, const unsigned char* mask, double* partial, CGState* st, double eps, int guards,
                        const double* rvec = nullptr, double tol = 0.0, const double* wvec = nullptr) {
#define FEMB_SPMV_ARGS n, crow, col, val, x, y, mask, partial, st, eps, guards, rvec, tol, wvec
#define FEMB_TMA(LRV)                                                                                                              \
  {                                                                                                                                \
    cudaFuncSetAttribute(spmv_tma_kernel<LRV, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TMA_SMEM);                 \
    launch_pdl(spmv_tma_kernel<LRV, FUSED>, grid, TMA_THREADS, TMA_SMEM, s, pdl_hint, n, nnz_hint, crow, col, val, x, y, mask, partial, st, eps, \
               guards, rvec, tol, pin_hint, wvec);                                                                               \
  }
#define FEMB_BSR(LRV)                                                                                                              \
  {                                                                                                                                \
    cudaFuncSetAttribute(spmv_bsr3_tma_kernel<LRV, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BSR_SMEM);            \
    spmv_bsr3_tma_kernel<LRV, FUSED><<<grid, TMA_THREADS, BSR_SMEM, s>>>(n / 3, nnz_hint, crow, col, val, x, y, mask, partial, st, eps, guards, rvec, tol, wvec); \
  }
  switch (lanes) {
#define FEMB_BSRV(UV)                                                                                                              \
  {                                                                                                                                \
    if (FUSED && rvec)                                                                                                             \
      spmv_bsr3_vec_kernel<FUSED, UV, FUSED><<<grid, BSRV_THREADS, 0, s>>>(n / 3, nnz_hint, crow, col, val, x, y, mask, partial, st, eps, guards, rvec, tol, wvec); \
    else                                                                                                                           \
      spmv_bsr3_vec_kernel<FUSED, UV, false><<<grid, BSRV_THREADS, 0, s>>>(n / 3, nnz_hint, crow, col, val, x, y, mask, partial, st, eps, guards, rvec, tol, wvec); \
  }
    case 300: FEMB_BSRV(4) break;
    case 301: FEMB_BSRV(2) break;
    case 201: FEMB_BSR(1) break;
    case 202: FEMB_BSR(2) break;
    case 204: FEMB_BSR(4) break;
    case 208: FEMB_BSR(8) break;
    case 216: FEMB_BSR(16) break;
    case 232: FEMB_BSR(32) break;
    case 101:
      if (col16_hint) {
        cudaFuncSetAttribute(spmv_tma16_kernel<FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TMA16_SMEM);
        launch_pdl(spmv_tma16_kernel<FUSED>, grid, TMA_THREADS, TMA16_SMEM, s, pdl_hint, n, nnz_hint, crow, col, val, x, y, mask, partial, st,
                   eps, guards, rvec, tol, pin_hint, wvec, col16_hint, tile_ok_hint);
      } else {
        FEMB_TMA(1)
      }
      break;
    case 102: FEMB_TMA(2) break;
    case 104: FEMB_TMA(4) break;
    case 108: FEMB_TMA(8) break;
    case 116: FEMB_TMA(16) break;
    case 132: FEMB_TMA(32) break;
    case 1: spmv_stream_kernel<1, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case 2: spmv_stream_kernel<2, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case 4: spmv_stream_kernel<4, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case 8: spmv_stream_kernel<8, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case 16: spmv_stream_kernel<16, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case 32: spmv_stream_kernel<32, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case -2: spmv_kernel<2, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case -4: spmv_kernel<4, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case -8: spmv_kernel<8, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    case -16: spmv_kernel<16, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
    default: spmv_kernel<32, FUSED><<<grid, SPMV_THREADS, 0, s>>>(FEMB_SPMV_ARGS); break;
  }
#undef FEMB_TMA
#undef FEMB_BSR
#undef FEMB_BSRV
#undef FEMB_SPMV_ARGS
}

static int spmv_grid(long long n, int lanes, bool merged = false) {
  if (lanes == 300 || lanes == 301) {  // warp per block row, persistent: every CTA that fits on the device
    static int fit[2][2] = {{0, 0}, {0, 0}};  // [U = 4 / 2][classic (also bounds the plain kernel) / merged]
    if (!fit[0][0]) {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit[0][0], spmv_bsr3_vec_kernel<true, 4, false>, BSRV_THREADS, 0);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit[1][0], spmv_bsr3_vec_kernel<true, 2, false>, BSRV_THREADS, 0);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit[0][1], spmv_bsr3_vec_kernel<true, 4, true>, BSRV_THREADS, 0);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit[1][1], spmv_bsr3_vec_kernel<true, 2, true>, BSRV_THREADS, 0);
      for (auto& f : fit)
        for (int& v : f)
          if (v < 1) v = 1;
    }
    const int per_sm = getenv("FEMB_BSRV_CTAS") ? atoi(getenv("FEMB_BSRV_CTAS")) : fit[lanes - 300][merged ? 1 : 0];
    const long long ctas = (n / 3 + BSRV_THREADS / 32 - 1) / (BSRV_THREADS / 32);
    return (int)std::max<long long>(1, std::min<long long>(ctas, (long long)SMS * per_sm));
  }
  if (lanes >= 200) return tma_grid(n / 3, lanes - 200);
  if (lanes >= 100) return tma_grid(n, lanes - 100);  // persistent: TMA_CTAS_PER_SM CTAs per SM
  const long long rows_per_block = SPMV_THREADS / (lanes < 0 ? -lanes : lanes);
  const long long tiles = std::max<long long>(1, (n + rows_per_block - 1) / rows_per_block);
  if (lanes < 0) return (int)std::min<long long>(tiles, (long long)SMS * 8);  // legacy vector kernel: persistent grid
  // stream kernel: equal share of row tiles over at most 32 CTAs per SM (measured: larger grids lose on the fused tail)
  const long long max_ctas = SMS * 32;
  const long long per = (tiles + max_ctas - 1) / max_ctas;
  return (int)((tiles + per - 1) / per);
}

}  // namespace femb

using namespace femb;

extern "C" int femb_spmv(int64_t n, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val, const double* x, double* y,
                         femb_stream stream) {
  FEMB_CHECK_ARG(n >= 0, "n >= 0");
  if (n == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  spmv_apply_env_once();
  const int lanes = pick_lanes(n, nnz);
  nnz_hint = nnz;
  launch_spmv<false>(lanes, spmv_grid(n, lanes), s, n, crow, col, val, x, y, nullptr, nullptr, nullptr, 0.0, 0);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_csr_jacobi(int64_t n, const int32_t* crow, const int32_t* col, const double* val, const uint8_t* mask, double* minv,
                               femb_stream stream) {
  if (n == 0) return FEMB_OK;
  jacobi_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(n, crow, col, val, mask, minv);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

struct CsrRef {
  long long nnz;  // scalar nonzeros, or 3x3 blocks when block == 3
  const int *crow, *col;
  const double* val;
  int block = 1;
};

static int cg_solve_impl(int64_t n, int nmat, const CsrRef* mats, const double* F, const uint8_t* mask, const double* minv, double* u,
                         double* work, double tol, int max_iter, double eps, int check_every, femb_cg_result* result_host,
                         femb_stream stream) {
  FEMB_CHECK_ARG(n > 0 && nmat >= 1 && nmat <= 8 && F && u && work && result_host, "null pointer / n <= 0 / nmat not in 1..8");
  if (check_every < 1) check_every = 16;
  spmv_apply_env_once();
  SolveCtx* ctx = solve_ctx(as_stream(stream));  // private capture-capable stream of the current device, ordered after the caller's
  if (!ctx) return FEMB_ERR_CUDA;
  cudaStream_t s = ctx->stream;
  const int guards = minv ? 0 : 1;  // the reference's PCG loop carries no guards and no eps (solver.py:795-810)
  if (minv) eps = 0.0;
  double *r = work, *p = work + n, *Ap = work + 2 * n;
  int lanes[8], g1[8], gmax = 1;
  for (int m = 0; m < nmat; ++m) lanes[m] = pick_lanes(n, mats[m].nnz, mats[m].block);
  // merged-reduction loop (2 kernels, 7 vector passes per iteration) for CG and Jacobi-PCG (the preconditioner's diagonal weights
  // the two extra sums) on every SpMV kernel that forms them; the LDG-streaming / block-TMA A/B kernels and FEMB_CG_CLASSIC=1
  // take the three-kernel loop
  static const bool classic_env = getenv("FEMB_CG_CLASSIC") != nullptr;
  const int ll = lanes[nmat - 1];
  // (3x3 block-CSR keeps the three-kernel loop for CG and PCG alike: on the 2 M-tet P2 operator the merged block SpMV measured
  // 1.96 ms per iteration against 1.49 ms (CG) / 1.47 ms (PCG) -- the warp-per-block-row kernel is latency-bound and pays for the
  // two extra streamed vectors; FEMB_BSR_MERGED=1 selects the merged loop for A/B runs)
  static const bool bsr_merged = getenv("FEMB_BSR_MERGED") != nullptr;
  const bool merged = !classic_env && ((ll >= 300 && bsr_merged) || (ll >= 100 && ll < 200) || ll < 0);
  // 16-bit delta-encoded column stream (DESIGN 3.4): the one-matrix merged loop on the LR = 1 TMA kernel, for solves of at
  // least 16 iterations (the encode pass and its readback cost about 1 ms on C4, two and a half SpMVs).  Encoded on every call, so a pattern changed in place
  // between two calls is always honoured; more than 1 % of tiles that do not encode -> the int32 kernel for the whole solve.
  // FEMB_SPMV_IDX32=1 forces the int32 kernel (A/B runs).
  static const bool idx32_env = getenv("FEMB_SPMV_IDX32") != nullptr;
  bool use16 = !idx32_env && merged && nmat == 1 && lanes[0] == 101 && max_iter >= 16;
  const long long ntiles16 = (n + TMA_THREADS - 1) / TMA_THREADS;
  const size_t flags_off = 256, col16_off = flags_off + (((size_t)ntiles16 + 255) & ~(size_t)255);
  if (use16) {
    const size_t need16 = col16_off + 2 * (((size_t)mats[0].nnz + 7) & ~(size_t)7);  // padded: the last tile's copy stays in bounds
    if (ctx->idx16_bytes < need16) {
      if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec), ctx->graph_exec = nullptr, ctx->graph_key_bytes = 0;
      FEMB_CUDA(cudaStreamSynchronize(s));
      if (ctx->idx16) cudaFree(ctx->idx16);
      ctx->idx16 = nullptr, ctx->idx16_bytes = 0;
      if (cudaMalloc(&ctx->idx16, need16) == cudaSuccess) ctx->idx16_bytes = need16;
      else ctx->idx16 = nullptr, use16 = false, cudaGetLastError();  // out of memory: the int32 stream needs no extra bytes
    }
  }
  if (use16) {
    unsigned char* base16 = static_cast<unsigned char*>(ctx->idx16);
    static_assert(2 * sizeof(CGState) + sizeof(int) <= 512 && 512 + sizeof(int) <= SOLVE_PINNED_BYTES, "pinned status buffer");
    int* bad_host = reinterpret_cast<int*>(static_cast<unsigned char*>(ctx->pinned) + 512);
    FEMB_CUDA(cudaMemsetAsync(base16, 0, sizeof(int), s));
    idx16_encode_kernel<<<(int)std::min<long long>(ntiles16, (long long)SMS * 16), TMA_THREADS, 0, s>>>(
        n, mats[0].crow, mats[0].col, reinterpret_cast<unsigned short*>(base16 + col16_off), base16 + flags_off, reinterpret_cast<int*>(base16));
    FEMB_LAUNCH_CHECK();
    FEMB_CUDA(cudaMemcpyAsync(bad_host, base16, sizeof(int), cudaMemcpyDeviceToHost, s));
    FEMB_CUDA(cudaStreamSynchronize(s));
    use16 = (long long)*bad_host * 100 <= ntiles16;
  }
  const unsigned short* col16 = use16 ? reinterpret_cast<const unsigned short*>(static_cast<unsigned char*>(ctx->idx16) + col16_off) : nullptr;
  const unsigned char* tile_ok = use16 ? static_cast<unsigned char*>(ctx->idx16) + flags_off : nullptr;
  for (int m = 0; m < nmat; ++m) {
    g1[m] = spmv_grid(n, lanes[m], merged && m == nmat - 1);  // one grid per matrix: setup (plain) and loop (fused) launches share it
    if (use16) g1[m] = tma16_grid(n);
    gmax = std::max(gmax, g1[m]);
  }
  const int g2 = grid_for(n, VEC_THREADS, 8);
  static const int vec_waves = getenv("FEMB_VEC_WAVES") ? atoi(getenv("FEMB_VEC_WAVES")) : 8;
  const int g2v = grid_for(n, VEC_THREADS, vec_waves);  // merged vector kernel (A/B: room for the next SpMV's early CTAs)
  // scalars + per-CTA partials: persistent per (thread, device), so their addresses survive from one solve to the next (graph cache)
  const size_t need = 256 + sizeof(double) * (size_t)std::max(3 * gmax, g2);
  if (ctx->dev_scratch_bytes < need) {
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec), ctx->graph_exec = nullptr, ctx->graph_key_bytes = 0;
    FEMB_CUDA(cudaStreamSynchronize(s));
    if (ctx->dev_scratch) cudaFree(ctx->dev_scratch);
    ctx->dev_scratch = nullptr, ctx->dev_scratch_bytes = 0;
    FEMB_CUDA(cudaMalloc(&ctx->dev_scratch, need + need / 2));
    ctx->dev_scratch_bytes = need + need / 2;
  }
  static_assert(sizeof(CGState) <= 256, "state slot");
  CGState* st = static_cast<CGState*>(ctx->dev_scratch);
  double* partial = reinterpret_cast<double*>(static_cast<unsigned char*>(ctx->dev_scratch) + 256);
  // ---- setup (solver.py:163-181)
  if (mask) cg_mask_kernel<<<g2, VEC_THREADS, 0, s>>>(n, u, mask);
  col16_hint = col16, tile_ok_hint = tile_ok;
  for (int m = 0; m < nmat; ++m)
    nnz_hint = mats[m].nnz, launch_spmv<false>(lanes[m], g1[m], s, n, mats[m].crow, mats[m].col, mats[m].val, u, Ap, nullptr, nullptr, nullptr, 0.0, m ? 2 : 0);
  col16_hint = nullptr, tile_ok_hint = nullptr;
  cg_init_kernel<<<g2, VEC_THREADS, 0, s>>>(n, F, Ap, mask, minv, r, p, partial);
  cg_init_finish<<<1, VEC_THREADS, 0, s>>>(g2, partial, st, max_iter);
  FEMB_LAUNCH_CHECK();
  // ---- `check_every` iterations as one graph: re-used when every value baked into it is unchanged
  struct GraphKey {
    long long n;
    int nmat, check_every, max_iter, guards, merged, pdl, lanes[8], g1[8], g2, g2v;
    long long nnz[8];
    const void *crow[8], *col[8], *val[8];
    int block[8];
    const void *mask, *minv, *u, *work, *st, *partial;
    double tol, eps;
    long long pin;
    const void* col16;
  } key;
  memset(&key, 0, sizeof(key));
  static_assert(sizeof(GraphKey) <= sizeof(ctx->graph_key), "graph key buffer");
  key.n = n, key.nmat = nmat, key.check_every = check_every, key.max_iter = max_iter, key.guards = guards, key.merged = merged ? 1 : 0;
  key.pdl = pdl_mode(), key.g2 = g2, key.g2v = g2v, key.mask = mask, key.minv = minv, key.u = u, key.work = work, key.st = st, key.partial = partial;
  key.tol = tol, key.eps = eps, key.pin = spmv_pin_entries(mats[nmat - 1].nnz), key.col16 = col16;
  for (int m = 0; m < nmat; ++m) {
    key.lanes[m] = lanes[m], key.g1[m] = g1[m];
    key.nnz[m] = mats[m].nnz, key.crow[m] = mats[m].crow, key.col[m] = mats[m].col, key.val[m] = mats[m].val, key.block[m] = mats[m].block;
  }
  static const bool no_cache = getenv("FEMB_NO_GRAPH_CACHE") != nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  if (!no_cache && ctx->graph_exec && ctx->graph_key_bytes == sizeof(key) && memcmp(ctx->graph_key, &key, sizeof(key)) == 0) exec = ctx->graph_exec;
  if (!exec) {
  FEMB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  for (int k = 0; k < check_every; ++k) {
    for (int m = 0; m + 1 < nmat; ++m)
      nnz_hint = mats[m].nnz, launch_spmv<false>(lanes[m], g1[m], s, n, mats[m].crow, mats[m].col, mats[m].val, p, Ap, nullptr, nullptr, st, 0.0, m ? 2 : 0);
    const int last = nmat - 1;
    nnz_hint = mats[last].nnz;
    if (merged) {
      // PDL pair: only when the loop is exactly [TMA SpMV, merged vector kernel] (one matrix); the first SpMV of the graph
      // depends on the previous graph launch the ordinary way
      const bool pdl = pdl_enabled() && nmat == 1 && lanes[last] >= 100 && lanes[last] < 200;
      pdl_hint = pdl && k > 0 && (pdl_mode() & 2);
      pin_hint = pdl ? spmv_pin_entries(mats[last].nnz) : 0;
      col16_hint = col16, tile_ok_hint = tile_ok;
      launch_spmv<true>(lanes[last], g1[last], s, n, mats[last].crow, mats[last].col, mats[last].val, p, Ap, mask, partial, st, eps,
                        guards | (last ? 2 : 0), r, tol, minv);
      pdl_hint = false, pin_hint = 0, col16_hint = nullptr, tile_ok_hint = nullptr;
      launch_pdl(cg_merged_kernel, g2v, VEC_THREADS, 0, s, pdl && (pdl_mode() & 1), n, u, r, p, Ap, minv, partial, st, max_iter, tol);
    } else {
      launch_spmv<true>(lanes[last], g1[last], s, n, mats[last].crow, mats[last].col, mats[last].val, p, Ap, mask, partial, st, eps,
                        guards | (last ? 2 : 0));
      cg_update_kernel<<<g2, VEC_THREADS, 0, s>>>(n, u, r, p, Ap, minv, partial, st, tol, eps, guards, max_iter);
      cg_direction_kernel<<<g2, VEC_THREADS, 0, s>>>(n, r, p, minv, st);
    }
  }
  cudaError_t ce = cudaStreamEndCapture(s, &graph);
  if (ce != cudaSuccess) {
    set_error(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
    return FEMB_ERR_CUDA;
  }
  FEMB_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  cudaGraphDestroy(graph);
  FEMB_CUDA(cudaGraphUpload(exec, s));  // the first launch must not pay for the upload inside the loop
  if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
  ctx->graph_exec = exec, ctx->graph_key_bytes = sizeof(key);
  memcpy(ctx->graph_key, &key, sizeof(key));
  }
  // Host polling is pipelined one graph deep: graph l+1 is already queued while the stop flag of graph l travels back
  // (kernels after the stop are no-ops), so the GPU never idles on the host round trip.
  static_assert(2 * sizeof(CGState) <= SOLVE_PINNED_BYTES, "pinned status buffer");
  CGState* hst = static_cast<CGState*>(ctx->pinned);  // [2] pinned
  cudaEvent_t* ev = ctx->poll_ev;
  cudaEvent_t* tev = ctx->time_ev;
  int rc = FEMB_OK;
  const int launches = (max_iter + check_every - 1) / check_every;
  hst[0].stop = hst[1].stop = 0;
  bool stopped = false;
  cudaEventRecord(tev[0], s);
  for (int l = 0; l < launches && !stopped; ++l) {
    if (cudaGraphLaunch(exec, s) != cudaSuccess || cudaMemcpyAsync(&hst[l & 1], st, sizeof(CGState), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaEventRecord(ev[l & 1], s) != cudaSuccess) {
      set_error(std::string("CG graph launch: ") + cudaGetErrorString(cudaGetLastError()));
      rc = FEMB_ERR_CUDA;
      break;
    }
    if (l >= 1) {
      cudaEventSynchronize(ev[(l - 1) & 1]);
      stopped = hst[(l - 1) & 1].stop != 0;
    }
  }
  cudaEventRecord(tev[1], s);
  CGState* fin = &hst[0];
  if (rc == FEMB_OK) {
    if (cudaMemcpyAsync(fin, st, sizeof(CGState), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
      set_error(std::string("CG final state: ") + cudaGetErrorString(cudaGetLastError()));
      rc = FEMB_ERR_CUDA;
    }
  }
  float ms = 0.f;
  if (rc == FEMB_OK) cudaEventElapsedTime(&ms, tev[0], tev[1]);
  if (rc != FEMB_OK) {  // a failed launch may have left the graph in an undefined state: drop it
    cudaGraphExecDestroy(ctx->graph_exec);
    ctx->graph_exec = nullptr, ctx->graph_key_bytes = 0;
    return rc;
  }
  result_host->iterations = fin->stop ? fin->iterations : max_iter;
  result_host->status = fin->stop ? fin->status : 2;
  result_host->rs = fin->rs_new;
  result_host->loop_ms = ms;
  result_host->index_bytes = use16 ? 2 : 4;
  return FEMB_OK;
}

extern "C" int femb_cg_solve(int64_t n, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val, const double* F,
                             const uint8_t* mask, const double* minv, double* u, double* work, double tol, int max_iter, double eps,
                             int check_every, femb_cg_result* result_host, femb_stream stream) {
  FEMB_CHECK_ARG(crow && col && val, "null CSR pointer");
  const CsrRef m{nnz, crow, col, val, 1};
  return cg_solve_impl(n, 1, &m, F, mask, minv, u, work, tol, max_iter, eps, check_every, result_host, stream);
}

extern "C" int femb_spmv_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* bval, const double* x,
                              double* y, femb_stream stream) {
  FEMB_CHECK_ARG(nb >= 0 && nnzb >= 0, "nb >= 0, nnzb >= 0");
  if (nb == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  const int lanes = pick_lanes(3 * nb, nnzb, 3);
  nnz_hint = nnzb;
  launch_spmv<false>(lanes, spmv_grid(3 * nb, lanes), s, 3 * nb, brow, bcol, bval, x, y, nullptr, nullptr, nullptr, 0.0, 0);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_cg_solve_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* bval, const double* F,
                                  const uint8_t* mask, const double* minv, double* u, double* work, double tol, int max_iter, double eps,
                                  int check_every, femb_cg_result* result_host, femb_stream stream) {
  FEMB_CHECK_ARG(brow && bcol && bval, "null BSR pointer");
  const CsrRef m{nnzb, brow, bcol, bval, 3};
  return cg_solve_impl(3 * nb, 1, &m, F, mask, minv, u, work, tol, max_iter, eps, check_every, result_host, stream);
}

extern "C" int femb_csr_bsr3_convert(int to_bsr, int64_t nb, const int32_t* brow, const double* in, double* out, femb_stream stream) {
  FEMB_CHECK_ARG(nb >= 0 && brow && in && out && in != out, "nb >= 0, non-null distinct buffers");
  if (nb == 0) return FEMB_OK;
  const int grid = grid_for(nb * 32, 256, 32);
  if (to_bsr) csr_bsr3_permute_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(nb, brow, in, out);
  else csr_bsr3_permute_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(nb, brow, in, out);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_bsr3_jacobi(int64_t nb, const int32_t* brow, const int32_t* bcol, const double* bval, const uint8_t* mask, double* minv,
                                femb_stream stream) {
  if (nb == 0) return FEMB_OK;
  bsr3_jacobi_kernel<<<grid_for(nb, 256), 256, 0, as_stream(stream)>>>(nb, brow, bcol, bval, mask, minv);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_cg_solve_multi(int64_t n, int nmat, const int64_t* nnz_host, const int32_t* const* crow_host,
                                   const int32_t* const* col_host, const double* const* val_host, const double* F, const uint8_t* mask,
                                   const double* minv, double* u, double* work, double tol, int max_iter, double eps, int check_every,
                                   femb_cg_result* result_host, femb_stream stream) {
  FEMB_CHECK_ARG(nmat >= 1 && nmat <= 8 && nnz_host && crow_host && col_host && val_host, "nmat in 1..8, non-null arrays");
  CsrRef m[8];
  for (int k = 0; k < nmat; ++k) m[k] = CsrRef{nnz_host[k], crow_host[k], col_host[k], val_host[k], 1};
  return cg_solve_impl(n, nmat, m, F, mask, minv, u, work, tol, max_iter, eps, check_every, result_host, stream);
}

// ---------------------------------------------------------------------------------------------------------------------
// conjugate_gradient_solver_Ku (solver.py:1029-1065): CG on an operator the caller supplies as a function.  The reference
// loop carries no guards, no eps and no node fixing; delta_u starts at zero.  The callback runs on the caller's stream between
// the fused vector kernels (it cannot be captured in a graph), scalars stay on the device, and the host reads the stop
// flag every `check_every` iterations (kernels after the stop are no-ops, so the state is the one at the reference's break).
namespace femb {

__global__ void __launch_bounds__(VEC_THREADS) cg_dot_kernel(long long n, const double* __restrict__ p, const double* __restrict__ Ap,
                                                             double* __restrict__ partial, CGState* __restrict__ st) {
  if (st->stop) return;
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dot += p[i] * Ap[i];
  cg_k1_epilogue_n<VEC_THREADS>(dot, partial, st, 0.0, 0);
}

}  // namespace femb

extern "C" int femb_cg_solve_operator(int64_t n, femb_apply_fn apply, void* ctx, const double* R, double* u, double* work, double tol,
                                      int max_iter, int check_every, femb_cg_result* result_host, femb_stream stream) {
  FEMB_CHECK_ARG(n > 0 && apply && R && u && work && result_host, "null pointer / n <= 0");
  if (check_every < 1) check_every = 8;
  cudaStream_t s = as_stream(stream);
  double *r = work, *p = work + n, *Ap = work + 2 * n;
  const int g2 = grid_for(n, VEC_THREADS, 8);
  Scratch scr(s);
  double* partial;
  CGState* st;
  FEMB_CUDA(scr.alloc(&partial, (size_t)g2));
  FEMB_CUDA(scr.alloc(&st, 1));
  cudaEvent_t t0, t1;
  FEMB_CUDA(cudaEventCreate(&t0));
  FEMB_CUDA(cudaEventCreate(&t1));
  int rc = FEMB_OK;
  CGState h;
  memset(&h, 0, sizeof(h));
  auto fail = [&](const char* what) {
    set_error(what);
    rc = FEMB_ERR_ARG;
  };
  // r = R - K(u), p = r, rs_old = r.r   (solver.py:1047-1049)
  if (apply(ctx, u, Ap, stream) != 0) fail("femb_cg_solve_operator: the operator callback failed");
  if (rc == FEMB_OK) {
    cg_init_kernel<<<g2, VEC_THREADS, 0, s>>>(n, R, Ap, nullptr, nullptr, r, p, partial);
    cg_init_finish<<<1, VEC_THREADS, 0, s>>>(g2, partial, st, max_iter);
    cudaEventRecord(t0, s);
    for (int it = 0; it < max_iter && rc == FEMB_OK; ++it) {
      if (apply(ctx, p, Ap, stream) != 0) {
        fail("femb_cg_solve_operator: the operator callback failed");
        break;
      }
      cg_dot_kernel<<<g2, VEC_THREADS, 0, s>>>(n, p, Ap, partial, st);
      cg_update_kernel<<<g2, VEC_THREADS, 0, s>>>(n, u, r, p, Ap, nullptr, partial, st, tol, 0.0, 0, max_iter);
      cg_direction_kernel<<<g2, VEC_THREADS, 0, s>>>(n, r, p, nullptr, st);
      if ((it + 1) % check_every == 0 || it + 1 == max_iter) {
        if (cudaMemcpyAsync(&h, st, sizeof(CGState), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
          set_error(std::string("femb_cg_solve_operator: ") + cudaGetErrorString(cudaGetLastError()));
          rc = FEMB_ERR_CUDA;
          break;
        }
        if (h.stop) break;
      }
    }
    cudaEventRecord(t1, s);
  }
  if (rc == FEMB_OK) {
    if (cudaMemcpyAsync(&h, st, sizeof(CGState), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
      set_error(std::string("femb_cg_solve_operator: ") + cudaGetErrorString(cudaGetLastError()));
      rc = FEMB_ERR_CUDA;
    }
  }
  float ms = 0.f;
  if (rc == FEMB_OK) cudaEventElapsedTime(&ms, t0, t1);
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  if (rc != FEMB_OK) {
    cudaStreamSynchronize(s);  // the scratch below is released stream-ordered; nothing of this solve may still be queued on error paths
    return rc;
  }
  result_host->iterations = h.stop ? h.iterations : max_iter;
  result_host->status = h.stop ? h.status : 2;
  result_host->rs = h.rs_new;
  result_host->loop_ms = ms;
  result_host->index_bytes = 0;  // the operator is the caller's callback
  return FEMB_OK;
}
