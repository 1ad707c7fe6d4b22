// Block kernels of the LOBPCG modal solver (lowest_modes, femb200/modes.py).  Multivectors are ROW-MAJOR and node-interleaved:
// value (dof r, column j) at X[r*ld + j], so the m values of one dof row are contiguous and one 3x3 block column of the SpMM
// gathers three contiguous m-wide rows.  The LOBPCG basis S = [X | W | P] is one [n, 3m] buffer (ld = 3m); K S and M S sit in
// two more.  Four kernels cover everything that touches n-long data:
//   spmm_bsr3        Y_K = K X and, in the same pass, Y_M = M X (K and M share one block pattern): each 3x3 block and its
//                    column index are read once for all m columns
//   mb_gram          G = A^T B (ka, kb <= 48): the whole 3m x 3m Gram of S against K S or M S in one pass; per-CTA partials
//                    summed in index order by a second kernel, so the result is deterministic
//   mb_combine       Y = beta Y + X C (X [n, <=48], C [<=48, <=16] passed by value): new X, P, KX, KP, MX, MP from the Ritz
//                    coefficients without repeating an SpMM
//   lobpcg_residual  R = KX - MX diag(lam), per-column |r|^2 and |x|^2 (deterministic), W = D^-1 R for the active columns
// The 3m x 3m Rayleigh-Ritz problems run on the host.
#include "common.cuh"
#include "spmv_dev.cuh"

namespace femb {

constexpr int MB_MAXM = 16;  // SpMM / residual columns and combine output columns
constexpr int MB_MAXK = 48;  // Gram and combine input columns: the basis [X W P] of 3m columns
constexpr int MB_THREADS = 256;
constexpr int GR_ROWS = 32;  // rows of A and B staged in shared memory per Gram tile

struct MbCoef {
  double c[MB_MAXK * MB_MAXM];  // 6 KB kernel parameter
};
struct MbLam {
  double v[MB_MAXM];
};

__device__ __forceinline__ double ld_stream(const double* p, unsigned long long pol) {
  double v;
  asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ int ld_stream(const int* p, unsigned long long pol) {
  int v;
  asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}

// One warp per block row.  Lane = (slot, c) with c = lane % mp (mp = m rounded up to a power of two) the column and
// slot = lane / mp one of 32/mp blocks handled side by side; lanes of one slot load the same 3x3 block (one uniform-address
// load), lanes of one column load x rows that are contiguous across c.  The matrix stream carries an L2 evict-first hint: it is
// read once per SpMM and should not push the multivectors out of L2.  Slots are summed by a fixed xor tree (deterministic).
template <bool HAS_M>
__global__ void __launch_bounds__(MB_THREADS) spmm_bsr3_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                                const double* __restrict__ kval, const double* __restrict__ mval,
                                                                const unsigned char* __restrict__ mask, int m, int log_mp,
                                                                const double* __restrict__ X, long long ldx, double* __restrict__ YK,
                                                                double* __restrict__ YM, long long ldy) {
  const unsigned long long pol = l2_evict_first_policy();
  const int lane = threadIdx.x & 31;
  const int mp = 1 << log_mp;
  const int c = lane & (mp - 1), slot = lane >> log_mp, nslot = 32 >> log_mp;
  const bool col_ok = c < m;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < nb; row += nwarps) {
    const int b0 = __ldg(brow + row), b1 = __ldg(brow + row + 1);
    double k0 = 0.0, k1 = 0.0, k2 = 0.0, m0 = 0.0, m1 = 0.0, m2 = 0.0;
    for (int b = b0 + slot; b < b1; b += nslot) {
      const long long j = ld_stream(bcol + b, pol);
      double x0 = 0.0, x1 = 0.0, x2 = 0.0;
      if (col_ok) {
        const double* xp = X + 3 * j * ldx + c;
        x0 = xp[0];
        x1 = xp[ldx];
        x2 = xp[2 * ldx];
        if (mask) {
          if (!mask[3 * j]) x0 = 0.0;
          if (!mask[3 * j + 1]) x1 = 0.0;
          if (!mask[3 * j + 2]) x2 = 0.0;
        }
      }
      const double* kb = kval + 9 * (long long)b;
      k0 += ld_stream(kb + 0, pol) * x0 + ld_stream(kb + 1, pol) * x1 + ld_stream(kb + 2, pol) * x2;
      k1 += ld_stream(kb + 3, pol) * x0 + ld_stream(kb + 4, pol) * x1 + ld_stream(kb + 5, pol) * x2;
      k2 += ld_stream(kb + 6, pol) * x0 + ld_stream(kb + 7, pol) * x1 + ld_stream(kb + 8, pol) * x2;
      if (HAS_M) {
        const double* mb = mval + 9 * (long long)b;
        m0 += ld_stream(mb + 0, pol) * x0 + ld_stream(mb + 1, pol) * x1 + ld_stream(mb + 2, pol) * x2;
        m1 += ld_stream(mb + 3, pol) * x0 + ld_stream(mb + 4, pol) * x1 + ld_stream(mb + 5, pol) * x2;
        m2 += ld_stream(mb + 6, pol) * x0 + ld_stream(mb + 7, pol) * x1 + ld_stream(mb + 8, pol) * x2;
      }
    }
    for (int o = mp; o < 32; o <<= 1) {
      k0 += __shfl_xor_sync(0xffffffffu, k0, o);
      k1 += __shfl_xor_sync(0xffffffffu, k1, o);
      k2 += __shfl_xor_sync(0xffffffffu, k2, o);
      if (HAS_M) {
        m0 += __shfl_xor_sync(0xffffffffu, m0, o);
        m1 += __shfl_xor_sync(0xffffffffu, m1, o);
        m2 += __shfl_xor_sync(0xffffffffu, m2, o);
      }
    }
    if (slot == 0 && col_ok) {
      const bool f0 = !mask || mask[3 * row], f1 = !mask || mask[3 * row + 1], f2 = !mask || mask[3 * row + 2];
      double* yk = YK + 3 * row * ldy + c;
      yk[0] = f0 ? k0 : 0.0;
      yk[ldy] = f1 ? k1 : 0.0;
      yk[2 * ldy] = f2 ? k2 : 0.0;
      if (HAS_M) {
        double* ym = YM + 3 * row * ldy + c;
        ym[0] = f0 ? m0 : 0.0;
        ym[ldy] = f1 ? m1 : 0.0;
        ym[2 * ldy] = f2 ? m2 : 0.0;
      }
    }
  }
}

// G = A^T B: a tile of GR_ROWS rows of A and B (zero-padded to 48 columns) is staged in shared memory; thread (bi, bj) of a
// 16 x 16 grid owns the 3 x 3 output block (3bi.., 3bj..), so 256 threads hold all 48 x 48 = 2304 accumulators.
__global__ void __launch_bounds__(MB_THREADS) mb_gram_kernel(long long n, int ka, const double* __restrict__ A, long long lda, int kb,
                                                             const double* __restrict__ B, long long ldb, double* __restrict__ partial) {
  __shared__ double sA[GR_ROWS][MB_MAXK], sB[GR_ROWS][MB_MAXK];
  const int t = threadIdx.x, bi = t >> 4, bj = t & 15;
  double acc[3][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
  for (long long r0 = (long long)blockIdx.x * GR_ROWS; r0 < n; r0 += (long long)gridDim.x * GR_ROWS) {
    const long long rows = n - r0 < GR_ROWS ? n - r0 : GR_ROWS;
    __syncthreads();
    for (int e = t; e < GR_ROWS * MB_MAXK; e += MB_THREADS) {
      const int r = e / MB_MAXK, c = e - r * MB_MAXK;
      sA[r][c] = (r < rows && c < ka) ? A[(r0 + r) * lda + c] : 0.0;
      sB[r][c] = (r < rows && c < kb) ? B[(r0 + r) * ldb + c] : 0.0;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < GR_ROWS; ++r) {
      const double a0 = sA[r][3 * bi], a1 = sA[r][3 * bi + 1], a2 = sA[r][3 * bi + 2];
      const double b0 = sB[r][3 * bj], b1 = sB[r][3 * bj + 1], b2 = sB[r][3 * bj + 2];
      acc[0][0] += a0 * b0; acc[0][1] += a0 * b1; acc[0][2] += a0 * b2;
      acc[1][0] += a1 * b0; acc[1][1] += a1 * b1; acc[1][2] += a1 * b2;
      acc[2][0] += a2 * b0; acc[2][1] += a2 * b1; acc[2][2] += a2 * b2;
    }
  }
  const long long kk = (long long)ka * kb;
#pragma unroll
  for (int p = 0; p < 3; ++p)
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int i = 3 * bi + p, j = 3 * bj + q;
      if (i < ka && j < kb) partial[blockIdx.x * kk + i * kb + j] = acc[p][q];
    }
}

// out[t] = sum over parts p = 0, 1, ... of partial[p*kk + t], in that order
__global__ void __launch_bounds__(MB_THREADS) mb_partial_finish(int nparts, int kk, const double* __restrict__ partial, double* __restrict__ out) {
  const int t = blockIdx.x * MB_THREADS + threadIdx.x;
  if (t >= kk) return;
  double s = 0.0;
  for (int p = 0; p < nparts; ++p) s += partial[(size_t)p * kk + t];
  out[t] = s;
}

// 16 lanes per row, lane j = output column j; the row of X is a broadcast load, C sits in shared memory.
__global__ void __launch_bounds__(MB_THREADS) mb_combine_kernel(long long n, int k, const double* __restrict__ X, long long ldx, int mc,
                                                                MbCoef C, double beta, double* __restrict__ Y, long long ldy) {
  __shared__ double sC[MB_MAXK * MB_MAXM];
  for (int e = threadIdx.x; e < k * mc; e += MB_THREADS) sC[e] = C.c[e];
  __syncthreads();
  const int j = threadIdx.x & 15;
  for (long long r = ((long long)blockIdx.x * MB_THREADS + threadIdx.x) >> 4; r < n; r += ((long long)gridDim.x * MB_THREADS) >> 4) {
    if (j >= mc) continue;
    const double* x = X + r * ldx;
    double s = 0.0;
    for (int i = 0; i < k; ++i) s += x[i] * sC[i * mc + j];
    double* y = Y + r * ldy + j;
    *y = beta != 0.0 ? beta * *y + s : s;
  }
}

// Lane j of a 16-lane row group handles column j; W slot a receives the residual of column active[a] (a shuffle within the
// row group), scaled by dinv (0 on fixed dofs).  Per-CTA sums of |r_j|^2 and |x_j|^2 go to partial[cta][2m] in a fixed order.
__global__ void __launch_bounds__(MB_THREADS) lobpcg_residual_kernel(long long n, int m, const double* __restrict__ X, long long ldx,
                                                                     const double* __restrict__ KX, const double* __restrict__ MX, long long ldk,
                                                                     MbLam lam, const double* __restrict__ dinv, int na,
                                                                     const int* __restrict__ active, double* __restrict__ W, long long ldw,
                                                                     double* __restrict__ partial) {
  __shared__ double red[2][MB_THREADS / 16][16];
  const int lane = threadIdx.x & 31, j = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int src_lane = (lane & 16) | (j < na ? __ldg(active + j) : 0);
  double lj = 0.0;  // unrolled select: indexing the parameter by lane would copy it to local memory
#pragma unroll
  for (int t = 0; t < MB_MAXM; ++t)
    if (t == j) lj = lam.v[t];
  double rr = 0.0, xx = 0.0;
  // rb is uniform across the warp (two rows per warp), so every lane reaches the shuffle
  for (long long rb = (long long)blockIdx.x * (MB_THREADS / 16) + (ty & ~1); rb < n; rb += (long long)gridDim.x * (MB_THREADS / 16)) {
    const long long r = rb + (ty & 1);
    const bool row_ok = r < n;
    double res = 0.0;
    if (row_ok && j < m) {
      const double x = X[r * ldx + j];
      res = KX[r * ldk + j] - lj * MX[r * ldk + j];
      rr += res * res;
      xx += x * x;
    }
    const double mine = __shfl_sync(0xffffffffu, res, src_lane);
    if (row_ok && j < na) W[r * ldw + j] = dinv[r] * mine;
  }
  red[0][ty][j] = rr;
  red[1][ty][j] = xx;
  __syncthreads();
  if (threadIdx.x < 2 * m) {
    const int w = threadIdx.x / m, c = threadIdx.x - w * m;
    double s = 0.0;
    for (int y = 0; y < MB_THREADS / 16; ++y) s += red[w][y][c];
    partial[(size_t)blockIdx.x * (2 * m) + threadIdx.x] = s;
  }
}

// Do the strided views (p, ld_p, kp columns) and (q, ld_q, kq columns) over n rows share an element?  Views with the same leading
// dimension may interleave (disjoint column windows of one buffer); otherwise any overlap of the address ranges counts.
static bool spans_meet(const double* p, long long np, const double* q, long long nq) {  // [p, p+np) and [q, q+nq), in doubles
  return np > 0 && nq > 0 && (uintptr_t)p < (uintptr_t)(q + nq) && (uintptr_t)q < (uintptr_t)(p + np);
}
static bool views_overlap(const double* p, long long ldp, int kp, const double* q, long long ldq, int kq, long long n) {
  if (n == 0 || !spans_meet(p, (n - 1) * ldp + kp, q, (n - 1) * ldq + kq)) return false;
  const uintptr_t p0 = (uintptr_t)p, q0 = (uintptr_t)q;
  if (ldp != ldq || (p0 - q0) % sizeof(double) != 0) return true;
  long long off = ((long long)(q - p)) % ldp;  // column of q within p's rows
  if (off < 0) off += ldp;
  auto hit = [&](long long a) { return a < kp && a + kq > 0; };  // [a, a+kq) meets [0, kp)
  return hit(off) || hit(off - ldp);
}

}  // namespace femb

using namespace femb;

extern "C" int femb_spmm_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* kval, const double* mval,
                              const uint8_t* mask, int m, const double* X, int64_t ldx, double* YK, double* YM, int64_t ldy, femb_stream stream) {
  FEMB_CHECK_ARG(m >= 1 && m <= MB_MAXM, "1 <= m <= 16");
  FEMB_CHECK_ARG(nb >= 0 && nnzb >= 0 && nnzb <= INT32_MAX, "nb >= 0, 0 <= nnzb < 2^31");
  FEMB_CHECK_ARG(brow && bcol && kval && X && YK, "non-null brow, bcol, kval, X, YK");
  FEMB_CHECK_ARG(!mval == !YM, "mval and YM are both given or both NULL");
  FEMB_CHECK_ARG(ldx >= m && ldy >= m, "ldx, ldy >= m");
  const long long n = 3 * nb;
  FEMB_CHECK_ARG(!views_overlap(X, ldx, m, YK, ldy, m, n) && !(YM && views_overlap(X, ldx, m, YM, ldy, m, n)) &&
                     !(YM && views_overlap(YK, ldy, m, YM, ldy, m, n)),
                 "outputs overlap the input or each other");
  if (nb == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  int log_mp = 0;
  while ((1 << log_mp) < m) ++log_mp;
  const int grid = grid_for(nb * 32, MB_THREADS, 32);
  if (mval)
    spmm_bsr3_kernel<true><<<grid, MB_THREADS, 0, s>>>(nb, brow, bcol, kval, mval, mask, m, log_mp, X, ldx, YK, YM, ldy);
  else
    spmm_bsr3_kernel<false><<<grid, MB_THREADS, 0, s>>>(nb, brow, bcol, kval, nullptr, mask, m, log_mp, X, ldx, YK, nullptr, ldy);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_mb_gram(int64_t n, int ka, const double* A, int64_t lda, int kb, const double* B, int64_t ldb, double* G,
                            femb_stream stream) {
  FEMB_CHECK_ARG(ka >= 1 && ka <= MB_MAXK && kb >= 1 && kb <= MB_MAXK, "1 <= ka, kb <= 48");
  FEMB_CHECK_ARG(n >= 0 && A && B && G, "n >= 0, non-null A, B, G");
  FEMB_CHECK_ARG(lda >= ka && ldb >= kb, "lda >= ka, ldb >= kb");
  FEMB_CHECK_ARG(n == 0 || (!spans_meet(G, (long long)ka * kb, A, (n - 1) * lda + ka) && !spans_meet(G, (long long)ka * kb, B, (n - 1) * ldb + kb)),
                 "G overlaps A or B");
  cudaStream_t s = as_stream(stream);
  const int kk = ka * kb;
  if (n == 0) {
    FEMB_CUDA(cudaMemsetAsync(G, 0, sizeof(double) * kk, s));
    return FEMB_OK;
  }
  const int grid = grid_for(n, GR_ROWS, 4);  // depends on n only: the same n sums in the same order on every run
  Scratch scr(s);
  double* partial;
  FEMB_CUDA(scr.alloc(&partial, (size_t)grid * kk));
  mb_gram_kernel<<<grid, MB_THREADS, 0, s>>>(n, ka, A, lda, kb, B, ldb, partial);
  mb_partial_finish<<<ceil_div(kk, MB_THREADS), MB_THREADS, 0, s>>>(grid, kk, partial, G);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_mb_combine(int64_t n, int k, const double* X, int64_t ldx, int mc, const double* C_host, double beta, double* Y,
                               int64_t ldy, femb_stream stream) {
  FEMB_CHECK_ARG(k >= 1 && k <= MB_MAXK && mc >= 1 && mc <= MB_MAXM, "1 <= k <= 48, 1 <= mc <= 16");
  FEMB_CHECK_ARG(n >= 0 && X && Y && C_host, "n >= 0, non-null X, Y, C_host");
  FEMB_CHECK_ARG(ldx >= k && ldy >= mc, "ldx >= k, ldy >= mc");
  FEMB_CHECK_ARG(!views_overlap(X, ldx, k, Y, ldy, mc, n), "Y overlaps X");
  if (n == 0) return FEMB_OK;
  MbCoef C;
  memset(&C, 0, sizeof(C));
  memcpy(C.c, C_host, sizeof(double) * k * mc);
  mb_combine_kernel<<<grid_for(n * 16, MB_THREADS, 16), MB_THREADS, 0, as_stream(stream)>>>(n, k, X, ldx, mc, C, beta, Y, ldy);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_lobpcg_residual(int64_t n, int m, const double* X, int64_t ldx, const double* KX, const double* MX, int64_t ldk,
                                    const double* lam_host, const double* dinv, int na, const int32_t* active, double* W, int64_t ldw,
                                    double* norms, femb_stream stream) {
  FEMB_CHECK_ARG(m >= 1 && m <= MB_MAXM && na >= 0 && na <= m, "1 <= m <= 16, 0 <= na <= m");
  FEMB_CHECK_ARG(n >= 0 && X && KX && MX && lam_host && dinv && norms && (na == 0 || (active && W)),
                 "non-null X, KX, MX, lam_host, dinv, norms (and active, W when na > 0)");
  FEMB_CHECK_ARG(ldx >= m && ldk >= m && (na == 0 || ldw >= na), "ldx, ldk >= m, ldw >= na");
  FEMB_CHECK_ARG(na == 0 || (!views_overlap(W, ldw, na, X, ldx, m, n) && !views_overlap(W, ldw, na, KX, ldk, m, n) &&
                             !views_overlap(W, ldw, na, MX, ldk, m, n)),
                 "W overlaps X, KX or MX");
  cudaStream_t s = as_stream(stream);
  if (n == 0) {
    FEMB_CUDA(cudaMemsetAsync(norms, 0, sizeof(double) * 2 * m, s));
    return FEMB_OK;
  }
  MbLam lam;
  memset(&lam, 0, sizeof(lam));
  memcpy(lam.v, lam_host, sizeof(double) * m);
  const int grid = grid_for(n, MB_THREADS / 16, 4);
  Scratch scr(s);
  double* partial;
  FEMB_CUDA(scr.alloc(&partial, (size_t)grid * 2 * m));
  lobpcg_residual_kernel<<<grid, MB_THREADS, 0, s>>>(n, m, X, ldx, KX, MX, ldk, lam, dinv, na, active, W, ldw, partial);
  mb_partial_finish<<<1, MB_THREADS, 0, s>>>(grid, 2 * m, partial, norms);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}
