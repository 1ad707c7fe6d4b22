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
// Two more kernels make up the V-cycle preconditioner of subdivided_lowest_modes (femb200/multigrid.py), on the same layout:
//   mg_smooth        one damped-Jacobi step X_out = X_in + omega dinv (R - A X_in) and/or the residual R - A X_in, on the SpMM's
//                    block traversal (each 3x3 block of A read once for all m columns)
//   mg_transfer      Y (+)= mask (S (x) I3) X for a node-level scalar CSR S: the prolongation P and the restriction R = P^T
// and one to the smoothed-aggregation hierarchy of femb200/amg.py, whose transfers are rectangular 3x3 block-CSR matrices:
//   mg_transfer_bsr3 Y (+)= mask (T X) on the SpMM's block traversal
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
// The traversal is shared by the SpMM and the multigrid smoother (mg_smooth_kernel below); the lane (slot 0, column c) of each row
// hands its three row sums of K X (and M X) to the epilogue: epi(row, c, k0, k1, k2, m0, m1, m2).
template <bool HAS_M, class Epi>
__device__ __forceinline__ void bsr3_warp_rows(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                               const double* __restrict__ kval, const double* __restrict__ mval,
                                               const unsigned char* __restrict__ mask, int m, int log_mp, const double* __restrict__ X,
                                               long long ldx, Epi epi) {
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
    if (slot == 0 && col_ok) epi(row, c, k0, k1, k2, m0, m1, m2);
  }
}

template <bool HAS_M>
__global__ void __launch_bounds__(MB_THREADS) spmm_bsr3_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                                const double* __restrict__ kval, const double* __restrict__ mval,
                                                                const unsigned char* __restrict__ mask, int m, int log_mp,
                                                                const double* __restrict__ X, long long ldx, double* __restrict__ YK,
                                                                double* __restrict__ YM, long long ldy) {
  bsr3_warp_rows<HAS_M>(nb, brow, bcol, kval, mval, mask, m, log_mp, X, ldx,
                        [&](long long row, int c, double k0, double k1, double k2, double m0, double m1, double m2) {
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
                        });
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

// One damped-Jacobi step on m columns: t = mask (R - A X_in), Res = t and X_out = X_in + omega dinv t (each output optional).
// HAS_X = false is X_in = 0: t = mask R and the matrix is not read, so the lanes of slot 0 of each warp cover the rows directly.
template <bool HAS_X>
__global__ void __launch_bounds__(MB_THREADS) mg_smooth_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                                const double* __restrict__ aval, const unsigned char* __restrict__ mask,
                                                                const double* __restrict__ dinv, double omega, int m, int log_mp,
                                                                const double* __restrict__ R, long long ldr, const double* __restrict__ X,
                                                                long long ldx, double* __restrict__ Xo, long long ldo, double* __restrict__ Res,
                                                                long long ldres) {
  auto epi = [&](long long row, int c, double a0, double a1, double a2, double, double, double) {
    const double a[3] = {a0, a1, a2};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const long long r = 3 * row + d;
      const double t = (!mask || mask[r]) ? R[r * ldr + c] - a[d] : 0.0;
      if (Res) Res[r * ldres + c] = t;
      if (Xo) Xo[r * ldo + c] = (HAS_X ? X[r * ldx + c] : 0.0) + omega * dinv[r] * t;
    }
  };
  if (HAS_X) {
    bsr3_warp_rows<false>(nb, brow, bcol, aval, nullptr, mask, m, log_mp, X, ldx, epi);
  } else {
    const int c = threadIdx.x & 31;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    if (c < m)
      for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < nb; row += nwarps) epi(row, c, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0);
  }
}

// Y[3i+d, j] (+)= mask_out[3i+d] sum_k val[k] X[3 col[k]+d, j] for a node-level scalar CSR (the prolongation or the restriction):
// one warp per output node, lanes (slot, c) as in the SpMM, slots over the row's entries, summed by the same fixed xor tree.
__global__ void __launch_bounds__(MB_THREADS) mg_transfer_kernel(long long n_out, const int* __restrict__ crow, const int* __restrict__ col,
                                                                  const double* __restrict__ val, const unsigned char* __restrict__ mask_out,
                                                                  int m, int log_mp, const double* __restrict__ X, long long ldx, int accumulate,
                                                                  double* __restrict__ Y, long long ldy) {
  const int lane = threadIdx.x & 31;
  const int mp = 1 << log_mp;
  const int c = lane & (mp - 1), slot = lane >> log_mp, nslot = 32 >> log_mp;
  const bool col_ok = c < m;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n_out; row += nwarps) {
    const int k0 = __ldg(crow + row), k1 = __ldg(crow + row + 1);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int k = k0 + slot; k < k1; k += nslot) {
      const long long j = __ldg(col + k);
      const double v = __ldg(val + k);
      if (col_ok) {
        const double* xp = X + 3 * j * ldx + c;
        s0 += v * xp[0];
        s1 += v * xp[ldx];
        s2 += v * xp[2 * ldx];
      }
    }
    for (int o = mp; o < 32; o <<= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (slot == 0 && col_ok) {
      const double s[3] = {s0, s1, s2};
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const long long r = 3 * row + d;
        const double v = (!mask_out || mask_out[r]) ? s[d] : 0.0;
        double* y = Y + r * ldy + c;
        *y = accumulate ? *y + v : v;
      }
    }
  }
}

// Y (+)= mask_out (T X) for a rectangular 3x3 block-CSR T (n_out block rows, columns < n_in): the SpMM's traversal with an
// epilogue that masks and writes or accumulates.
__global__ void __launch_bounds__(MB_THREADS) mg_transfer_bsr3_kernel(long long n_out, const int* __restrict__ trow, const int* __restrict__ tcol,
                                                                       const double* __restrict__ tval, const unsigned char* __restrict__ mask_out,
                                                                       int m, int log_mp, const double* __restrict__ X, long long ldx, int accumulate,
                                                                       double* __restrict__ Y, long long ldy) {
  bsr3_warp_rows<false>(n_out, trow, tcol, tval, nullptr, nullptr, m, log_mp, X, ldx,
                        [&](long long row, int c, double t0, double t1, double t2, double, double, double) {
                          const double t[3] = {t0, t1, t2};
#pragma unroll
                          for (int d = 0; d < 3; ++d) {
                            const long long r = 3 * row + d;
                            const double v = (!mask_out || mask_out[r]) ? t[d] : 0.0;
                            double* y = Y + r * ldy + c;
                            *y = accumulate ? *y + v : v;
                          }
                        });
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

extern "C" int femb_mg_smooth_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* aval, const uint8_t* mask,
                                   const double* dinv, double omega, int m, const double* R, int64_t ldr, const double* X_in, int64_t ldx,
                                   double* X_out, int64_t ldo, double* Res, int64_t ldres, femb_stream stream) {
  FEMB_CHECK_ARG(m >= 1 && m <= MB_MAXM, "1 <= m <= 16");
  FEMB_CHECK_ARG(nb >= 0 && nnzb >= 0 && nnzb <= INT32_MAX, "nb >= 0, 0 <= nnzb < 2^31");
  FEMB_CHECK_ARG(brow && bcol && aval && R && (X_out || Res) && (!X_out || dinv),
                 "non-null brow, bcol, aval, R, at least one of X_out and Res (and dinv with X_out)");
  FEMB_CHECK_ARG(ldr >= m && (!X_in || ldx >= m) && (!X_out || ldo >= m) && (!Res || ldres >= m), "ldr, ldx, ldo, ldres >= m");
  const long long n = 3 * nb;
  const bool bad = (X_out && X_in && views_overlap(X_out, ldo, m, X_in, ldx, m, n)) || (X_out && views_overlap(X_out, ldo, m, R, ldr, m, n)) ||
                   (Res && X_in && views_overlap(Res, ldres, m, X_in, ldx, m, n)) || (Res && views_overlap(Res, ldres, m, R, ldr, m, n)) ||
                   (X_out && Res && views_overlap(X_out, ldo, m, Res, ldres, m, n));
  FEMB_CHECK_ARG(!bad, "outputs overlap the inputs or each other");
  if (nb == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  int log_mp = 0;
  while ((1 << log_mp) < m) ++log_mp;
  const int grid = grid_for(nb * 32, MB_THREADS, 32);
  if (X_in)
    mg_smooth_kernel<true><<<grid, MB_THREADS, 0, s>>>(nb, brow, bcol, aval, mask, dinv, omega, m, log_mp, R, ldr, X_in, ldx, X_out, ldo, Res, ldres);
  else
    mg_smooth_kernel<false><<<grid, MB_THREADS, 0, s>>>(nb, brow, bcol, aval, mask, dinv, omega, m, log_mp, R, ldr, nullptr, 0, X_out, ldo, Res, ldres);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_mg_transfer(int64_t n_out, int64_t n_in, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val,
                                const uint8_t* mask_out, int m, const double* X, int64_t ldx, int accumulate, double* Y, int64_t ldy,
                                femb_stream stream) {
  FEMB_CHECK_ARG(m >= 1 && m <= MB_MAXM, "1 <= m <= 16");
  FEMB_CHECK_ARG(n_out >= 0 && n_in >= 0 && nnz >= 0 && nnz <= INT32_MAX, "n_out, n_in >= 0, 0 <= nnz < 2^31");
  FEMB_CHECK_ARG(crow && col && val && X && Y, "non-null crow, col, val, X, Y");
  FEMB_CHECK_ARG(ldx >= m && ldy >= m, "ldx, ldy >= m");
  FEMB_CHECK_ARG(accumulate == 0 || accumulate == 1, "accumulate is 0 or 1");
  FEMB_CHECK_ARG(n_in == 0 || n_out == 0 || !spans_meet(Y, (3 * n_out - 1) * ldy + m, X, (3 * n_in - 1) * ldx + m), "Y overlaps X");
  if (n_out == 0) return FEMB_OK;
  int log_mp = 0;
  while ((1 << log_mp) < m) ++log_mp;
  mg_transfer_kernel<<<grid_for(n_out * 32, MB_THREADS, 32), MB_THREADS, 0, as_stream(stream)>>>(n_out, crow, col, val, mask_out, m, log_mp, X, ldx,
                                                                                                accumulate, Y, ldy);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_mg_transfer_bsr3(int64_t n_out, int64_t n_in, int64_t nnzb, const int32_t* trow, const int32_t* tcol, const double* tval,
                                     const uint8_t* mask_out, int m, const double* X, int64_t ldx, int accumulate, double* Y, int64_t ldy,
                                     femb_stream stream) {
  FEMB_CHECK_ARG(m >= 1 && m <= MB_MAXM, "1 <= m <= 16");
  FEMB_CHECK_ARG(n_out >= 0 && n_in >= 0 && nnzb >= 0 && nnzb <= INT32_MAX, "n_out, n_in >= 0, 0 <= nnzb < 2^31");
  FEMB_CHECK_ARG(trow && tcol && tval && X && Y, "non-null trow, tcol, tval, X, Y");
  FEMB_CHECK_ARG(ldx >= m && ldy >= m, "ldx, ldy >= m");
  FEMB_CHECK_ARG(accumulate == 0 || accumulate == 1, "accumulate is 0 or 1");
  FEMB_CHECK_ARG(n_in == 0 || n_out == 0 || !spans_meet(Y, (3 * n_out - 1) * ldy + m, X, (3 * n_in - 1) * ldx + m), "Y overlaps X");
  if (n_out == 0) return FEMB_OK;
  int log_mp = 0;
  while ((1 << log_mp) < m) ++log_mp;
  mg_transfer_bsr3_kernel<<<grid_for(n_out * 32, MB_THREADS, 32), MB_THREADS, 0, as_stream(stream)>>>(n_out, trow, tcol, tval, mask_out, m, log_mp,
                                                                                                      X, ldx, accumulate, Y, ldy);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}
