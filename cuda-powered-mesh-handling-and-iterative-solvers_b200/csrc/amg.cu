// Setup kernels of the smoothed-aggregation multigrid (femb200/amg.py).  Every level is a square 3x3 block-CSR operator; an
// aggregate a of fine nodes becomes two coarse pseudo-nodes 2a (translations) and 2a+1 (rotations), so the transfers P and R are
// rectangular 3x3 block-CSR matrices and the V-cycle of femb200/multigrid.py runs on every level unchanged.
//   aggregate   distance-2 maximal independent set (Bell, Dalton & Olson 2012) by synchronous rounds over the node graph; roots
//               take their neighbours, the rest join the neighbouring aggregate with the lowest id.  Pure functions of the
//               previous round's state: the result does not depend on thread scheduling.
//   tentative   one warp per aggregate: CholQR2 of the aggregate's [3 n_a, 6] near-nullspace (rigid-body modes on the finest
//               level), streamed over its nodes -> two 3x3 blocks per fine node, the coarse near-nullspace R and the coarse mask
//   spgemm      C = X Y for 3x3 block-CSR (symbolic: one warp per row, a bounded shared-memory column list; numeric: the warp
//               walks X's row in order and lanes own distinct output blocks per step, so every block sums in a fixed order)
//   transpose   R = P^T (stable radix sort of the block columns; blocks transposed)
#include <cub/cub.cuh>

#include "common.cuh"

namespace femb {

constexpr int AMG_THREADS = 256;
constexpr int SPG_WARPS = 4;      // warps per CTA of the SpGEMM passes
constexpr int SPG_CAP = 2048;     // distinct block columns one output row may hold (8 KB of shared memory per warp)

enum : int { ST_OUT = 0, ST_UNDECIDED = 1, ST_ROOT = 2 };

// fixed 32-bit integer hash (lowbias32) of the node id: the MIS priorities
__host__ __device__ __forceinline__ unsigned node_hash(unsigned x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

// (state, priority, id) packed so that the largest key wins: 2 bits state, 31 bits hash, 31 bits id
__device__ __forceinline__ unsigned long long mis_key(int state, long long i) {
  return ((unsigned long long)state << 62) | ((unsigned long long)(node_hash((unsigned)i) >> 1) << 31) | (unsigned long long)i;
}

__device__ __forceinline__ bool node_in(const unsigned char* mask, long long i) { return !mask || mask[3 * i] || mask[3 * i + 1] || mask[3 * i + 2]; }

__global__ void agg_init_kernel(long long nb, const unsigned char* __restrict__ mask, signed char* __restrict__ st) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x)
    st[i] = node_in(mask, i) ? ST_UNDECIDED : -1;
}

// t1[i] = max key over i and its included neighbours
__global__ void agg_max1_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol, const signed char* __restrict__ st,
                                unsigned long long* __restrict__ t1) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x) {
    if (st[i] < 0) continue;
    unsigned long long m = mis_key(st[i], i);
    for (int b = brow[i]; b < brow[i + 1]; ++b) {
      const int j = bcol[b];
      if (st[j] >= 0) {
        const unsigned long long k = mis_key(st[j], j);
        m = k > m ? k : m;
      }
    }
    t1[i] = m;
  }
}

// an undecided node whose key is the largest within distance 2 becomes a root; one with a root within distance 2 drops out
__global__ void agg_max2_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol, const signed char* __restrict__ st,
                                const unsigned long long* __restrict__ t1, signed char* __restrict__ st_out, int* __restrict__ undecided) {
  int left = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x) {
    int s = st[i];
    if (s == ST_UNDECIDED) {
      unsigned long long m = t1[i];
      for (int b = brow[i]; b < brow[i + 1]; ++b) {
        const int j = bcol[b];
        if (st[j] >= 0) m = t1[j] > m ? t1[j] : m;
      }
      if ((long long)(m & 0x7fffffffull) == i) s = ST_ROOT;
      else if ((int)(m >> 62) == ST_ROOT) s = ST_OUT;
      left += s == ST_UNDECIDED;
    }
    st_out[i] = (signed char)s;
  }
  left = __reduce_add_sync(0xffffffffu, left);
  if ((threadIdx.x & 31) == 0 && left) atomicAdd(undecided, left);  // an integer count: exact in any order
}

__global__ void agg_root_flag_kernel(long long nb, const signed char* __restrict__ st, int* __restrict__ flag) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i <= nb; i += (long long)gridDim.x * blockDim.x)
    flag[i] = i < nb && st[i] == ST_ROOT;
}

// roots take their rank; their neighbours join them (two roots are never within distance 2, so a node has at most one root neighbour)
__global__ void agg_roots_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol, const signed char* __restrict__ st,
                                 const int* __restrict__ rank, int* __restrict__ agg1) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x) {
    int a = -1;
    if (st[i] == ST_ROOT) {
      a = rank[i];
    } else if (st[i] >= 0) {
      for (int b = brow[i]; b < brow[i + 1]; ++b)
        if (st[bcol[b]] == ST_ROOT) a = rank[bcol[b]];
    }
    agg1[i] = a;
  }
}

// every node still left joins the aggregated neighbour with the lowest aggregate id (reads agg1 only, writes agg)
__global__ void agg_rest_kernel(long long nb, const int* __restrict__ brow, const int* __restrict__ bcol, const signed char* __restrict__ st,
                                const int* __restrict__ agg1, int* __restrict__ agg) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nb; i += (long long)gridDim.x * blockDim.x) {
    int a = agg1[i];
    if (a < 0 && st[i] >= 0)
      for (int b = brow[i]; b < brow[i + 1]; ++b) {
        const int c = agg1[bcol[b]];
        if (c >= 0 && (a < 0 || c < a)) a = c;
      }
    agg[i] = a;
  }
}

// ------------------------------------------------------------------------------------------------------------ tentative P
// Cholesky of a 6x6 Gram (lower triangle, g[i*(i+1)/2 + j], j <= i) with pivot dropping: a pivot d <= drop * max_k G_kk zeroes
// column k of L and clears kept bit k.
__device__ __forceinline__ void chol6_drop(const double* g, double drop, double L[6][6], int& kept) {
  double gmax = 0.0;
#pragma unroll
  for (int k = 0; k < 6; ++k) gmax = fmax(gmax, g[k * (k + 1) / 2 + k]);
#pragma unroll
  for (int k = 0; k < 6; ++k) {
#pragma unroll
    for (int i = 0; i < 6; ++i) L[i][k] = 0.0;
    double d = g[k * (k + 1) / 2 + k];
#pragma unroll
    for (int j = 0; j < k; ++j) d -= L[k][j] * L[k][j];
    if (!(d > drop * gmax)) {
      kept &= ~(1 << k);
      continue;
    }
    const double lkk = sqrt(d);
    L[k][k] = lkk;
#pragma unroll
    for (int i = k + 1; i < 6; ++i) {
      double s = g[i * (i + 1) / 2 + k];
#pragma unroll
      for (int j = 0; j < k; ++j) s -= L[i][j] * L[k][j];
      L[i][k] = s / lkk;
    }
  }
}

// q L^T = b for one row (dropped columns: q_k = 0)
__device__ __forceinline__ void row_solve(const double* b, const double L[6][6], double* q) {
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double s = b[k];
#pragma unroll
    for (int j = 0; j < k; ++j) s -= q[j] * L[k][j];
    q[k] = L[k][k] != 0.0 ? s / L[k][k] : 0.0;
  }
}

__device__ __forceinline__ void gram_add(double* g, const double* q) {
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) g[i * (i + 1) / 2 + j] += q[i] * q[j];
}

// Row d of node i of the aggregate's local near-nullspace [e_d | (e_k x (x_i - c)) s], masked dofs zero.  The finest level forms it
// from the coordinates; coarser levels carry the global modes B = [T_e | e_k x x] and re-centre them on the aggregate's centroid c
// (their pseudo-nodes sit at the centroids of the aggregates they came from): (e_k x (x - c)) s = (B_rot,k - sum_e (e_k x c)_e B_e) s.
__device__ __forceinline__ void nullspace_row(long long i, int d, const double* __restrict__ coords, const double* __restrict__ B,
                                              const unsigned char* __restrict__ mask, const double* c, double s, double* b) {
  if (mask && !mask[3 * i + d]) {
#pragma unroll
    for (int k = 0; k < 6; ++k) b[k] = 0.0;
    return;
  }
  if (B) {
#pragma unroll
    for (int k = 0; k < 6; ++k) b[k] = B[(3 * i + d) * 6 + k];
    const double ec[3][3] = {{0.0, -c[2], c[1]}, {c[2], 0.0, -c[0]}, {-c[1], c[0], 0.0}};  // ec[k][e] = (e_k x c)_e
#pragma unroll
    for (int k = 0; k < 3; ++k) b[3 + k] = (b[3 + k] - ec[k][0] * b[0] - ec[k][1] * b[1] - ec[k][2] * b[2]) * s;
    return;
  }
  const double r[3] = {(coords[3 * i] - c[0]) * s, (coords[3 * i + 1] - c[1]) * s, (coords[3 * i + 2] - c[2]) * s};
#pragma unroll
  for (int k = 0; k < 3; ++k) b[k] = k == d ? 1.0 : 0.0;
  // column 3+k is e_k x r; its component d
  b[3] = d == 0 ? 0.0 : (d == 1 ? -r[2] : r[1]);
  b[4] = d == 0 ? r[2] : (d == 1 ? 0.0 : -r[0]);
  b[5] = d == 0 ? -r[1] : (d == 1 ? r[0] : 0.0);
}

template <int N>
__device__ __forceinline__ void warp_sum_n(double* v) {
#pragma unroll
  for (int k = 0; k < N; ++k) v[k] = warp_sum(v[k]);
}

__global__ void __launch_bounds__(AMG_THREADS) amg_tentative_kernel(long long n_agg, const int* __restrict__ aptr, const int* __restrict__ anode,
                                                                    const unsigned char* __restrict__ mask, const double* __restrict__ coords,
                                                                    const double* __restrict__ B, double drop, const int* __restrict__ prow,
                                                                    int* __restrict__ pcol, double* __restrict__ pval, double* __restrict__ Bc,
                                                                    unsigned char* __restrict__ mask_c, double* __restrict__ coords_c) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long a = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; a < n_agg; a += nwarps) {
    const int p0 = aptr[a], p1 = aptr[a + 1];
    double c[3] = {0.0, 0.0, 0.0}, s = 1.0;
    {  // centroid and scale 1 / diameter (diameter: twice the largest distance from the centroid)
      for (int p = p0 + lane; p < p1; p += 32)
#pragma unroll
        for (int e = 0; e < 3; ++e) c[e] += coords[3 * (long long)anode[p] + e];
      warp_sum_n<3>(c);
      for (int e = 0; e < 3; ++e) c[e] /= (double)(p1 - p0);
      double rmax = 0.0;
      for (int p = p0 + lane; p < p1; p += 32) {
        const long long i = anode[p];
        const double dx = coords[3 * i] - c[0], dy = coords[3 * i + 1] - c[1], dz = coords[3 * i + 2] - c[2];
        rmax = fmax(rmax, sqrt(dx * dx + dy * dy + dz * dz));
      }
      for (int o = 16; o > 0; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
      s = rmax > 0.0 ? 1.0 / (2.0 * rmax) : 1.0;
    }
    double g[21], L1[6][6], L2[6][6], b[6], q1[6], q2[6];
    int kept = 63;
    // pass 1: G1 = B^T B
    for (int k = 0; k < 21; ++k) g[k] = 0.0;
    for (int p = p0 + lane; p < p1; p += 32)
      for (int d = 0; d < 3; ++d) {
        nullspace_row(anode[p], d, coords, B, mask, c, s, b);
        gram_add(g, b);
      }
    warp_sum_n<21>(g);
    chol6_drop(g, drop, L1, kept);
    // pass 2: G2 = Q1^T Q1, Q1 = B L1^-T
    for (int k = 0; k < 21; ++k) g[k] = 0.0;
    for (int p = p0 + lane; p < p1; p += 32)
      for (int d = 0; d < 3; ++d) {
        nullspace_row(anode[p], d, coords, B, mask, c, s, b);
        row_solve(b, L1, q1);
        gram_add(g, q1);
      }
    warp_sum_n<21>(g);
    chol6_drop(g, drop, L2, kept);
    // pass 3: Q = Q1 L2^-T -> blocks (i, 2a) = Q[:, 0:3], (i, 2a+1) = Q[:, 3:6]
    for (int p = p0 + lane; p < p1; p += 32) {
      const long long i = anode[p];
      const long long q = prow[i];
      for (int d = 0; d < 3; ++d) {
        nullspace_row(i, d, coords, B, mask, c, s, b);
        row_solve(b, L1, q1);
        row_solve(q1, L2, q2);
        for (int e = 0; e < 3; ++e) {
          pval[9 * q + 3 * d + e] = (kept >> e) & 1 ? q2[e] : 0.0;
          pval[9 * (q + 1) + 3 * d + e] = (kept >> (3 + e)) & 1 ? q2[3 + e] : 0.0;
        }
      }
      pcol[q] = (int)(2 * a);
      pcol[q + 1] = (int)(2 * a + 1);
    }
    // R = R2 R1 = L2^T L1^T: row k of R holds the coefficients of coarse dof 6a + k in the local columns.  The local rotation
    // columns are (e_m x x - e_m x c) s, so the global rigid-body modes are the local columns times T (T = I, but T[3+m][3+m] = 1/s
    // and T[d][3+m] = (e_m x c)_d): the coarse near-nullspace is R T, in global modes on every level.
    for (int e = lane; e < 36; e += 32) {
      const int k = e / 6, col = e - 6 * k;
      double rk[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        double r = 0.0;
        if ((kept >> k) & 1)
#pragma unroll
          for (int j = 0; j < 6; ++j) r += L2[j][k] * L1[i][j];
        rk[i] = r;
      }
      double v = rk[col];
      if (col >= 3) {
        v = rk[col] / s;
        const double zero[3] = {0.0, 0.0, 0.0};
        for (int d = 0; d < 3; ++d) {
          double t[6];
          nullspace_row(0, d, c, nullptr, nullptr, zero, 1.0, t);  // row d of [I3 | e_m x c]
          v += rk[d] * t[col];
        }
      }
      Bc[36 * a + e] = v;
    }
    if (lane < 6) mask_c[6 * a + lane] = (kept >> lane) & 1;
    if (lane < 6) coords_c[6 * a + lane] = c[lane % 3];  // both pseudo-nodes sit at the centroid
  }
}

__global__ void amg_flag_kernel(long long nb, const int* __restrict__ agg, int* __restrict__ flag, unsigned* __restrict__ key) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i <= nb; i += (long long)gridDim.x * blockDim.x) {
    flag[i] = i < nb && agg[i] >= 0;
    if (i < nb) key[i] = (unsigned)(agg[i] + 1);  // excluded nodes (agg -1) sort first
  }
}

__global__ void amg_prow_kernel(long long nb, const int* __restrict__ scan, int* __restrict__ prow) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i <= nb; i += (long long)gridDim.x * blockDim.x) prow[i] = 2 * scan[i];
}

// ptr[a] = first position of key a + key0 in the sorted keys (a = 0..n)
__global__ void lower_bound_kernel(long long n, long long len, const unsigned* __restrict__ keys, unsigned key0, int* __restrict__ ptr) {
  for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a <= n; a += (long long)gridDim.x * blockDim.x) {
    const unsigned k = (unsigned)a + key0;
    long long lo = 0, hi = len;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (keys[mid] < k) lo = mid + 1;
      else hi = mid;
    }
    ptr[a] = (int)lo;
  }
}

__global__ void iota_kernel(long long n, int* __restrict__ v) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) v[i] = (int)i;
}

static int sort_pairs(Scratch& scr, const unsigned* kin, unsigned* kout, const int* vin, int* vout, long long n, int end_bit, cudaStream_t s) {
  size_t tb = 0;
  FEMB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, kin, kout, vin, vout, (int)n, 0, end_bit, s));
  void* tmp;
  FEMB_CUDA(scr.alloc((char**)&tmp, tb));
  FEMB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, kin, kout, vin, vout, (int)n, 0, end_bit, s));
  return FEMB_OK;
}

static int scan_int(Scratch& scr, const int* in, int* out, long long n, cudaStream_t s) {
  size_t tb = 0;
  FEMB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, (int)n, s));
  void* tmp;
  FEMB_CUDA(scr.alloc((char**)&tmp, tb));
  FEMB_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, in, out, (int)n, s));
  return FEMB_OK;
}

static int key_bits(long long v) {
  int b = 1;
  while (b < 32 && (1ll << b) <= v) ++b;
  return b;
}

// ---------------------------------------------------------------------------------------------------------------- SpGEMM
// Symbolic pass, one warp per row of C = X Y: the distinct block columns of the row gathered in a shared list (lanes take the
// blocks of one Y row side by side; a column already listed is skipped, new ones are appended in lane order).  FILL = false
// writes the count, FILL = true the sorted columns at ccol[crow[i]..] (rank = number of smaller listed columns).
template <bool FILL>
__global__ void __launch_bounds__(SPG_WARPS * 32) spgemm_symbolic_kernel(long long n_rows, const int* __restrict__ xrow, const int* __restrict__ xcol,
                                                                         const int* __restrict__ yrow, const int* __restrict__ ycol,
                                                                         int* __restrict__ count, const int* __restrict__ crow,
                                                                         int* __restrict__ ccol, int* __restrict__ overflow) {
  __shared__ int list_all[SPG_WARPS][SPG_CAP];
  const int lane = threadIdx.x & 31;
  int* list = list_all[threadIdx.x >> 5];
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_rows; i += nwarps) {
    int len = 0;
    for (int k = xrow[i]; k < xrow[i + 1]; ++k) {
      const int r = xcol[k], j1 = yrow[r + 1];
      for (int jb = yrow[r]; jb < j1; jb += 32) {
        const int j = jb + lane;
        const int c = j < j1 ? ycol[j] : -1;
        bool fresh = c >= 0;
        const int lim = len < SPG_CAP ? len : SPG_CAP;
        for (int t = 0; t < lim && fresh; ++t) fresh = list[t] != c;
        const unsigned ballot = __ballot_sync(0xffffffffu, fresh);
        const int pos = len + __popc(ballot & ((1u << lane) - 1u));
        if (fresh && pos < SPG_CAP) list[pos] = c;
        len += __popc(ballot);
        __syncwarp();
      }
    }
    if (len > SPG_CAP) {
      if (lane == 0 && overflow) atomicMax(overflow, len);
      len = 0;
    }
    if (!FILL) {
      if (lane == 0) count[i] = len;
    } else {
      const long long c0 = crow[i];
      for (int t = lane; t < len; t += 32) {
        const int v = list[t];
        int rank = 0;
        for (int u = 0; u < len; ++u) rank += list[u] < v;
        ccol[c0 + rank] = v;
      }
    }
    __syncwarp();
  }
}

// Numeric pass, one warp per row: for each block k of X's row in order, lanes take the blocks of Y's row col(k) (distinct
// columns, hence distinct output blocks) and add X_k Y_j to the output block found by binary search in the row's columns.
__global__ void __launch_bounds__(SPG_WARPS * 32) spgemm_numeric_kernel(long long n_rows, const int* __restrict__ xrow, const int* __restrict__ xcol,
                                                                        const double* __restrict__ xval, const int* __restrict__ yrow,
                                                                        const int* __restrict__ ycol, const double* __restrict__ yval,
                                                                        const int* __restrict__ crow, const int* __restrict__ ccol, double* cval) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_rows; i += nwarps) {
    const int c0 = crow[i], c1 = crow[i + 1];
    for (long long e = 9ll * c0 + lane; e < 9ll * c1; e += 32) cval[e] = 0.0;
    __syncwarp();
    for (int k = xrow[i]; k < xrow[i + 1]; ++k) {
      const int r = xcol[k];
      double xb[9];
#pragma unroll
      for (int e = 0; e < 9; ++e) xb[e] = xval[9ll * k + e];
      for (int j = yrow[r] + lane; j < yrow[r + 1]; j += 32) {
        const int c = ycol[j];
        int lo = c0, hi = c1;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (ccol[mid] < c) lo = mid + 1;
          else hi = mid;
        }
        const double* yb = yval + 9ll * j;
        double* cb = cval + 9ll * lo;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
          for (int q = 0; q < 3; ++q) cb[3 * p + q] += xb[3 * p] * yb[q] + xb[3 * p + 1] * yb[3 + q] + xb[3 * p + 2] * yb[6 + q];
      }
      __syncwarp();
    }
  }
}

// --------------------------------------------------------------------------------------------------------------- transpose
__global__ void row_of_kernel(long long n_rows, const int* __restrict__ prow, int* __restrict__ row) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_rows; i += (long long)gridDim.x * blockDim.x)
    for (int b = prow[i]; b < prow[i + 1]; ++b) row[b] = (int)i;
}

__global__ void transpose_fill_kernel(long long nnzb, const int* __restrict__ order, const int* __restrict__ row, const double* __restrict__ pval,
                                      int* __restrict__ rcol, double* __restrict__ rval) {
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < nnzb; p += (long long)gridDim.x * blockDim.x) {
    const long long b = order[p];
    rcol[p] = row[b];
#pragma unroll
    for (int u = 0; u < 3; ++u)
#pragma unroll
      for (int v = 0; v < 3; ++v) rval[9 * p + 3 * u + v] = pval[9 * b + 3 * v + u];
  }
}

}  // namespace femb

using namespace femb;

extern "C" int femb_amg_aggregate(int64_t nb, const int32_t* brow, const int32_t* bcol, const uint8_t* mask, int32_t* agg, int64_t* n_agg_host,
                                  femb_stream stream) {
  FEMB_CHECK_ARG(nb >= 0 && nb < INT32_MAX, "0 <= nb < 2^31");
  FEMB_CHECK_ARG(brow && bcol && agg && n_agg_host, "non-null brow, bcol, agg, n_agg_host");
  *n_agg_host = 0;
  if (nb == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  Scratch scr(s);
  signed char *st0, *st1;
  unsigned long long* t1;
  int *undecided, *flag, *rank, *agg1;
  FEMB_CUDA(scr.alloc(&st0, nb));
  FEMB_CUDA(scr.alloc(&st1, nb));
  FEMB_CUDA(scr.alloc(&t1, nb));
  FEMB_CUDA(scr.alloc(&undecided, 1));
  FEMB_CUDA(scr.alloc(&flag, nb + 1));
  FEMB_CUDA(scr.alloc(&rank, nb + 1));
  FEMB_CUDA(scr.alloc(&agg1, nb));
  const int grid = grid_for(nb, AMG_THREADS);
  agg_init_kernel<<<grid, AMG_THREADS, 0, s>>>(nb, mask, st0);
  FEMB_LAUNCH_CHECK();
  for (long long round = 0;; ++round) {  // each round makes at least the largest undecided key a root: at most nb rounds
    FEMB_CUDA(cudaMemsetAsync(undecided, 0, sizeof(int), s));
    agg_max1_kernel<<<grid, AMG_THREADS, 0, s>>>(nb, brow, bcol, st0, t1);
    agg_max2_kernel<<<grid, AMG_THREADS, 0, s>>>(nb, brow, bcol, st0, t1, st1, undecided);
    FEMB_LAUNCH_CHECK();
    std::swap(st0, st1);
    int left = 0;
    FEMB_CUDA(cudaMemcpyAsync(&left, undecided, sizeof(int), cudaMemcpyDeviceToHost, s));
    FEMB_CUDA(cudaStreamSynchronize(s));
    if (left == 0) break;
    if (round > nb) {
      set_error("femb_amg_aggregate: the independent-set rounds did not terminate");
      return FEMB_ERR_CUDA;
    }
  }
  agg_root_flag_kernel<<<grid_for(nb + 1, AMG_THREADS), AMG_THREADS, 0, s>>>(nb, st0, flag);
  FEMB_LAUNCH_CHECK();
  if (int rc = scan_int(scr, flag, rank, nb + 1, s)) return rc;
  agg_roots_kernel<<<grid, AMG_THREADS, 0, s>>>(nb, brow, bcol, st0, rank, agg1);
  agg_rest_kernel<<<grid, AMG_THREADS, 0, s>>>(nb, brow, bcol, st0, agg1, agg);
  FEMB_LAUNCH_CHECK();
  int n_agg = 0;
  FEMB_CUDA(cudaMemcpyAsync(&n_agg, rank + nb, sizeof(int), cudaMemcpyDeviceToHost, s));
  FEMB_CUDA(cudaStreamSynchronize(s));
  *n_agg_host = n_agg;
  return FEMB_OK;
}

extern "C" int femb_amg_tentative(int64_t nb, int64_t n_agg, const int32_t* agg, const uint8_t* mask, const double* coords, const double* B,
                                  double drop, int32_t* prow, int32_t* pcol, double* pval, double* Bc, uint8_t* mask_c, double* coords_c,
                                  femb_stream stream) {
  FEMB_CHECK_ARG(nb >= 0 && nb < INT32_MAX && n_agg >= 0 && n_agg <= nb, "0 <= n_agg <= nb < 2^31");
  FEMB_CHECK_ARG(agg && prow && coords && (n_agg == 0 || (pcol && pval && Bc && mask_c && coords_c)),
                 "non-null agg, prow, coords (and pcol, pval, Bc, mask_c, coords_c when n_agg > 0)");
  FEMB_CHECK_ARG(drop >= 0.0 && drop < 1.0, "0 <= drop < 1");
  cudaStream_t s = as_stream(stream);
  Scratch scr(s);
  int *flag, *scan, *ids, *anode, *aptr;
  unsigned *key, *key_sorted;
  FEMB_CUDA(scr.alloc(&flag, nb + 1));
  FEMB_CUDA(scr.alloc(&scan, nb + 1));
  FEMB_CUDA(scr.alloc(&key, nb));
  FEMB_CUDA(scr.alloc(&key_sorted, nb));
  FEMB_CUDA(scr.alloc(&ids, nb));
  FEMB_CUDA(scr.alloc(&anode, nb));
  FEMB_CUDA(scr.alloc(&aptr, n_agg + 1));
  amg_flag_kernel<<<grid_for(nb + 1, AMG_THREADS), AMG_THREADS, 0, s>>>(nb, agg, flag, key);
  FEMB_LAUNCH_CHECK();
  if (int rc = scan_int(scr, flag, scan, nb + 1, s)) return rc;
  amg_prow_kernel<<<grid_for(nb + 1, AMG_THREADS), AMG_THREADS, 0, s>>>(nb, scan, prow);
  FEMB_LAUNCH_CHECK();
  if (nb == 0 || n_agg == 0) return FEMB_OK;
  // node lists of the aggregates, each in increasing node id (stable sort by aggregate)
  iota_kernel<<<grid_for(nb, AMG_THREADS), AMG_THREADS, 0, s>>>(nb, ids);
  if (int rc = sort_pairs(scr, key, key_sorted, ids, anode, nb, key_bits(n_agg + 1), s)) return rc;
  lower_bound_kernel<<<grid_for(n_agg + 1, AMG_THREADS), AMG_THREADS, 0, s>>>(n_agg, nb, key_sorted, 1u, aptr);
  amg_tentative_kernel<<<grid_for(n_agg * 32, AMG_THREADS, 16), AMG_THREADS, 0, s>>>(n_agg, aptr, anode, mask, coords, B, drop, prow, pcol, pval,
                                                                                  Bc, mask_c, coords_c);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_bsr3_spgemm(int64_t n_rows, const int32_t* xrow, const int32_t* xcol, const double* xval, const int32_t* yrow,
                                const int32_t* ycol, const double* yval, int32_t* crow, int32_t* ccol, double* cval, int64_t* nnz_host,
                                femb_stream stream) {
  FEMB_CHECK_ARG(n_rows >= 0 && n_rows < INT32_MAX, "0 <= n_rows < 2^31");
  FEMB_CHECK_ARG(xrow && xcol && yrow && ycol && crow, "non-null xrow, xcol, yrow, ycol, crow");
  FEMB_CHECK_ARG(!ccol == !cval && (ccol ? xval && yval : nnz_host != nullptr),
                 "symbolic pass: ccol = cval = NULL and nnz_host given; numeric pass: ccol, cval, xval, yval given");
  cudaStream_t s = as_stream(stream);
  const int grid = grid_for(n_rows * 32, SPG_WARPS * 32, 16);
  if (!ccol) {
    Scratch scr(s);
    int *count, *overflow;
    FEMB_CUDA(scr.alloc(&count, n_rows + 1));
    FEMB_CUDA(scr.alloc(&overflow, 1));
    FEMB_CUDA(cudaMemsetAsync(count, 0, sizeof(int) * (n_rows + 1), s));
    FEMB_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int), s));
    if (n_rows)
      spgemm_symbolic_kernel<false><<<grid, SPG_WARPS * 32, 0, s>>>(n_rows, xrow, xcol, yrow, ycol, count, nullptr, nullptr, overflow);
    FEMB_LAUNCH_CHECK();
    if (int rc = scan_int(scr, count, crow, n_rows + 1, s)) return rc;
    int nnz = 0, over = 0;
    FEMB_CUDA(cudaMemcpyAsync(&nnz, crow + n_rows, sizeof(int), cudaMemcpyDeviceToHost, s));
    FEMB_CUDA(cudaMemcpyAsync(&over, overflow, sizeof(int), cudaMemcpyDeviceToHost, s));
    FEMB_CUDA(cudaStreamSynchronize(s));
    if (over) {
      set_error("femb_bsr3_spgemm: a row of the product has " + std::to_string(over) + " blocks, beyond the kernel's capacity of " +
                std::to_string(SPG_CAP) + " per row");
      return FEMB_ERR_UNSUPPORTED;
    }
    *nnz_host = nnz;
    return FEMB_OK;
  }
  if (n_rows == 0) return FEMB_OK;
  spgemm_symbolic_kernel<true><<<grid, SPG_WARPS * 32, 0, s>>>(n_rows, xrow, xcol, yrow, ycol, nullptr, crow, ccol, nullptr);
  spgemm_numeric_kernel<<<grid, SPG_WARPS * 32, 0, s>>>(n_rows, xrow, xcol, xval, yrow, ycol, yval, crow, ccol, cval);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_bsr3_transpose(int64_t n_rows, int64_t n_cols, int64_t nnzb, const int32_t* prow, const int32_t* pcol, const double* pval,
                                   int32_t* rrow, int32_t* rcol, double* rval, femb_stream stream) {
  FEMB_CHECK_ARG(n_rows >= 0 && n_rows < INT32_MAX && n_cols >= 0 && n_cols < INT32_MAX && nnzb >= 0 && nnzb < INT32_MAX,
                 "0 <= n_rows, n_cols, nnzb < 2^31");
  FEMB_CHECK_ARG(prow && rrow && (nnzb == 0 || (pcol && pval && rcol && rval)), "non-null prow, rrow (and pcol, pval, rcol, rval when nnzb > 0)");
  cudaStream_t s = as_stream(stream);
  if (nnzb == 0) {
    FEMB_CUDA(cudaMemsetAsync(rrow, 0, sizeof(int) * (n_cols + 1), s));
    return FEMB_OK;
  }
  Scratch scr(s);
  int *ids, *order, *row;
  unsigned* key_sorted;
  FEMB_CUDA(scr.alloc(&ids, nnzb));
  FEMB_CUDA(scr.alloc(&order, nnzb));
  FEMB_CUDA(scr.alloc(&row, nnzb));
  FEMB_CUDA(scr.alloc(&key_sorted, nnzb));
  iota_kernel<<<grid_for(nnzb, AMG_THREADS), AMG_THREADS, 0, s>>>(nnzb, ids);
  row_of_kernel<<<grid_for(n_rows, AMG_THREADS), AMG_THREADS, 0, s>>>(n_rows, prow, row);
  FEMB_LAUNCH_CHECK();
  if (int rc = sort_pairs(scr, reinterpret_cast<const unsigned*>(pcol), key_sorted, ids, order, nnzb, key_bits(n_cols), s)) return rc;
  lower_bound_kernel<<<grid_for(n_cols + 1, AMG_THREADS), AMG_THREADS, 0, s>>>(n_cols, nnzb, key_sorted, 0u, rrow);
  transpose_fill_kernel<<<grid_for(nnzb, AMG_THREADS), AMG_THREADS, 0, s>>>(nnzb, order, row, pval, rcol, rval);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}
