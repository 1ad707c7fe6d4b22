// Solid element kernels: C3D4 (closed form) and the isoparametric family C3D10 / C3D8 / C3D6 / C3D20 / C3D15:
// stiffness, consistent mass, stress recovery.
//
// Reference behaviour being reproduced (solver/element.py): compute_c3d4_{B,K}_matrix :835-903,
// compute_c3d10_* :1026-1239, compute_c3d8_* :1601-1803, compute_c3d6_* :2482-2676, volumes :514, :1248, :2198.
// Nothing here materialises B for the K paths: with isotropic D the node-pair block is
//   K_ab[i][j] = lambda g_a[i] g_b[j] + mu g_a[j] g_b[i] + mu delta_ij (g_a . g_b)
// which is B_a^T D B_b written out (Voigt order xx,yy,zz,xy,yz,zx, engineering shear).
#include "common.cuh"

namespace femb {

// ------------------------------------------------------------------------------------------------
// C3D4: one thread per element, 256-bit stores of complete 32-byte sectors.
// ------------------------------------------------------------------------------------------------
template <typename T>
struct Tet {
  T g[4][3];
  T det;
};

template <typename T, typename I>
__device__ __forceinline__ void tet_setup(const T* __restrict__ coords, const I* __restrict__ conn, long long e, Tet<T>& t,
                                          long long* ids = nullptr) {
  long long n[4];
  if (sizeof(I) == 8) {  // one 256-bit load of the element's four int64 ids
    asm volatile("ld.global.nc.L1::no_allocate.v4.s64 {%0,%1,%2,%3}, [%4];" : "=l"(n[0]), "=l"(n[1]), "=l"(n[2]), "=l"(n[3]) : "l"(conn + 4 * e));
  } else {
    const int4 q = __ldg(reinterpret_cast<const int4*>(conn) + e);
    n[0] = q.x, n[1] = q.y, n[2] = q.z, n[3] = q.w;
  }
  if (ids)
#pragma unroll
    for (int a = 0; a < 4; ++a) ids[a] = n[a];
  T x[4][3];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int k = 0; k < 3; ++k) x[a][k] = __ldg(coords + 3 * n[a] + k);
  T e1[3], e2[3], e3[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    e1[k] = x[1][k] - x[0][k];
    e2[k] = x[2][k] - x[0][k];
    e3[k] = x[3][k] - x[0][k];
  }
  // cofactor columns of inv([e1;e2;e3])
  T c1[3] = {e2[1] * e3[2] - e2[2] * e3[1], e2[2] * e3[0] - e2[0] * e3[2], e2[0] * e3[1] - e2[1] * e3[0]};
  T c2[3] = {e3[1] * e1[2] - e3[2] * e1[1], e3[2] * e1[0] - e3[0] * e1[2], e3[0] * e1[1] - e3[1] * e1[0]};
  T c3[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
  t.det = e1[0] * c1[0] + e1[1] * c1[1] + e1[2] * c1[2];
  const T id = T(1) / t.det;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    t.g[1][k] = c1[k] * id;
    t.g[2][k] = c2[k] * id;
    t.g[3][k] = c3[k] * id;
    t.g[0][k] = -(t.g[1][k] + t.g[2][k] + t.g[3][k]);
  }
}

template <typename T>
__device__ __forceinline__ void store_row12(T* p, const T* v) {
#pragma unroll
  for (int k = 0; k < 12; ++k) p[k] = v[k];
}
template <>
__device__ __forceinline__ void store_row12<double>(double* p, const double* v) {
  st256(p, v[0], v[1], v[2], v[3]);
  st256(p + 4, v[4], v[5], v[6], v[7]);
  st256(p + 8, v[8], v[9], v[10], v[11]);
}

template <typename T>
__device__ __forceinline__ void store_row4(T* p, const T* v) {
#pragma unroll
  for (int k = 0; k < 4; ++k) p[k] = v[k];
}
template <>
__device__ __forceinline__ void store_row4<double>(double* p, const double* v) {
  st256(p, v[0], v[1], v[2], v[3]);
}

// WHAT: 0 gradients [M,4,3]; 1 B [M,6,12]; 2 K [M,12,12]; 3 Poisson [M,4,4]; 4 mass [M,12,12]; 5 volume [M]
template <typename T, typename I, int WHAT>
__global__ void __launch_bounds__(128) c3d4_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M,
                                                   T lam, T mu, T* __restrict__ out, int* __restrict__ flag) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    Tet<T> t;
    tet_setup(coords, conn, e, t);
    if (WHAT != 5 && WHAT != 4 && fabs((double)t.det) < 1e-12 && flag) *flag = 1;
    const T V = fabs(t.det) / T(6);
    if (WHAT == 5) {
      out[e] = V;
    } else if (WHAT == 0) {
      T* o = out + e * 12;
      T v[12];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int k = 0; k < 3; ++k) v[3 * a + k] = t.g[a][k];
      store_row12(o, v);
    } else if (WHAT == 1) {
      T* o = out + e * 72;
      // rows: xx, yy, zz, xy, yz, zx (element.py:870-879)
      const int c0[6] = {0, -1, -1, 1, -1, 2};  // which gradient component lands in dof column 0 / 1 / 2
      const int c1[6] = {-1, 1, -1, 0, 2, -1};
      const int c2[6] = {-1, -1, 2, -1, 1, 0};
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        T v[12];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          v[3 * a + 0] = c0[r] >= 0 ? t.g[a][c0[r]] : T(0);
          v[3 * a + 1] = c1[r] >= 0 ? t.g[a][c1[r]] : T(0);
          v[3 * a + 2] = c2[r] >= 0 ? t.g[a][c2[r]] : T(0);
        }
        store_row12(o + 12 * r, v);
      }
    } else if (WHAT == 2) {
      T* o = out + e * 144;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          T v[12];
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const T dot = t.g[a][0] * t.g[b][0] + t.g[a][1] * t.g[b][1] + t.g[a][2] * t.g[b][2];
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              T k = lam * t.g[a][i] * t.g[b][j] + mu * t.g[a][j] * t.g[b][i];
              if (i == j) k += mu * dot;
              v[3 * b + j] = k * V;
            }
          }
          store_row12(o + 12 * (3 * a + i), v);
        }
      }
    } else if (WHAT == 3) {
      T* o = out + e * 16;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        T v[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) v[b] = (t.g[a][0] * t.g[b][0] + t.g[a][1] * t.g[b][1] + t.g[a][2] * t.g[b][2]) * V;
        store_row4(o + 4 * a, v);
      }
    } else if (WHAT == 4) {
      T* o = out + e * 144;
      const T m = lam * V / T(20);  // lam carries rho
#pragma unroll
      for (int r = 0; r < 12; ++r) {
        T v[12];
#pragma unroll
        for (int c = 0; c < 12; ++c) v[c] = (r % 3 == c % 3) ? (r == c ? 2 * m : m) : T(0);
        store_row12(o + 12 * r, v);
      }
    }
  }
}

template <typename T, typename I>
static int c3d4_dispatch(int what, const void* coords, const void* conn, long long M, double E, double nu, void* out, int* flag,
                         cudaStream_t s) {
  if (M == 0) return FEMB_OK;
  const double c = E / ((1 + nu) * (1 - 2 * nu));
  T lam = (T)(c * nu), mu = (T)(c * (1 - 2 * nu) / 2);
  if (what == 4) lam = (T)E;
  const int grid = grid_for(M, 128);
  const T* X = static_cast<const T*>(coords);
  const I* C = static_cast<const I*>(conn);
  T* O = static_cast<T*>(out);
  switch (what) {
    case 0: c3d4_kernel<T, I, 0><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    case 1: c3d4_kernel<T, I, 1><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    case 2: c3d4_kernel<T, I, 2><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    case 3: c3d4_kernel<T, I, 3><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    case 4: c3d4_kernel<T, I, 4><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    case 5: c3d4_kernel<T, I, 5><<<grid, 128, 0, s>>>(X, C, M, lam, mu, O, flag); break;
    default: set_error("femb_c3d4: unknown `what`"); return FEMB_ERR_ARG;
  }
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

// Geometric stiffness of the stress of a displacement field (not in the reference), one thread per element.  The strain is
// constant on a C3D4, so H = sum_a g_a (x) u_a, sigma = lam tr(H) I + mu (H + H^T) and s_ab = V g_a^T sigma g_b are formed in
// registers; block (a,b) of the [12,12] output is s_ab I3.  s_ab is computed once for a <= b and mirrored (bitwise symmetric).
template <typename T, typename I>
__global__ void __launch_bounds__(128) c3d4_geometric_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M,
                                                             const T* __restrict__ disp, T lam, T mu, T* __restrict__ out) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    Tet<T> t;
    long long n[4];
    tet_setup(coords, conn, e, t, n);
    T H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // H[i][k] = du_k / dx_i
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const T u[3] = {__ldg(disp + 3 * n[a]), __ldg(disp + 3 * n[a] + 1), __ldg(disp + 3 * n[a] + 2)};
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) H[3 * i + k] += t.g[a][i] * u[k];
    }
    const T V = fabs(t.det) / T(6), tr = lam * (H[0] + H[4] + H[8]);
    T sig[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k) sig[3 * i + k] = V * (mu * (H[3 * i + k] + H[3 * k + i]) + (i == k ? tr : T(0)));
    T s[4][4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const T sg[3] = {sig[0] * t.g[b][0] + sig[1] * t.g[b][1] + sig[2] * t.g[b][2],
                       sig[3] * t.g[b][0] + sig[4] * t.g[b][1] + sig[5] * t.g[b][2],
                       sig[6] * t.g[b][0] + sig[7] * t.g[b][1] + sig[8] * t.g[b][2]};
#pragma unroll
      for (int a = 0; a <= b; ++a) s[a][b] = s[b][a] = t.g[a][0] * sg[0] + t.g[a][1] * sg[1] + t.g[a][2] * sg[2];
    }
    T* o = out + e * 144;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        T v[12];
#pragma unroll
        for (int c = 0; c < 12; ++c) v[c] = (c % 3 == i) ? s[a][c / 3] : T(0);
        store_row12(o + 12 * (3 * a + i), v);
      }
  }
}

// ------------------------------------------------------------------------------------------------
// Volumes through the reference's sub-tet tables
// ------------------------------------------------------------------------------------------------
__constant__ int c_vol_tets[2][6][4] = {
    {{0, 1, 3, 4}, {1, 2, 3, 6}, {1, 3, 4, 5}, {3, 4, 5, 7}, {3, 5, 6, 7}, {3, 5, 6, 1}},   // hex  (element.py:1282-1287)
    {{0, 1, 2, 3}, {1, 2, 4, 3}, {2, 4, 5, 3}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}}};  // wedge (element.py:2226-2228)

template <typename T>
__device__ __forceinline__ T abs_tet_vol(const T (*x)[3], const int* t) {
  T a[3], b[3], c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    a[k] = x[t[1]][k] - x[t[0]][k];
    b[k] = x[t[2]][k] - x[t[0]][k];
    c[k] = x[t[3]][k] - x[t[0]][k];
  }
  const T d = a[0] * (b[1] * c[2] - b[2] * c[1]) - a[1] * (b[0] * c[2] - b[2] * c[0]) + a[2] * (b[0] * c[1] - b[1] * c[0]);
  return fabs(d) / T(6);
}

template <typename T, typename I, int NEN>
__global__ void volumes_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M, int stride, T* __restrict__ vol) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    T x[NEN][3];
#pragma unroll
    for (int a = 0; a < NEN; ++a) {
      const long long n = ldidx(conn + e * stride + a);
#pragma unroll
      for (int k = 0; k < 3; ++k) x[a][k] = __ldg(coords + 3 * n + k);
    }
    if (NEN == 4) {
      const int t[4] = {0, 1, 2, 3};
      vol[e] = abs_tet_vol<T>(x, t);
    } else {
      const int which = NEN == 8 ? 0 : 1, nt = NEN == 8 ? 6 : 3;
      T v = 0;
      for (int s = 0; s < nt; ++s) v += abs_tet_vol<T>(x, c_vol_tets[which][s]);
      vol[e] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Isoparametric solids.  One CTA = EPB elements; the natural-coordinate tables live in shared memory.
//   phase A1: thread (element, point, i)    -> row i of J = sum_a dN_a[i] x_a
//   phase A2: thread (element, point)       -> J^-1 (closed form), detJ * w
//   phase A3: thread (element, point, node) -> gradient g_a = J^-1 dN_a
//   phase B : thread (element, a<=b)        -> 3x3 node-pair block accumulated over the points, written (and mirrored)
//             into a shared K tile
//   phase C : the whole CTA streams the tile to global memory with coalesced stores
// ------------------------------------------------------------------------------------------------
// shared -> global bulk copy (TMA engine, 1-D): the finished K tile drains to HBM while the CTA already works on its next
// elements.  Source and destination 16-byte aligned, size a multiple of 16 bytes.
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

struct SolidTab {
  const double* dN;  // [nq][nen][3]
  const double* w;   // [nq]
  const double* N;   // [nq][nen] shape-function values (mass)
};

template <typename T, typename I, int NEN, int EPB>
__global__ void __launch_bounds__(512) solid_K_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M, SolidTab tab, int nq, int mode,
                               T lam, T mu, T* __restrict__ out) {
  constexpr int ND = 3 * NEN;
  constexpr int NPAIR = NEN * (NEN + 1) / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* kt = reinterpret_cast<T*>(smem_raw);         // [EPB][ND][ND]   (first: 16-byte aligned for the vector stores)
  T* xs = kt + (size_t)EPB * ND * ND;             // [EPB][NEN][3]
  T* gs = xs + EPB * NEN * 3;                     // [EPB][nq][NEN][3]
  T* wd = gs + (size_t)EPB * nq * NEN * 3;        // [EPB][nq]
  T* js = wd + EPB * nq;                          // [EPB][nq][9]  J, then J^-1
  T* dns = js + (size_t)EPB * nq * 9;             // [nq][NEN][3]
  T* nsh = dns + (size_t)nq * NEN * 3;            // [nq][NEN]
  T* wsh = nsh + (size_t)nq * NEN;                // [nq]
  const int tid = threadIdx.x;
  const int nslice = mode == 4 ? nq : 1;
  // element tiles whose byte size is a multiple of 16 leave through the TMA engine (all but C3D15: 45*45 entries)
  constexpr bool BULK = (ND * ND * sizeof(T)) % 16 == 0;
  for (int t = tid; t < nq * NEN * 3; t += blockDim.x) dns[t] = (T)tab.dN[t];
  for (int t = tid; t < nq * NEN; t += blockDim.x) nsh[t] = (T)tab.N[t];
  for (int t = tid; t < nq; t += blockDim.x) wsh[t] = (T)tab.w[t];

  for (long long e0 = (long long)blockIdx.x * EPB; e0 < M; e0 += (long long)gridDim.x * EPB) {
    const int ne = (int)min((long long)EPB, M - e0);
    __syncthreads();
    for (int t = tid; t < ne * NEN; t += blockDim.x) {
      const long long n = ldidx(conn + e0 * NEN + t);
#pragma unroll
      for (int k = 0; k < 3; ++k) xs[t * 3 + k] = __ldg(coords + 3 * n + k);
    }
    __syncthreads();
    // ---- phase A1: rows of J
    for (int t = tid; t < ne * nq * 3; t += blockDim.x) {
      const int eq = t / 3, i = t - eq * 3, el = eq / nq, q = eq - el * nq;
      const T* x = xs + el * NEN * 3;
      const T* dn = dns + (size_t)q * NEN * 3 + i;
      T j0 = 0, j1 = 0, j2 = 0;
#pragma unroll
      for (int a = 0; a < NEN; ++a) {
        const T d = dn[a * 3];
        j0 += d * x[a * 3], j1 += d * x[a * 3 + 1], j2 += d * x[a * 3 + 2];
      }
      T* J = js + (size_t)eq * 9 + i * 3;
      J[0] = j0, J[1] = j1, J[2] = j2;
    }
    __syncthreads();
    // ---- phase A2: inverse and weight
    for (int t = tid; t < ne * nq; t += blockDim.x) {
      const int el = t / nq, q = t - el * nq;
      T J[9], Ji[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) J[k] = js[(size_t)t * 9 + k];
      const T det = inv3(J, Ji);
#pragma unroll
      for (int k = 0; k < 9; ++k) js[(size_t)t * 9 + k] = Ji[k];
      T wt;
      if (mode == 6) {  // consistent mass: rho |detJ| w (rho arrives in `lam`)
        wt = lam * fabs(det) * wsh[q];
      } else if (mode == 5) {  // C3D6 single=True: |volume| of the reference's 3-tet split (element.py:2226-2228, 2652-2656)
        const T* x = xs + el * NEN * 3;
        T xx[6][3];
        for (int a = 0; a < 6 && a < NEN; ++a)
          for (int k = 0; k < 3; ++k) xx[a][k] = x[a * 3 + k];
        wt = 0;
        for (int s = 0; s < 3; ++s) wt += abs_tet_vol<T>(xx, c_vol_tets[1][s]);
      } else {
        wt = mode == 4 ? det : det * wsh[q];
      }
      wd[t] = wt;
    }
    __syncthreads();
    // ---- phase A3: gradients (not needed by the mass)
    if (mode != 6)
      for (int t = tid; t < ne * nq * NEN; t += blockDim.x) {
        const int eq = t / NEN, a = t - eq * NEN, q = eq % nq;
        const T* Ji = js + (size_t)eq * 9;
        const T* dn = dns + ((size_t)q * NEN + a) * 3;
        const T d0 = dn[0], d1 = dn[1], d2 = dn[2];
        T* g = gs + (size_t)t * 3;
        g[0] = Ji[0] * d0 + Ji[1] * d1 + Ji[2] * d2;
        g[1] = Ji[3] * d0 + Ji[4] * d1 + Ji[5] * d2;
        g[2] = Ji[6] * d0 + Ji[7] * d1 + Ji[8] * d2;
      }
    __syncthreads();
    for (int slice = 0; slice < nslice; ++slice) {
      if (BULK) {  // the previous tile must have been read out of shared memory before phase B overwrites it
        if (tid == 0) bulk_wait_read();
        __syncthreads();
      }
      // ---- phase B
      for (int t = tid; t < ne * NPAIR; t += blockDim.x) {
        const int el = t / NPAIR;
        int p = t - el * NPAIR;
        int a = 0;
        while (p >= NEN - a) {
          p -= NEN - a;
          ++a;
        }
        const int b = a + p;
        T acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        const int q0 = mode == 4 ? slice : 0, q1 = mode == 4 ? slice + 1 : nq;
        if (mode == 6) {  // m_ab = sum_q rho |detJ| w N_a N_b on the diagonal of the 3x3 block
          T m = 0;
          for (int q = 0; q < nq; ++q) m += wd[el * nq + q] * (nsh[q * NEN + a] * nsh[q * NEN + b]);
          acc[0] = acc[4] = acc[8] = m;
        } else {
          // S[i][j] = sum_q w g_a[i] g_b[j]; the block is lam S + mu S^T + mu tr(S) I -- 12 FMAs per point instead of forming
          // lam g_a[i] g_b[j] + mu g_a[j] g_b[i] + mu delta_ij g_a.g_b point by point (33 operations)
          T S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
          for (int q = q0; q < q1; ++q) {
            const T* g = gs + ((size_t)el * nq + q) * NEN * 3;
            const T w = wd[el * nq + q];
            const T wa[3] = {w * g[a * 3], w * g[a * 3 + 1], w * g[a * 3 + 2]};
            const T gb[3] = {g[b * 3], g[b * 3 + 1], g[b * 3 + 2]};
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
              for (int j = 0; j < 3; ++j) S[i * 3 + j] += wa[i] * gb[j];
          }
          const T tr = mu * (S[0] + S[4] + S[8]);
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) acc[i * 3 + j] = lam * S[i * 3 + j] + mu * S[j * 3 + i] + (i == j ? tr : T(0));
        }
        T* K = kt + (size_t)el * ND * ND;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            K[(3 * a + i) * ND + 3 * b + j] = acc[i * 3 + j];
            K[(3 * b + j) * ND + 3 * a + i] = acc[i * 3 + j];
          }
      }
      __syncthreads();
      // ---- phase C
      T* dst = out + ((size_t)slice * M + e0) * ND * ND;
      const int total = ne * ND * ND;
      if (BULK) {
        if (tid == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the generic-proxy writes of phase B, ordered by the barrier above
          bulk_s2g(dst, kt, (unsigned)(total * sizeof(T)));
        }
        continue;  // no barrier here: the wait + barrier before the next phase B protects the tile
      }
      if (sizeof(T) == 8 && (ND * ND) % 2 == 0) {  // even tiles: every element starts 16-byte aligned
        for (int t = 2 * tid; t < total; t += 2 * blockDim.x)
          st128(reinterpret_cast<double*>(dst) + t, (double)kt[t], (double)kt[t + 1]);
      } else {  // C3D15: 45*45 is odd
        for (int t = tid; t < total; t += blockDim.x) dst[t] = kt[t];
      }
      __syncthreads();
    }
  }
  if (BULK && tid == 0) bulk_wait_all();  // shared memory must outlive the last copy
}

// ------------------------------------------------------------------------------------------------
// C3D10 stiffness, one WARP per element (no CTA barriers: the phases of different warps overlap on the LSU / fp64 pipes).
// solid_K_kernel above spends its time in the shared-memory pipe (l1tex 87 %, ~640 wavefronts per element): derivative
// tables, Jacobians and gradients all travel through shared memory at 2 loads per FMA.  Here
//   phase A  lane (q, h) = (lane/2, lane%2), q < nq <= 16: the point's derivative table lives in REGISTERS for the whole kernel;
//            J_q (both halves, redundantly), its inverse, the gradients of nodes 5h..5h+4 -> shared gs[q][a][3], w det -> wd[q]
//   phase B  lane = tile (t, b), 30 tiles: node pairs (2t, b) and (2t+1, b), b >= 2t; per point three 128-bit loads for the two
//            a-rows (the same five addresses across the warp), three 64-bit loads for the b-row (ten addresses), 18 FMAs;
//            K_ab = lam S + mu S^T + mu tr(S) I and its mirror image go to the warp's K tile
//   store    the tile leaves through the TMA engine while the warp is already in phase A of its next element
// Connectivity is requested two elements ahead and coordinates one element ahead.
//
// GEO = true: the geometric stiffness of the stress of `disp` (femb_solid_geometric) with the same layout.  Displacements are
// gathered beside the coordinates; in phase A lane (q, h) also forms G = sum_a dN_a (x) u_a, H = J^-1 G and
// S_q = w_q |detJ_q| sigma_q in registers and stores t_a = S_q g_a next to g_a (ts[q][a][3]); in phase B the tile's lane sums
// s_ab = sum_q t_a . g_b (6 FMAs per point) and the blocks s_ab I3 go through the same tile and TMA store.
// ------------------------------------------------------------------------------------------------
constexpr int C10W_WARPS = 4, C10W_MAXQ = 16;
constexpr int C10W_GQ = 36;   // gs row stride per point (30 used): with 36 the 128-bit stores of phase A and loads of phase B are conflict-free
constexpr int C10W_PER_WARP = 900 + C10W_MAXQ * C10W_GQ + C10W_MAXQ + 32;   // K tile | gs | wd | xs   (T units, a multiple of 4)
constexpr int C10W_PER_WARP_GEO = C10W_PER_WARP + 32 + C10W_MAXQ * C10W_GQ;  // ... | us | ts

// NQ > 0: the number of points is a compile-time constant (the reference's 11-point rule): phase B unrolls completely and its
// loads run ahead of the FMAs of earlier points; NQ = 0: any nq_rt <= 16.
template <typename T, typename I, int MINB, int NQ, bool GEO>
__global__ void __launch_bounds__(C10W_WARPS * 32, MINB) c3d10_K_warp_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M,
                                                                             SolidTab tab, int nq_rt, T lam, T mu, T* __restrict__ out,
                                                                             const T* __restrict__ disp) {
  constexpr int NEN = 10, ND = 30;
  const int nq = NQ ? NQ : nq_rt;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  T* kt = reinterpret_cast<T*>(smem_raw) + (size_t)w * (GEO ? C10W_PER_WARP_GEO : C10W_PER_WARP);
  T* gs = kt + ND * ND;
  T* wd = gs + C10W_MAXQ * C10W_GQ;
  T* xs = wd + C10W_MAXQ;
  T* us = xs + 32;                // GEO only
  T* ts = us + 32;                // GEO only
  const long long nwarps = (long long)gridDim.x * C10W_WARPS, warp0 = (long long)blockIdx.x * C10W_WARPS + w;
  // phase-A role
  const int q = lane >> 1, h = lane & 1;
  const bool act = q < nq;
  T dn[NEN][3], wq = 0;
#pragma unroll
  for (int a = 0; a < NEN; ++a)
#pragma unroll
    for (int k = 0; k < 3; ++k) dn[a][k] = act ? (T)tab.dN[((size_t)q * NEN + a) * 3 + k] : T(0);
  if (act) wq = (T)tab.w[q];
  // phase-B role
  int t = 0, b = 0;
  if (lane < 10) t = 0, b = lane;
  else if (lane < 18) t = 1, b = lane - 8;
  else if (lane < 24) t = 2, b = lane - 14;
  else if (lane < 28) t = 3, b = lane - 18;
  else t = 4, b = min(lane, 29) - 20;
  const bool tile = lane < 30;
  const int a0 = 2 * t, a1 = a0 + 1;
  // gather pipeline: lane l < 30 owns component l%3 of node l/3
  const int ga = lane < 30 ? lane / 3 : 0, gc = lane < 30 ? lane - 3 * (lane / 3) : 0;
  long long n1 = 0;   // node of the element after the current one
  T xv = 0;           // coordinate of the current element
  if (warp0 < M) xv = __ldg(coords + 3 * ldidx(conn + warp0 * NEN + ga) + gc);
  if (warp0 + nwarps < M) n1 = ldidx(conn + (warp0 + nwarps) * NEN + ga);
  T uv = 0;           // GEO: displacement of the current element
  if (GEO && warp0 < M) uv = __ldg(disp + 3 * ldidx(conn + warp0 * NEN + ga) + gc);
  for (long long e = warp0; e < M; e += nwarps) {
    xs[lane] = xv;
    if (GEO) us[lane] = uv;
    __syncwarp();
    if (GEO && e + nwarps < M) uv = __ldg(disp + 3 * n1 + gc);
    if (e + nwarps < M) xv = __ldg(coords + 3 * n1 + gc);
    if (e + 2 * nwarps < M) n1 = ldidx(conn + (e + 2 * nwarps) * NEN + ga);
    // ---- phase A
    if constexpr (GEO) {
      if (act) {
        T J[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, G[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int a = 0; a < NEN; ++a)
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) J[3 * i + k] += dn[a][i] * xs[3 * a + k], G[3 * i + k] += dn[a][i] * us[3 * a + k];
        T Ji[9], S[9];
        const T wa = fabs(inv3(J, Ji)) * wq;
        {
          T H[9];   // H[i][k] = du_k / dx_i
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) H[i * 3 + k] = Ji[i * 3] * G[k] + Ji[i * 3 + 1] * G[3 + k] + Ji[i * 3 + 2] * G[6 + k];
          const T tr = lam * (H[0] + H[4] + H[8]);
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) S[3 * i + k] = wa * (mu * (H[3 * i + k] + H[3 * k + i]) + (i == k ? tr : T(0)));
        }
        T gv[18], tv[18];
#pragma unroll
        for (int aa = 0; aa < 6; ++aa) {
          const int ah = aa < 4 ? aa + 6 : aa;
          const T d0 = h ? dn[ah][0] : dn[aa][0], d1 = h ? dn[ah][1] : dn[aa][1], d2 = h ? dn[ah][2] : dn[aa][2];
          const T g0 = Ji[0] * d0 + Ji[1] * d1 + Ji[2] * d2, g1 = Ji[3] * d0 + Ji[4] * d1 + Ji[5] * d2, g2 = Ji[6] * d0 + Ji[7] * d1 + Ji[8] * d2;
          gv[3 * aa] = g0, gv[3 * aa + 1] = g1, gv[3 * aa + 2] = g2;
#pragma unroll
          for (int i = 0; i < 3; ++i) tv[3 * aa + i] = S[3 * i] * g0 + S[3 * i + 1] * g1 + S[3 * i + 2] * g2;
        }
        const int nv = h ? 12 : 18;
        T* g = gs + q * C10W_GQ + h * 18;
        T* tq = ts + q * C10W_GQ + h * 18;
        if (sizeof(T) == 8) {
          double2* g2 = reinterpret_cast<double2*>(g);
          double2* t2 = reinterpret_cast<double2*>(tq);
#pragma unroll
          for (int k = 0; k < 9; ++k)
            if (2 * k < nv) {
              g2[k] = make_double2((double)gv[2 * k], (double)gv[2 * k + 1]);
              t2[k] = make_double2((double)tv[2 * k], (double)tv[2 * k + 1]);
            }
        } else {
#pragma unroll
          for (int k = 0; k < 18; ++k)
            if (k < nv) g[k] = gv[k], tq[k] = tv[k];
        }
      }
    } else if (act) {
      T J[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      T xr[30];
      if (sizeof(T) == 8) {  // the same address for the whole warp: 15 broadcast 128-bit loads
        const double2* xv2 = reinterpret_cast<const double2*>(xs);
#pragma unroll
        for (int k = 0; k < 15; ++k) {
          const double2 v = xv2[k];
          xr[2 * k] = (T)v.x, xr[2 * k + 1] = (T)v.y;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 30; ++k) xr[k] = xs[k];
      }
#pragma unroll
      for (int a = 0; a < NEN; ++a) {
#pragma unroll
        for (int i = 0; i < 3; ++i)
          J[3 * i] += dn[a][i] * xr[3 * a], J[3 * i + 1] += dn[a][i] * xr[3 * a + 1], J[3 * i + 2] += dn[a][i] * xr[3 * a + 2];
      }
      T Ji[9];
      const T det = inv3(J, Ji);
      if (h == 0) wd[q] = det * wq;
      // half 0: nodes 0..5 (18 values), half 1: nodes 6..9 (12 values, the last two slots unused) -- both ranges start 16-byte aligned
      T gv[18];
#pragma unroll
      for (int aa = 0; aa < 6; ++aa) {
        const int ah = aa < 4 ? aa + 6 : aa;   // half 1 has no nodes 4, 5: it repeats half 0's (discarded)
        const T d0 = h ? dn[ah][0] : dn[aa][0], d1 = h ? dn[ah][1] : dn[aa][1], d2 = h ? dn[ah][2] : dn[aa][2];
        gv[3 * aa] = Ji[0] * d0 + Ji[1] * d1 + Ji[2] * d2;
        gv[3 * aa + 1] = Ji[3] * d0 + Ji[4] * d1 + Ji[5] * d2;
        gv[3 * aa + 2] = Ji[6] * d0 + Ji[7] * d1 + Ji[8] * d2;
      }
      T* g = gs + q * C10W_GQ + h * 18;
      if (sizeof(T) == 8) {
        double2* g2 = reinterpret_cast<double2*>(g);
#pragma unroll
        for (int k = 0; k < 6; ++k) g2[k] = make_double2((double)gv[2 * k], (double)gv[2 * k + 1]);
        if (h == 0) {
#pragma unroll
          for (int k = 6; k < 9; ++k) g2[k] = make_double2((double)gv[2 * k], (double)gv[2 * k + 1]);
        }
      } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) g[k] = gv[k];
        if (h == 0) {
#pragma unroll
          for (int k = 12; k < 18; ++k) g[k] = gv[k];
        }
      }
    }
    __syncwarp();
    // ---- phase B
    T k0[9], k1[9];
    if constexpr (GEO) {
      T s0 = 0, s1 = 0;
#pragma unroll
      for (int p = 0; p < (NQ ? NQ : C10W_MAXQ); ++p) {
        if (!NQ && p >= nq) break;
        const T* g = gs + p * C10W_GQ;
        const T* tq = ts + p * C10W_GQ + 6 * t;
        T ar[6];
        if (sizeof(T) == 8) {
          const double2* v = reinterpret_cast<const double2*>(tq);
          const double2 v0 = v[0], v1 = v[1], v2 = v[2];
          ar[0] = (T)v0.x, ar[1] = (T)v0.y, ar[2] = (T)v1.x, ar[3] = (T)v1.y, ar[4] = (T)v2.x, ar[5] = (T)v2.y;
        } else {
#pragma unroll
          for (int k = 0; k < 6; ++k) ar[k] = tq[k];
        }
        const T gb0 = g[3 * b], gb1 = g[3 * b + 1], gb2 = g[3 * b + 2];
        s0 += ar[0] * gb0 + ar[1] * gb1 + ar[2] * gb2;
        s1 += ar[3] * gb0 + ar[4] * gb1 + ar[5] * gb2;
      }
#pragma unroll
      for (int k = 0; k < 9; ++k) k0[k] = k % 4 ? T(0) : s0, k1[k] = k % 4 ? T(0) : s1;
    } else {
    T S0[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, S1[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int p = 0; p < (NQ ? NQ : C10W_MAXQ); ++p) {
      if (!NQ && p >= nq) break;
      const T* g = gs + p * C10W_GQ;
      const T wt = wd[p];
      T ar[6];
      if (sizeof(T) == 8) {  // rows 2t, 2t+1: 48 bytes at a 16-byte aligned offset
        const double2* v = reinterpret_cast<const double2*>(g + 6 * t);
        const double2 v0 = v[0], v1 = v[1], v2 = v[2];
        ar[0] = (T)v0.x, ar[1] = (T)v0.y, ar[2] = (T)v1.x, ar[3] = (T)v1.y, ar[4] = (T)v2.x, ar[5] = (T)v2.y;
      } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) ar[k] = g[6 * t + k];
      }
      const T gb0 = g[3 * b], gb1 = g[3 * b + 1], gb2 = g[3 * b + 2];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const T u0 = wt * ar[i], u1 = wt * ar[3 + i];
        S0[3 * i] += u0 * gb0, S0[3 * i + 1] += u0 * gb1, S0[3 * i + 2] += u0 * gb2;
        S1[3 * i] += u1 * gb0, S1[3 * i + 1] += u1 * gb1, S1[3 * i + 2] += u1 * gb2;
      }
    }
    {
      const T tr0 = mu * (S0[0] + S0[4] + S0[8]), tr1 = mu * (S1[0] + S1[4] + S1[8]);
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          k0[3 * i + j] = lam * S0[3 * i + j] + mu * S0[3 * j + i] + (i == j ? tr0 : T(0));
          k1[3 * i + j] = lam * S1[3 * i + j] + mu * S1[3 * j + i] + (i == j ? tr1 : T(0));
        }
      // diagonal blocks: one triangle decides both (w g_i g_j and w g_j g_i round differently)
      if (b == a0) k0[3] = k0[1], k0[6] = k0[2], k0[7] = k0[5];
      if (b == a1) k1[3] = k1[1], k1[6] = k1[2], k1[7] = k1[5];
    }
    }
    // the previous tile must have been read out of shared memory before it is overwritten
    if (lane == 0) bulk_wait_read();
    __syncwarp();
    if (tile) {
      const bool up1 = b >= a1, mir0 = b > a0, mir1 = b > a1;
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          kt[(3 * a0 + i) * ND + 3 * b + j] = k0[3 * i + j];
          if (up1) kt[(3 * a1 + i) * ND + 3 * b + j] = k1[3 * i + j];
        }
      if (sizeof(T) == 8) {
        // mirror image: row 3b+j holds (K_{a0,b})^T | (K_{a1,b})^T in columns 6t..6t+5 -- 48 bytes, 16-byte aligned: three 128-bit
        // stores (as 8-byte stores the lanes of a warp hit only the even banks: 144 of the 409 shared-memory wavefronts per
        // element were these).  For b == a1 the second half lands on the diagonal block written above, with the same values
        // (symmetrised); for b == a0 the first half would, and the second half belongs to the lane of tile (t, a1): skipped.
        if (mir0) {
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            double2* row = reinterpret_cast<double2*>(kt + (3 * b + j) * ND + 6 * t);
            row[0] = make_double2((double)k0[j], (double)k0[3 + j]);
            row[1] = make_double2((double)k0[6 + j], (double)k1[j]);
            row[2] = make_double2((double)k1[3 + j], (double)k1[6 + j]);
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            if (mir0) kt[(3 * b + j) * ND + 3 * a0 + i] = k0[3 * i + j];
            if (mir1) kt[(3 * b + j) * ND + 3 * a1 + i] = k1[3 * i + j];
          }
      }
    }
    __syncwarp();
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      bulk_s2g(out + (size_t)e * ND * ND, kt, (unsigned)(ND * ND * sizeof(T)));
    }
  }
  if (lane == 0) bulk_wait_all();
}

template <typename T, typename I, int MINB, int NQ, bool GEO = false>
static int launch_c3d10_warp(const T* X, const I* C, long long M, SolidTab tab, int nq, T lam, T mu, T* O, cudaStream_t s,
                             const T* D = nullptr) {
  const size_t smem = sizeof(T) * (size_t)C10W_WARPS * (GEO ? C10W_PER_WARP_GEO : C10W_PER_WARP);
  auto kern = c3d10_K_warp_kernel<T, I, MINB, NQ, GEO>;
  FEMB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  FEMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C10W_WARPS * 32, smem));
  if (per_sm < 1) per_sm = 1;
  const int grid = (int)std::min<long long>((M + C10W_WARPS - 1) / C10W_WARPS, (long long)SMS * per_sm);
  kern<<<grid, C10W_WARPS * 32, smem, s>>>(X, C, M, tab, nq, lam, mu, O, D);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

// what 0: J [M,3,3]; 1: gradients [M,NEN,3]; 2: B [M,6,3*NEN] -- single point, one thread per element
template <typename T, typename I, int NEN>
__global__ void solid_point_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M, SolidTab tab, int what,
                                   T* __restrict__ out) {
  constexpr int ND = 3 * NEN;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    T J[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < NEN; ++a) {
      const long long n = ldidx(conn + e * NEN + a);
      T x[3] = {__ldg(coords + 3 * n), __ldg(coords + 3 * n + 1), __ldg(coords + 3 * n + 2)};
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const T d = (T)tab.dN[a * 3 + i];
#pragma unroll
        for (int k = 0; k < 3; ++k) J[i * 3 + k] += d * x[k];
      }
    }
    if (what == 0) {
      for (int k = 0; k < 9; ++k) out[e * 9 + k] = J[k];
      continue;
    }
    T Ji[9];
    inv3(J, Ji);
    if (what == 2)
      for (int k = 0; k < 6 * ND; ++k) out[e * 6 * ND + k] = 0;
    for (int a = 0; a < NEN; ++a) {
      T g[3];
#pragma unroll
      for (int i = 0; i < 3; ++i)
        g[i] = Ji[i * 3 + 0] * (T)tab.dN[a * 3 + 0] + Ji[i * 3 + 1] * (T)tab.dN[a * 3 + 1] + Ji[i * 3 + 2] * (T)tab.dN[a * 3 + 2];
      if (what == 1) {
        for (int i = 0; i < 3; ++i) out[(e * NEN + a) * 3 + i] = g[i];
      } else {
        T* B = out + e * 6 * ND;
        B[0 * ND + 3 * a + 0] = g[0];
        B[1 * ND + 3 * a + 1] = g[1];
        B[2 * ND + 3 * a + 2] = g[2];
        B[3 * ND + 3 * a + 0] = g[1];
        B[3 * ND + 3 * a + 1] = g[0];
        B[4 * ND + 3 * a + 1] = g[2];
        B[4 * ND + 3 * a + 2] = g[1];
        B[5 * ND + 3 * a + 0] = g[2];
        B[5 * ND + 3 * a + 2] = g[0];
      }
    }
  }
}

// Stress recovery (compute_c3d4_element_stress :905-939, compute_c3d10_element_stress :1127-1189, c3d8 :1696-1752,
// c3d6 :2570-2629): one thread per element walks the points.  With G = sum_a dN_a (x) u_a in natural coordinates the
// displacement gradient is H = J^-1 G, so B is never formed:  strain = (H00, H11, H22, H10+H01, H21+H12, H20+H02),
// stress = D strain, von Mises from the tensor.  single != 0: S[M,3,3] = sum_q w_q S_q and V[M] = sum_q w_q vm_q
// (the reference weights the von Mises values themselves); single == 0: S[nq,M,3,3], V[nq,M].
template <typename T, typename I, int NEN>
__global__ void solid_stress_kernel(const T* __restrict__ coords, const I* __restrict__ conn, long long M, const T* __restrict__ disp,
                                    SolidTab tab, int nq, int single, T lam, T mu, T* __restrict__ S, T* __restrict__ V) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    T sacc[6] = {0, 0, 0, 0, 0, 0}, vacc = 0;
    for (int q = 0; q < nq; ++q) {
      const double* dn = tab.dN + (size_t)q * NEN * 3;
      T J[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, G[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      for (int a = 0; a < NEN; ++a) {
        const long long n = ldidx(conn + e * NEN + a);
        const T x[3] = {__ldg(coords + 3 * n), __ldg(coords + 3 * n + 1), __ldg(coords + 3 * n + 2)};
        const T u[3] = {__ldg(disp + 3 * n), __ldg(disp + 3 * n + 1), __ldg(disp + 3 * n + 2)};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const T d = (T)dn[a * 3 + i];
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            J[i * 3 + k] += d * x[k];
            G[i * 3 + k] += d * u[k];
          }
        }
      }
      T Ji[9], H[9];
      inv3(J, Ji);
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) H[i * 3 + k] = Ji[i * 3] * G[k] + Ji[i * 3 + 1] * G[3 + k] + Ji[i * 3 + 2] * G[6 + k];
      const T exx = H[0], eyy = H[4], ezz = H[8], gxy = H[3] + H[1], gyz = H[7] + H[5], gzx = H[6] + H[2];
      const T tr = lam * (exx + eyy + ezz);
      const T s[6] = {tr + 2 * mu * exx, tr + 2 * mu * eyy, tr + 2 * mu * ezz, mu * gxy, mu * gyz, mu * gzx};
      const T d0 = s[0] - s[1], d1 = s[1] - s[2], d2 = s[2] - s[0];
      const T vm = sqrt((d0 * d0 + d1 * d1 + d2 * d2 + 6 * (s[3] * s[3] + s[4] * s[4] + s[5] * s[5])) / 2);
      if (single) {
        const T w = (T)tab.w[q];
#pragma unroll
        for (int k = 0; k < 6; ++k) sacc[k] += w * s[k];
        vacc += w * vm;
      } else {
        T* o = S + ((size_t)q * M + e) * 9;
        o[0] = s[0], o[1] = s[3], o[2] = s[5], o[3] = s[3], o[4] = s[1], o[5] = s[4], o[6] = s[5], o[7] = s[4], o[8] = s[2];
        V[(size_t)q * M + e] = vm;
      }
    }
    if (single) {
      T* o = S + e * 9;
      o[0] = sacc[0], o[1] = sacc[3], o[2] = sacc[5], o[3] = sacc[3], o[4] = sacc[1], o[5] = sacc[4], o[6] = sacc[5], o[7] = sacc[4],
      o[8] = sacc[2];
      V[e] = vacc;
    }
  }
}

// Natural-coordinate shape functions N[nen] and derivatives dN[nen][3], evaluated on the host in fp64.  The C3D10 / C3D8 /
// C3D6 derivative tables are the reference's as written; N follows the formulas in its comments (the reference has no
// code that evaluates N).  C3D20 / C3D15 are the standard serendipity hex (VTK/Abaqus order) and 15-node wedge: the
// reference's C3D20 table is wrong and raises, C3D15 is absent (SURVEY a12/a13) -- parity unpinned.
static void shape_c3d4(const double*, double* N, double* o) {
  const double t[12] = {-1, -1, -1, 1, 0, 0, 0, 1, 0, 0, 0, 1};
  memcpy(o, t, sizeof(t));
  N[0] = N[1] = N[2] = N[3] = 0.25;  // unused by the P1 paths
}
static void shape_c3d10(const double* p, double* N, double* o) {  // element.py:1042-1055, N from :941-962
  const double xi = p[0], eta = p[1], zeta = p[2], L3 = 1 - xi - eta - zeta, n3 = -4 * L3 + 1;
  const double t[30] = {4 * xi - 1, 0, 0, 0, 4 * eta - 1, 0, 0, 0, 4 * zeta - 1, n3, n3, n3, 4 * eta, 4 * xi, 0,
                        0, 4 * zeta, 4 * eta, 4 * zeta, 0, 4 * xi, 4 * (1 - 2 * xi - eta - zeta), -4 * xi, -4 * xi,
                        -4 * eta, 4 * (1 - xi - 2 * eta - zeta), -4 * eta, -4 * zeta, -4 * zeta, 4 * (1 - xi - eta - 2 * zeta)};
  memcpy(o, t, sizeof(t));
  const double L[4] = {xi, eta, zeta, L3};
  for (int a = 0; a < 4; ++a) N[a] = L[a] * (2 * L[a] - 1);
  N[4] = 4 * xi * eta, N[5] = 4 * eta * zeta, N[6] = 4 * zeta * xi, N[7] = 4 * xi * L3, N[8] = 4 * eta * L3, N[9] = 4 * zeta * L3;
}
static const int HSX[8] = {-1, 1, 1, -1, -1, 1, 1, -1}, HSY[8] = {-1, -1, 1, 1, -1, -1, 1, 1}, HSZ[8] = {-1, -1, -1, -1, 1, 1, 1, 1};
static void shape_c3d8(const double* p, double* N, double* o) {  // element.py:1617-1626, N from :1536-1554
  for (int a = 0; a < 8; ++a) {
    const double fx = 1 + HSX[a] * p[0], fy = 1 + HSY[a] * p[1], fz = 1 + HSZ[a] * p[2];
    o[3 * a + 0] = 0.125 * HSX[a] * fy * fz;
    o[3 * a + 1] = 0.125 * HSY[a] * fx * fz;
    o[3 * a + 2] = 0.125 * HSZ[a] * fx * fy;
    N[a] = 0.125 * fx * fy * fz;
  }
}
static void shape_c3d6(const double* p, double* N, double* o) {  // element.py:2499-2506
  const double r = p[0], s = p[1], t = p[2], L0 = 1 - r - s;
  const double v[18] = {-0.5 * (1 - t), -0.5 * (1 - t), -0.5 * L0, 0.5 * (1 - t), 0.0, -0.5 * r,
                        0.0, 0.5 * (1 - t), -0.5 * s, -0.5 * (1 + t), -0.5 * (1 + t), 0.5 * L0,
                        0.5 * (1 + t), 0.0, 0.5 * r, 0.0, 0.5 * (1 + t), 0.5 * s};
  memcpy(o, v, sizeof(v));
  N[0] = 0.5 * L0 * (1 - t), N[1] = 0.5 * r * (1 - t), N[2] = 0.5 * s * (1 - t);
  N[3] = 0.5 * L0 * (1 + t), N[4] = 0.5 * r * (1 + t), N[5] = 0.5 * s * (1 + t);
}
static void shape_c3d20(const double* p, double* N, double* o) {
  const double x = p[0], y = p[1], z = p[2];
  for (int a = 0; a < 8; ++a) {  // corners: (1+x xa)(1+y ya)(1+z za)(x xa + y ya + z za - 2)/8
    const double xa = HSX[a], ya = HSY[a], za = HSZ[a];
    const double fx = 1 + x * xa, fy = 1 + y * ya, fz = 1 + z * za, s = x * xa + y * ya + z * za - 2;
    N[a] = 0.125 * fx * fy * fz * s;
    o[3 * a + 0] = 0.125 * xa * fy * fz * (s + fx);
    o[3 * a + 1] = 0.125 * ya * fx * fz * (s + fy);
    o[3 * a + 2] = 0.125 * za * fx * fy * (s + fz);
  }
  // mid-edge nodes: 8-11 bottom ring (0-1,1-2,2-3,3-0), 12-15 top ring, 16-19 vertical (0-4 .. 3-7)
  static const int ring[4][2] = {{0, -1}, {1, 0}, {0, 1}, {-1, 0}};
  for (int k = 0; k < 4; ++k)
    for (int top = 0; top < 2; ++top) {
      const int a = 8 + 4 * top + k;
      const double xa = ring[k][0], ya = ring[k][1], za = top ? 1.0 : -1.0, fz = 1 + z * za;
      if (xa == 0) {  // varies quadratically in x
        const double fy = 1 + y * ya;
        N[a] = 0.25 * (1 - x * x) * fy * fz;
        o[3 * a + 0] = -0.5 * x * fy * fz, o[3 * a + 1] = 0.25 * (1 - x * x) * ya * fz, o[3 * a + 2] = 0.25 * (1 - x * x) * fy * za;
      } else {        // quadratic in y
        const double fx = 1 + x * xa;
        N[a] = 0.25 * (1 - y * y) * fx * fz;
        o[3 * a + 0] = 0.25 * (1 - y * y) * xa * fz, o[3 * a + 1] = -0.5 * y * fx * fz, o[3 * a + 2] = 0.25 * (1 - y * y) * fx * za;
      }
    }
  for (int k = 0; k < 4; ++k) {
    const int a = 16 + k;
    const double xa = HSX[k], ya = HSY[k], fx = 1 + x * xa, fy = 1 + y * ya;
    N[a] = 0.25 * (1 - z * z) * fx * fy;
    o[3 * a + 0] = 0.25 * (1 - z * z) * xa * fy, o[3 * a + 1] = 0.25 * (1 - z * z) * fx * ya, o[3 * a + 2] = -0.5 * z * fx * fy;
  }
}
static void shape_c3d15(const double* p, double* N, double* o) {
  const double r = p[0], s = p[1], t = p[2], q = 1 - t * t;
  const double L[3] = {1 - r - s, r, s}, dLr[3] = {-1, 1, 0}, dLs[3] = {-1, 0, 1};
  for (int i = 0; i < 3; ++i)
    for (int top = 0; top < 2; ++top) {  // corners: L/2 [(2L-1)(1 -+ t) - (1-t^2)]
      const int a = i + 3 * top;
      const double sg = top ? 1.0 : -1.0, h = 1 + sg * t, dl = 0.5 * ((4 * L[i] - 1) * h - q);
      N[a] = 0.5 * L[i] * ((2 * L[i] - 1) * h - q);
      o[3 * a + 0] = dl * dLr[i], o[3 * a + 1] = dl * dLs[i], o[3 * a + 2] = 0.5 * L[i] * ((2 * L[i] - 1) * sg + 2 * t);
    }
  static const int ed[3][2] = {{0, 1}, {1, 2}, {2, 0}};
  for (int k = 0; k < 3; ++k)
    for (int top = 0; top < 2; ++top) {  // triangle mid-edges 6-8 (bottom), 9-11 (top): 2 Li Lj (1 -+ t)
      const int a = 6 + 3 * top + k, i = ed[k][0], j = ed[k][1];
      const double sg = top ? 1.0 : -1.0, h = 1 + sg * t;
      N[a] = 2 * L[i] * L[j] * h;
      o[3 * a + 0] = 2 * (dLr[i] * L[j] + L[i] * dLr[j]) * h, o[3 * a + 1] = 2 * (dLs[i] * L[j] + L[i] * dLs[j]) * h;
      o[3 * a + 2] = 2 * L[i] * L[j] * sg;
    }
  for (int i = 0; i < 3; ++i) {  // vertical mid-edges 12-14: Li (1-t^2)
    const int a = 12 + i;
    N[a] = L[i] * q;
    o[3 * a + 0] = dLr[i] * q, o[3 * a + 1] = dLs[i] * q, o[3 * a + 2] = -2 * t * L[i];
  }
}

template <int NEN>
static void shape_of(const double* p, double* N, double* dN) {
  if (NEN == 4) shape_c3d4(p, N, dN);
  if (NEN == 10) shape_c3d10(p, N, dN);
  if (NEN == 8) shape_c3d8(p, N, dN);
  if (NEN == 6) shape_c3d6(p, N, dN);
  if (NEN == 20) shape_c3d20(p, N, dN);
  if (NEN == 15) shape_c3d15(p, N, dN);
}

// uploads [dN | w | N] for the caller's points; `tab` points into scratch memory owned by `scr`
template <int NEN>
static int upload_tables(const double* pts, int nq, Scratch& scr, cudaStream_t s, SolidTab& tab) {
  FEMB_CHECK_ARG(nq >= 1 && nq <= 64, "1 <= nq <= 64");
  double tabh[64 * 20 * 3 + 64 + 64 * 20];  // pageable source: cudaMemcpyAsync stages it before returning
  double* wh = tabh + (size_t)nq * NEN * 3;
  double* Nh = wh + nq;
  for (int q = 0; q < nq; ++q) {
    shape_of<NEN>(pts + 4 * q, Nh + (size_t)q * NEN, tabh + (size_t)q * NEN * 3);
    wh[q] = pts[4 * q + 3];
  }
  double* tabd;
  const size_t ntab = (size_t)nq * NEN * 4 + nq;
  FEMB_CUDA(scr.alloc(&tabd, ntab));
  FEMB_CUDA(cudaMemcpyAsync(tabd, tabh, ntab * sizeof(double), cudaMemcpyHostToDevice, s));
  tab = SolidTab{tabd, tabd + (size_t)nq * NEN * 3, tabd + (size_t)nq * NEN * 3 + nq};
  return FEMB_OK;
}

template <typename T, typename I, int NEN, int EPB>
static int launch_solid_K(const T* X, const I* C, long long M, SolidTab tab, int nq, int what, T lam, T mu, T* O, cudaStream_t s) {
  constexpr int ND = 3 * NEN, NPAIR = NEN * (NEN + 1) / 2;
  const size_t smem = sizeof(T) * ((size_t)EPB * ND * ND + (size_t)EPB * NEN * 3 + (size_t)EPB * nq * NEN * 3 + (size_t)EPB * nq +
                                   (size_t)EPB * nq * 9 + (size_t)nq * NEN * 4 + nq);
  FEMB_CHECK_ARG(smem <= 227 * 1024, "too many integration points for the shared-memory tile of this element type");
  auto kern = solid_K_kernel<T, I, NEN, EPB>;
  FEMB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int threads = EPB * NPAIR;
  threads = ((threads + 31) / 32) * 32;
  if (threads > 512) threads = 512;
  if (threads < 64) threads = 64;
  const int grid = (int)std::min<long long>((M + EPB - 1) / EPB, (long long)SMS * 16);
  kern<<<grid, threads, smem, s>>>(X, C, M, tab, nq, what, lam, mu, O);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

template <typename T, typename I, int NEN>
static int solid_dispatch(int what, const void* coords, const void* conn, long long M, const double* pts, int nq, double E, double nu,
                          void* out, cudaStream_t s) {
  if (M == 0) return FEMB_OK;
  Scratch scr(s);
  SolidTab tab;
  if (int rc = upload_tables<NEN>(pts, nq, scr, s, tab)) return rc;
  const T* X = static_cast<const T*>(coords);
  const I* C = static_cast<const I*>(conn);
  T* O = static_cast<T*>(out);
  if (what <= 2) {
    solid_point_kernel<T, I, NEN><<<grid_for(M, 128), 128, 0, s>>>(X, C, M, tab, what, O);
    FEMB_LAUNCH_CHECK();
    return FEMB_OK;
  }
  FEMB_CHECK_ARG(what >= 3 && what <= 6, "femb_solid: what in 0..6");
  FEMB_CHECK_ARG(what != 5 || NEN == 6, "what=5 is the C3D6 single-point mode");
  const int nqk = what == 5 ? 1 : nq;
  const double c = E / ((1 + nu) * (1 - 2 * nu));
  T lam = (T)(c * nu), mu = (T)(c * (1 - 2 * nu) / 2);
  if (what == 6) lam = (T)E, mu = 0;  // E carries rho
  // C3D10 stiffness with up to 16 points: the warp-per-element kernel (FEMB_SOLID_WARP=0: the CTA-phased kernel below; 2: two CTAs per SM; 5: point loop not unrolled)
  static const int warp_env = getenv("FEMB_SOLID_WARP") ? atoi(getenv("FEMB_SOLID_WARP")) : 3;
  if (NEN == 10 && what == 3 && nq <= C10W_MAXQ && warp_env > 0) {
    if (warp_env == 2) return launch_c3d10_warp<T, I, 2, 0>(X, C, M, tab, nq, lam, mu, O, s);
    if (warp_env == 5 || nq != 11) return launch_c3d10_warp<T, I, 3, 0>(X, C, M, tab, nq, lam, mu, O, s);   // 5: A/B of the unrolled form
    return launch_c3d10_warp<T, I, 3, 11>(X, C, M, tab, nq, lam, mu, O, s);
  }
  // elements per CTA: several small CTAs per SM overlap each other's barrier-separated phases
  static const int epb_env = getenv("FEMB_SOLID_EPB") ? atoi(getenv("FEMB_SOLID_EPB")) : 0;
  const int epb = epb_env ? epb_env : (NEN >= 20 ? 2 : 4);
  switch (epb) {
    case 1: return launch_solid_K<T, I, NEN, 1>(X, C, M, tab, nqk, what, lam, mu, O, s);
    case 2: return launch_solid_K<T, I, NEN, 2>(X, C, M, tab, nqk, what, lam, mu, O, s);
    case 8: if (NEN <= 10) return launch_solid_K<T, I, NEN, (NEN <= 10 ? 8 : 4)>(X, C, M, tab, nqk, what, lam, mu, O, s);
    default: return launch_solid_K<T, I, NEN, (NEN >= 20 ? 2 : 4)>(X, C, M, tab, nqk, what, lam, mu, O, s);
  }
}

template <typename T, typename I, int NEN>
static int stress_dispatch(const void* coords, const void* conn, long long M, const void* disp, const double* pts, int nq, double E,
                           double nu, int single, void* S, void* V, cudaStream_t s) {
  if (M == 0) return FEMB_OK;
  Scratch scr(s);
  SolidTab tab;
  if (int rc = upload_tables<NEN>(pts, nq, scr, s, tab)) return rc;
  const double c = E / ((1 + nu) * (1 - 2 * nu));
  solid_stress_kernel<T, I, NEN><<<grid_for(M, 128), 128, 0, s>>>(static_cast<const T*>(coords), static_cast<const I*>(conn), M,
                                                                   static_cast<const T*>(disp), tab, nq, single, (T)(c * nu),
                                                                   (T)(c * (1 - 2 * nu) / 2), static_cast<T*>(S), static_cast<T*>(V));
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

template <typename T, typename I>
static int geometric_dispatch(int kind, const void* coords, const void* conn, long long M, const void* disp, const double* pts, int nq,
                              double E, double nu, void* out, cudaStream_t s) {
  if (M == 0) return FEMB_OK;
  const double c = E / ((1 + nu) * (1 - 2 * nu));
  const T lam = (T)(c * nu), mu = (T)(c * (1 - 2 * nu) / 2);
  const T* X = static_cast<const T*>(coords);
  const I* C = static_cast<const I*>(conn);
  const T* D = static_cast<const T*>(disp);
  T* O = static_cast<T*>(out);
  if (kind == FEMB_C3D4) {
    c3d4_geometric_kernel<T, I><<<grid_for(M, 128), 128, 0, s>>>(X, C, M, D, lam, mu, O);
    FEMB_LAUNCH_CHECK();
    return FEMB_OK;
  }
  Scratch scr(s);
  SolidTab tab;
  if (int rc = upload_tables<10>(pts, nq, scr, s, tab)) return rc;
  if (nq == 14) return launch_c3d10_warp<T, I, 3, 14, true>(X, C, M, tab, nq, lam, mu, O, s, D);   // the default degree-5 rule
  return launch_c3d10_warp<T, I, 3, 0, true>(X, C, M, tab, nq, lam, mu, O, s, D);
}

template <typename I>
__global__ void to_c3d4_kernel(const I* __restrict__ conn, long long M, int nen, int k, const int* __restrict__ table, long long* __restrict__ out) {
  const long long total = M * k * 4;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long e = t / (k * 4);
    const int r = (int)(t - e * k * 4);
    out[t] = ldidx(conn + e * nen + table[r]);
  }
}

}  // namespace femb

using namespace femb;

#define DISPATCH_TI(fn, fp, ib, ...)                                        \
  ((fp) == 8 ? ((ib) == 8 ? fn<double, long long>(__VA_ARGS__) : fn<double, int>(__VA_ARGS__)) \
             : ((ib) == 8 ? fn<float, long long>(__VA_ARGS__) : fn<float, int>(__VA_ARGS__)))

extern "C" int femb_c3d4(int what, const void* coords, int fp, const void* conn, int ib, int64_t M, double E, double nu, void* out,
                         int32_t* flag, femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (ib == 4 || ib == 8), "fp in {4,8}, ib in {4,8}");
  FEMB_CHECK_ARG(M >= 0, "M >= 0");
  return DISPATCH_TI(c3d4_dispatch, fp, ib, what, coords, conn, M, E, nu, out, flag, as_stream(stream));
}

template <typename T, typename I>
static int volumes_dispatch(int kind, const void* coords, const void* conn, long long M, int stride, void* vol, cudaStream_t s) {
  if (M == 0) return FEMB_OK;
  const int grid = grid_for(M, 128);
  const T* X = static_cast<const T*>(coords);
  const I* C = static_cast<const I*>(conn);
  if (kind == FEMB_C3D4 || kind == FEMB_C3D10) volumes_kernel<T, I, 4><<<grid, 128, 0, s>>>(X, C, M, stride, (T*)vol);
  else if (kind == FEMB_C3D8) volumes_kernel<T, I, 8><<<grid, 128, 0, s>>>(X, C, M, stride, (T*)vol);
  else if (kind == FEMB_C3D6) volumes_kernel<T, I, 6><<<grid, 128, 0, s>>>(X, C, M, stride, (T*)vol);
  else {
    set_error("femb_elem_volumes: kind must be C3D4/C3D10/C3D8/C3D6");
    return FEMB_ERR_ARG;
  }
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_elem_volumes(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, int conn_stride, void* vol,
                                 femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (ib == 4 || ib == 8), "fp in {4,8}, ib in {4,8}");
  return DISPATCH_TI(volumes_dispatch, fp, ib, kind, coords, conn, M, conn_stride, vol, as_stream(stream));
}

template <typename T, typename I>
static int solid_dispatch_kind(int kind, int what, const void* coords, const void* conn, long long M, const double* pts, int nq, double E,
                               double nu, void* out, cudaStream_t s) {
  switch (kind) {
    case FEMB_C3D10: return solid_dispatch<T, I, 10>(what, coords, conn, M, pts, nq, E, nu, out, s);
    case FEMB_C3D8: return solid_dispatch<T, I, 8>(what, coords, conn, M, pts, nq, E, nu, out, s);
    case FEMB_C3D6: return solid_dispatch<T, I, 6>(what, coords, conn, M, pts, nq, E, nu, out, s);
    case FEMB_C3D20: return solid_dispatch<T, I, 20>(what, coords, conn, M, pts, nq, E, nu, out, s);
    case FEMB_C3D15: return solid_dispatch<T, I, 15>(what, coords, conn, M, pts, nq, E, nu, out, s);
  }
  set_error("femb_solid: kind must be C3D10/C3D8/C3D6/C3D20/C3D15");
  return FEMB_ERR_ARG;
}

template <typename T, typename I>
static int stress_dispatch_kind(int kind, const void* coords, const void* conn, long long M, const void* disp, const double* pts, int nq,
                                double E, double nu, int single, void* S, void* V, cudaStream_t s) {
  switch (kind) {
    case FEMB_C3D4: return stress_dispatch<T, I, 4>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
    case FEMB_C3D10: return stress_dispatch<T, I, 10>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
    case FEMB_C3D8: return stress_dispatch<T, I, 8>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
    case FEMB_C3D6: return stress_dispatch<T, I, 6>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
    case FEMB_C3D20: return stress_dispatch<T, I, 20>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
    case FEMB_C3D15: return stress_dispatch<T, I, 15>(coords, conn, M, disp, pts, nq, E, nu, single, S, V, s);
  }
  set_error("femb_solid_stress: kind must be C3D4/C3D10/C3D8/C3D6/C3D20/C3D15");
  return FEMB_ERR_ARG;
}

extern "C" int femb_solid_stress(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, const void* disp,
                                 const double* pts_host, int nq, double E, double nu, int single, void* stress, void* vm,
                                 femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (ib == 4 || ib == 8), "fp in {4,8}, ib in {4,8}");
  FEMB_CHECK_ARG(pts_host != nullptr, "pts_host");
  return DISPATCH_TI(stress_dispatch_kind, fp, ib, kind, coords, conn, M, disp, pts_host, nq, E, nu, single, stress, vm,
                     as_stream(stream));
}

extern "C" int femb_solid(int kind, int what, const void* coords, int fp, const void* conn, int ib, int64_t M, const double* pts_host,
                          int nq, double E, double nu, void* out, femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (ib == 4 || ib == 8), "fp in {4,8}, ib in {4,8}");
  FEMB_CHECK_ARG(pts_host != nullptr, "pts_host");
  return DISPATCH_TI(solid_dispatch_kind, fp, ib, kind, what, coords, conn, M, pts_host, nq, E, nu, out, as_stream(stream));
}

extern "C" int femb_solid_geometric(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, const void* disp,
                                    const double* pts_host, int nq, double E, double nu, void* out, femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (ib == 4 || ib == 8), "fp in {4,8}, ib in {4,8}");
  FEMB_CHECK_ARG(kind == FEMB_C3D4 || kind == FEMB_C3D10, "femb_solid_geometric: kind must be C3D4 or C3D10");
  FEMB_CHECK_ARG(M >= 0, "M >= 0");
  FEMB_CHECK_ARG(kind == FEMB_C3D4 || (pts_host != nullptr && nq >= 1 && nq <= C10W_MAXQ),
                 "femb_solid_geometric: C3D10 needs pts_host [nq,4] with 1 <= nq <= 16");
  FEMB_CHECK_ARG(M == 0 || (coords && conn && disp && out), "femb_solid_geometric: coords, conn, disp and out must be non-null");
  return DISPATCH_TI(geometric_dispatch, fp, ib, kind, coords, conn, M, disp, pts_host, nq, E, nu, out, as_stream(stream));
}

extern "C" int femb_default_points(int kind, double* p) {
  // fp32-rounded 1/sqrt(3) (quirk q1: element.py:2460-2463, shell.py:657-663)
  const double g32 = (double)(1.0f / sqrtf(3.0f));
  if (kind == FEMB_C3D10) {  // element.py:995-1024
    static const double pts[11][4] = {{.25, .25, .25, .1}, {.1, .1, .1, .05}, {.1, .1, .7, .05}, {.1, .7, .1, .05},
                                      {.7, .1, .1, .05},   {.1, .4, .4, .03}, {.4, .1, .4, .03}, {.4, .4, .1, .03},
                                      {.3, .3, .3, .02},   {.2, .2, .6, .02}, {.2, .6, .2, .02}};
    memcpy(p, pts, sizeof(pts));
    return 11;
  }
  if (kind == FEMB_C3D8) {  // element.py:1583-1599, exact in fp64
    const double g = 1.0 / sqrt(3.0);
    int q = 0;
    for (int a = -1; a <= 1; a += 2)
      for (int b = -1; b <= 1; b += 2)
        for (int c = -1; c <= 1; c += 2, ++q) {
          p[4 * q] = a * g, p[4 * q + 1] = b * g, p[4 * q + 2] = c * g, p[4 * q + 3] = 1.0;
        }
    return 8;
  }
  if (kind == FEMB_C3D6) {  // element.py:2448-2480
    const double tri[3][2] = {{1.0 / 6, 1.0 / 6}, {2.0 / 3, 1.0 / 6}, {1.0 / 6, 2.0 / 3}};
    int q = 0;
    for (int i = 0; i < 3; ++i)
      for (int j = -1; j <= 1; j += 2, ++q) {
        p[4 * q] = tri[i][0], p[4 * q + 1] = tri[i][1], p[4 * q + 2] = j * g32, p[4 * q + 3] = 1.0 / 3;
      }
    return 6;
  }
  if (kind == FEMB_C3D20) {  // element.py:1898-1919: xi slowest, +-sqrt(3/5) rounded to fp32 (q1), weights in fp64
    const double g = (double)sqrtf((float)(3.0 / 5.0)), gp[3] = {-g, 0.0, g}, gw[3] = {5.0 / 9.0, 8.0 / 9.0, 5.0 / 9.0};
    int q = 0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k, ++q) p[4 * q] = gp[i], p[4 * q + 1] = gp[j], p[4 * q + 2] = gp[k], p[4 * q + 3] = gw[i] * gw[j] * gw[k];
    return 27;
  }
  if (kind == FEMB_C3D15) {  // not in the reference: 3-point triangle rule x 3-point Gauss, exact constants
    const double tri[3][2] = {{1.0 / 6, 1.0 / 6}, {2.0 / 3, 1.0 / 6}, {1.0 / 6, 2.0 / 3}};
    const double g = sqrt(0.6), gp[3] = {-g, 0.0, g}, gw[3] = {5.0 / 9.0, 8.0 / 9.0, 5.0 / 9.0};
    int q = 0;
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k, ++q) p[4 * q] = tri[i][0], p[4 * q + 1] = tri[i][1], p[4 * q + 2] = gp[k], p[4 * q + 3] = gw[k] / 6;
    return 9;
  }
  if (kind == FEMB_S4) {  // shell.py:651-672
    const double s[4][2] = {{1, -1}, {1, 1}, {-1, 1}, {-1, -1}};
    for (int q = 0; q < 4; ++q) p[4 * q] = s[q][0] * g32, p[4 * q + 1] = s[q][1] * g32, p[4 * q + 2] = 0, p[4 * q + 3] = 1.0;
    return 4;
  }
  set_error("femb_default_points: unknown kind");
  return -1;
}

extern "C" int femb_shape_tables(int kind, const double* pts_host, int nq, double* N_host, double* dN_host) {
  FEMB_CHECK_ARG(pts_host && N_host && dN_host && nq >= 0, "pts_host, N_host, dN_host, nq >= 0");
  for (int q = 0; q < nq; ++q) {
    const double* p = pts_host + 4 * q;
    switch (kind) {
      case FEMB_C3D4: shape_of<4>(p, N_host + q * 4, dN_host + q * 12); break;
      case FEMB_C3D10: shape_of<10>(p, N_host + q * 10, dN_host + q * 30); break;
      case FEMB_C3D8: shape_of<8>(p, N_host + q * 8, dN_host + q * 24); break;
      case FEMB_C3D6: shape_of<6>(p, N_host + q * 6, dN_host + q * 18); break;
      case FEMB_C3D20: shape_of<20>(p, N_host + q * 20, dN_host + q * 60); break;
      case FEMB_C3D15: shape_of<15>(p, N_host + q * 15, dN_host + q * 45); break;
      default: set_error("femb_shape_tables: unknown kind"); return FEMB_ERR_ARG;
    }
  }
  return FEMB_OK;
}

namespace femb {
// what 0: Voigt [M,6] (xx,yy,zz,xy,yz,zx) -> tensor [M,3,3] (element.py:308-330); 1: tensor [M,3,3] -> von Mises [M] (:332-353)
template <typename T>
__global__ void stress_helper_kernel(const T* __restrict__ in, long long M, int what, T* __restrict__ out) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < M; e += (long long)gridDim.x * blockDim.x) {
    if (what == 0) {
      const T* v = in + e * 6;
      T* o = out + e * 9;
      o[0] = v[0], o[1] = v[3], o[2] = v[5], o[3] = v[3], o[4] = v[1], o[5] = v[4], o[6] = v[5], o[7] = v[4], o[8] = v[2];
    } else {
      const T* s = in + e * 9;
      const T d0 = s[0] - s[4], d1 = s[4] - s[8], d2 = s[8] - s[0];
      out[e] = sqrt((d0 * d0 + d1 * d1 + d2 * d2 + 6 * (s[1] * s[1] + s[5] * s[5] + s[2] * s[2])) / 2);
    }
  }
}
}  // namespace femb

extern "C" int femb_stress_helper(int what, const void* in, int fp, int64_t M, void* out, femb_stream stream) {
  FEMB_CHECK_ARG((fp == 4 || fp == 8) && (what == 0 || what == 1) && M >= 0, "fp in {4,8}, what in {0,1}, M >= 0");
  if (M == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  if (fp == 8) stress_helper_kernel<double><<<grid_for(M, 256), 256, 0, s>>>((const double*)in, M, what, (double*)out);
  else stress_helper_kernel<float><<<grid_for(M, 256), 256, 0, s>>>((const float*)in, M, what, (float*)out);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}

extern "C" int femb_mass_points(int kind, double* p) {
  const double g = sqrt(0.6), gp[3] = {-g, 0.0, g}, gw[3] = {5.0 / 9.0, 8.0 / 9.0, 5.0 / 9.0};
  if (kind == FEMB_C3D10) {  // degree-5 14-point rule: orbits (a,a,a,1-3a) x 2 and (b,b,1/2-b,1/2-b)
    const double a[2] = {0.3108859192633006098, 0.09273525031089122640}, wa[2] = {0.01878132095300264180, 0.01224884051939365826};
    const double b = 0.04550370412564964949, wb = 0.007091003462846911073, h = 0.5 - b;
    int q = 0;
    for (int o = 0; o < 2; ++o) {
      const double c = 1 - 3 * a[o];
      const double pt[4][3] = {{a[o], a[o], a[o]}, {c, a[o], a[o]}, {a[o], c, a[o]}, {a[o], a[o], c}};
      for (int k = 0; k < 4; ++k, ++q) p[4 * q] = pt[k][0], p[4 * q + 1] = pt[k][1], p[4 * q + 2] = pt[k][2], p[4 * q + 3] = wa[o];
    }
    const double pt[6][3] = {{b, b, h}, {b, h, b}, {h, b, b}, {b, h, h}, {h, b, h}, {h, h, b}};
    for (int k = 0; k < 6; ++k, ++q) p[4 * q] = pt[k][0], p[4 * q + 1] = pt[k][1], p[4 * q + 2] = pt[k][2], p[4 * q + 3] = wb;
    return 14;
  }
  if (kind == FEMB_C3D8 || kind == FEMB_C3D20) {  // 3x3x3 Gauss
    int q = 0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k, ++q) p[4 * q] = gp[i], p[4 * q + 1] = gp[j], p[4 * q + 2] = gp[k], p[4 * q + 3] = gw[i] * gw[j] * gw[k];
    return 27;
  }
  if (kind == FEMB_C3D6 || kind == FEMB_C3D15) {  // degree-4 6-point triangle rule x 3-point Gauss
    const double ta = 0.4459484909159648863, twa = 0.1116907948390057328, tb = 0.09157621350977074346, twb = 0.05497587182766093382;
    const double tri[6][3] = {{ta, ta, twa}, {1 - 2 * ta, ta, twa}, {ta, 1 - 2 * ta, twa}, {tb, tb, twb}, {1 - 2 * tb, tb, twb}, {tb, 1 - 2 * tb, twb}};
    int q = 0;
    for (int i = 0; i < 6; ++i)
      for (int k = 0; k < 3; ++k, ++q) p[4 * q] = tri[i][0], p[4 * q + 1] = tri[i][1], p[4 * q + 2] = gp[k], p[4 * q + 3] = tri[i][2] * gw[k];
    return 18;
  }
  set_error("femb_mass_points: kind must be C3D10/C3D8/C3D6/C3D20/C3D15");
  return -1;
}

extern "C" int femb_to_c3d4(int kind, const void* conn, int ib, int64_t M, int64_t* out, femb_stream stream) {
  static const int t10[32] = {0, 4, 6, 7, 4, 1, 5, 8, 6, 5, 2, 9, 7, 8, 9, 3, 4, 6, 7, 5, 6, 7, 9, 5, 4, 7, 8, 5, 5, 8, 7, 9};  // :977-986
  static const int t8[24] = {0, 1, 3, 4, 1, 2, 3, 6, 1, 3, 4, 5, 3, 4, 5, 7, 3, 5, 6, 7, 3, 5, 6, 2};                          // :1567-1574
  static const int t6[12] = {0, 1, 2, 3, 1, 2, 3, 5, 1, 3, 4, 5};                                                              // :2435-2439
  static const int t20[96] = {0,  8,  12, 19, 8,  1,  13, 9,  9,  1,  2,  10, 10, 2,  14, 11, 11, 2,  3,  15, 15, 3,  19, 0,   // :1864-1889
                              12, 4,  16, 19, 16, 4,  5,  17, 17, 5,  13, 18, 18, 5,  6,  14, 14, 6,  18, 7,  19, 7,  15, 11,
                              8,  9,  10, 11, 8,  10, 11, 12, 12, 13, 14, 15, 16, 17, 18, 19, 0,  8,  9,  10, 0,  10, 11, 12,
                              1,  9,  10, 13, 1,  13, 14, 17, 2,  10, 14, 15, 3,  11, 15, 19, 4,  12, 16, 19, 5,  13, 17, 18};
  const int* tab;
  int k, nen;
  if (kind == FEMB_C3D10) tab = t10, k = 8, nen = 10;
  else if (kind == FEMB_C3D8) tab = t8, k = 6, nen = 8;
  else if (kind == FEMB_C3D6) tab = t6, k = 3, nen = 6;
  else if (kind == FEMB_C3D20) tab = t20, k = 24, nen = 20;
  else {
    set_error("femb_to_c3d4: kind must be C3D10/C3D8/C3D6/C3D20");
    return FEMB_ERR_ARG;
  }
  if (M == 0) return FEMB_OK;
  cudaStream_t s = as_stream(stream);
  Scratch scr(s);
  int* dtab;
  FEMB_CUDA(scr.alloc(&dtab, (size_t)k * 4));
  FEMB_CUDA(cudaMemcpyAsync(dtab, tab, sizeof(int) * k * 4, cudaMemcpyHostToDevice, s));
  const int grid = grid_for(M * k * 4, 256);
  if (ib == 8) to_c3d4_kernel<long long><<<grid, 256, 0, s>>>((const long long*)conn, M, nen, k, dtab, (long long*)out);
  else to_c3d4_kernel<int><<<grid, 256, 0, s>>>((const int*)conn, M, nen, k, dtab, (long long*)out);
  FEMB_LAUNCH_CHECK();
  return FEMB_OK;
}
