// Multi-GPU conjugate gradient over NVLink peer memory (one process per GPU, rows partitioned, SURVEY.md section 8e).
//
// The reference has no distributed code.  Each rank owns a block of rows (local numbering [owned, interior rows first |
// padding to a cache line | ghost]) and keeps its search direction p in a cudaIpc-shared "symmetric" buffer.  One iteration
// of CG / Jacobi-PCG is TWO kernels in one CUDA graph (merged-reduction loop, default):
//   m1    SpMV on the owned rows -- scalar CSR: the TMA-pipelined row tiles of spmv_dev.cuh; 3-dof operators: 3x3 block-CSR,
//         warp per block row -- interior rows first; a CTA (warp) waits for halo flag A of its neighbours only before its first
//         boundary tile (row).  Partials of p.Ap, z.Ap, (M^-1 Ap).Ap; the last CTA sends the rank's sums to every rank as
//         "LL words": (epoch << 32 | half of a double) in ONE 8-byte store, so value and flag arrive together (no system
//         fence, no separate flag)
//   m2    waits for the words of all ranks, sums them in rank order (identical on every rank), alpha, beta from the recurrence,
//         u += alpha p, r -= alpha Ap, p = z + beta p in one pass; the thread that updates a boundary row stores the new value
//         straight into the ghost slots of the neighbours that need it (st.global on mapped peer pointers through NVSwitch);
//         the last CTA raises flag A on the neighbours and sends the exactly summed r.z (consumed one SpMV later: that is where
//         the reference's convergence test is applied, so the returned state is the reference's at its break)
// FEMB_DIST_CLASSIC=1 keeps round 1's three-kernel loop (k1 SpMV + p.Ap, k2 update + r.r, k3 direction + halo push; slot stores,
// system fence and flag stores for the two waited all-reduces) for scalar CSR without a preconditioner, for A/B runs.
// There is no NCCL call and no host involvement inside the loop: the "collectives" are peer stores plus epochs.
// All spin loops carry a timeout so a lost rank turns into an error, not a hang.  Lessons measured on 8 B200 (DESIGN.md 3.5):
// let ONE thread per CTA read the reduction slots (every thread doing it made the slot line an L2 hot spot worth 17 us per
// kernel); read x through the read-only path (plain loads cost 17 %), which is safe because ghosts start on their own
// 128-byte line and are first touched after flag A while L1 is flushed at every launch; a single persistent cooperative
// kernel with software grid barriers (dist_cg_persistent_kernel, FEMB_DIST_PERSISTENT=1) is slower than launch boundaries; a
// stop flag must only ever be raised by the LAST CTA of a kernel (profiles/r02_race_note.md).
#include <cstdlib>

#include "spmv_dev.cuh"

namespace femb {

constexpr int MAXP = 16;
constexpr long long SPIN_TIMEOUT_CYCLES = 4000000000ll;  // ~2 s at 2 GHz

// layout of every rank's symmetric buffer (identical on all ranks)
struct SymHeader {
  volatile long long flagA[MAXP];  // halo arrived from rank q (epoch)
  volatile long long flagB[MAXP];  // p.Ap partial of rank q arrived
  volatile long long flagC[MAXP];  // r.r partial of rank q arrived
  volatile double redB[MAXP];
  volatile double redC[MAXP];
  volatile double red2[2][4][MAXP];  // (previous layout of the merged loop's slots; kept so the header size is unchanged)
  double pad[MAXP];
  // merged-reduction CG all-reduce, "LL" style: ll[epoch parity][source rank][word].  A word is (epoch << 32) | half of a
  // double, written with ONE 8-byte store, so data and flag arrive together: no fence, no separate flag store, and the
  // receiver knows a value is complete the moment it sees the epoch.  Words 0..5 = lo/hi of p.Ap, r.Ap, Ap.Ap (epoch B),
  // words 6..7 = lo/hi of the exactly summed r.r (epoch C).
  volatile unsigned long long ll[2][MAXP][8];
  volatile long long flagS[MAXP];  // start barrier of the iteration graph (rank q has finished its setup and enqueued its loop)
  long long pad2[MAXP];
};
static_assert(sizeof(SymHeader) % 256 == 0, "header keeps p 256-byte aligned");

struct DistState {
  double rs_old, rs_new, pAp, alpha, beta;
  int it, stop, status, iterations;
  long long epochA, epochB, epochC;
  unsigned int ticket_push, ticket1, ticket2, ticket3;
  long long* trace;  // optional [TRACE_ITERS][12] globaltimer stamps (FEMB_DIST_TRACE=1)
};

constexpr int TRACE_ITERS = 64;
__device__ __forceinline__ void trace_stamp(DistState* st, int slot) {
  if (st->trace && st->it < TRACE_ITERS) {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    st->trace[st->it * 12 + slot] = t;
  }
}

struct Peers {
  SymHeader* hdr[MAXP];  // every rank's header as mapped in this process (own included)
  int rank, P;
  int nnbr;
  int nbr[MAXP];
  int send_ptr[MAXP + 1];      // prefix into send_idx per neighbour
  long long ghost_off[MAXP];   // where my block starts inside neighbour's p (n_owned_q + recv_off_q[rank]), in doubles
};

__device__ __forceinline__ double* sym_p(SymHeader* h) { return reinterpret_cast<double*>(h + 1); }

__device__ __forceinline__ bool spin_until(volatile long long* flag, long long expect, DistState* st) {
  const long long t0 = clock64();
  while (*flag < expect) {
    if (clock64() - t0 > SPIN_TIMEOUT_CYCLES) {
      st->stop = 3, st->status = 3;
      return false;
    }
  }
  return true;
}

// block-level wait: thread 0 polls the listed ranks' flags in MY header, everyone else parks on the barrier
__device__ __forceinline__ void wait_flags(volatile long long* flags, const int* ranks, int count, long long expect, DistState* st) {
  if (threadIdx.x < count) spin_until(flags + ranks[threadIdx.x], expect, st);  // one lane per flag: the polls overlap
  __syncthreads();
}

// ---- push: p boundary -> neighbours' ghost slots, then flag A --------------------------------------------------------
__global__ void __launch_bounds__(256) dist_push_kernel(Peers pe, const int* __restrict__ send_idx, DistState* st) {
  if (st->stop) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 0);
  const double* p = sym_p(pe.hdr[pe.rank]);
  const int total = pe.send_ptr[pe.nnbr];
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    int k = 0;
    while (t >= pe.send_ptr[k + 1]) ++k;
    double* dst = sym_p(pe.hdr[pe.nbr[k]]) + pe.ghost_off[k];
    dst[t - pe.send_ptr[k]] = p[send_idx[t]];
  }
  __threadfence_system();
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&st->ticket_push, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last && threadIdx.x == 0) {
    st->ticket_push = 0;
    const long long e = st->epochA + 1;
    st->epochA = e;
    __threadfence_system();
    for (int k = 0; k < pe.nnbr; ++k) pe.hdr[pe.nbr[k]]->flagA[pe.rank] = e;
    trace_stamp(st, 1);
  }
}

struct GraphHaloWaiter {
  SymHeader* me;
  const int* nbr;
  int nnbr;
  long long epoch;
  DistState* st;
  __device__ __forceinline__ void operator()() const { wait_flags(me->flagA, nbr, nnbr, epoch, st); }
};

// ---- k1: SpMV on owned rows + p.Ap partial -> everyone ---------------------------------------------------------------
template <int LR, bool FUSED, bool NC>
__global__ void __launch_bounds__(TMA_THREADS) dist_spmv_kernel(Peers pe, long long n_owned, long long nnz, const int* __restrict__ crow,
                                                                const int* __restrict__ col, const double* __restrict__ val,
                                                                double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                                double* __restrict__ partial, DistState* st, long long n_interior) {
  if (st->stop) return;
  SymHeader* me = pe.hdr[pe.rank];
  if (FUSED && blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 2), trace_stamp(st, 3);
  __shared__ int nbr[MAXP];
  if (threadIdx.x < MAXP) nbr[threadIdx.x] = pe.nbr[threadIdx.x];
  __syncthreads();
  const double* x = sym_p(me);
  // TMA-pipelined row tiles; interior tiles need no ghost entry, so a CTA waits for the halo only when it reaches its
  // first boundary tile.  x is read with plain (L1-cached, L2-coherent) loads: peers write its ghost part.
  const GraphHaloWaiter hw{me, nbr, pe.nnbr, st->epochA, st};
  const double dot = spmv_tma_rows<LR, NC, TMA_THREADS, TMA_STAGES, TMA_CAP, GraphHaloWaiter>(
      n_owned, nnz, crow, col, val, x, y, mask, false, FUSED, pe.nnbr > 0 ? n_interior : 0x7fffffffffffffffll, hw);
  if (st->stop == 3) return;
  if (!FUSED) return;
  const double t = block_sum<TMA_THREADS>(dot);
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
    for (int k = threadIdx.x; k < (int)gridDim.x; k += TMA_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<TMA_THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket1 = 0;
      const long long e = st->epochB + 1;
      st->epochB = e;
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->redB[pe.rank] = a;
      __threadfence_system();
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->flagB[pe.rank] = e;
      trace_stamp(st, 4);
    }
  }
}

constexpr int DV_THREADS = 256;

__device__ __forceinline__ double sum_slots_serial(volatile double* red, int P) {
  double a = 0.0;
  for (int q = 0; q < P; ++q) a += red[q];  // rank order: identical result on every rank
  return a;
}
// block-uniform: ONE thread reads the P slots and broadcasts through shared memory.  (Every thread reading them turns the
// 64-byte slot line into an L2 hot spot: 1184 CTAs x 8 warps x P requests cost ~17 us per kernel at P = 8.)
__device__ __forceinline__ double sum_slots(volatile double* red, int P) {
  __shared__ double bc;
  if (threadIdx.x == 0) bc = sum_slots_serial(red, P);
  __syncthreads();
  const double v = bc;
  __syncthreads();
  return v;
}

__device__ __forceinline__ void ll_store(volatile unsigned long long* w, double v, int half, long long epoch) {
  const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
  const unsigned long long part = half ? (bits >> 32) : (bits & 0xffffffffull);
  *w = ((unsigned long long)(unsigned)epoch << 32) | part;
}
// spin until the word carries `epoch`; returns its 32 data bits
__device__ __forceinline__ unsigned ll_wait(volatile unsigned long long* w, long long epoch, DistState* st) {
  const long long t0 = clock64();
  unsigned long long v;
  while ((unsigned)((v = *w) >> 32) != (unsigned)epoch) {
    if (clock64() - t0 > SPIN_TIMEOUT_CYCLES) {
      st->stop = 3, st->status = 3;
      break;
    }
  }
  return (unsigned)v;
}

// ---- k2: u += alpha p ; r -= alpha Ap ; r.r partial -> everyone -------------------------------------------------------
__global__ void __launch_bounds__(DV_THREADS) dist_update_kernel(Peers pe, long long n, double* __restrict__ u, double* __restrict__ r,
                                                                 const double* __restrict__ Ap, double* __restrict__ partial, DistState* st,
                                                                 double eps, int guards) {
  if (st->stop) return;
  SymHeader* me = pe.hdr[pe.rank];
  __shared__ int all[MAXP];
  if (threadIdx.x < MAXP) all[threadIdx.x] = threadIdx.x;
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 5);
  wait_flags(me->flagB, all, pe.P, st->epochB, st);
  {  // block-uniform (one read per CTA): CTA 0 may raise the flag below while this CTA is still on its way here
    __shared__ int stop_now;
    if (threadIdx.x == 0) stop_now = st->stop;
    __syncthreads();
    if (stop_now) return;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 6);
  const double pAp = sum_slots(me->redB, pe.P);
  const double alpha = st->rs_old / (pAp + eps);
  if (guards && (fabs(pAp) < eps || pAp < 0.0 || !isfinite(alpha))) {  // solver.py:187-198, same verdict on every rank/CTA
    if (blockIdx.x == 0 && threadIdx.x == 0) st->stop = 1, st->status = 1, st->iterations = st->it + 1, st->pAp = pAp;
    return;
  }
  const double* p = sym_p(me);
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double ri = r[i] - alpha * Ap[i];
    u[i] += alpha * p[i];
    r[i] = ri;
    dot += ri * ri;
  }
  const double t = block_sum<DV_THREADS>(dot);
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
    for (int k = threadIdx.x; k < (int)gridDim.x; k += DV_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<DV_THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket2 = 0;
      st->pAp = pAp, st->alpha = alpha;
      const long long e = st->epochC + 1;
      st->epochC = e;
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->redC[pe.rank] = a;
      __threadfence_system();
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->flagC[pe.rank] = e;
      trace_stamp(st, 7);
    }
  }
}

// ---- k3: convergence / beta ; p = r + beta p -------------------------------------------------------------------------
struct BoundaryPush {     // boundary rows [n_interior, n): destinations of each row's value (CSR over boundary rows)
  const int* ptr;         // [nb+1], nullptr = no folded push
  const unsigned char* k; // neighbour index of each destination
  const int* off;         // offset inside that neighbour's block of ghosts
  long long n_interior;
};

__global__ void __launch_bounds__(DV_THREADS) dist_direction_kernel(Peers pe, long long n, const double* __restrict__ r, DistState* st,
                                                                    double tol, double eps, int guards, int max_iter, BoundaryPush bp) {
  if (st->stop) return;
  SymHeader* me = pe.hdr[pe.rank];
  __shared__ int all[MAXP];
  if (threadIdx.x < MAXP) all[threadIdx.x] = threadIdx.x;
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 8);
  wait_flags(me->flagC, all, pe.P, st->epochC, st);
  {  // block-uniform (one read per CTA), see dist_update_kernel
    __shared__ int stop_now;
    if (threadIdx.x == 0) stop_now = st->stop;
    __syncthreads();
    if (stop_now) return;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 9);
  const double rs_new = sum_slots(me->redC, pe.P);
  const double beta = rs_new / (st->rs_old + eps);
  const bool conv = sqrt(rs_new) < tol;                  // solver.py:210-212
  const bool bad = guards && !isfinite(beta);            // solver.py:216-218
  if (conv || bad) {
    if (blockIdx.x == 0 && threadIdx.x == 0) st->stop = 1, st->status = conv ? 0 : 1, st->iterations = st->it + 1, st->rs_new = rs_new;
    return;
  }
  double* p = sym_p(me);
  const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x, gsz = (long long)gridDim.x * blockDim.x;
  const long long n_plain = bp.ptr ? bp.n_interior : n;
  // boundary rows first (their values have the longest way to go): one thread per row writes it locally and stores it
  // straight into the ghost slots of every neighbour that needs it
  if (bp.ptr) {
    for (long long b = gtid; b < n - bp.n_interior; b += gsz) {
      const long long i = bp.n_interior + b;
      const double v = r[i] + beta * p[i];
      p[i] = v;
      for (int e = bp.ptr[b]; e < bp.ptr[b + 1]; ++e) {
        const int k = bp.k[e];
        (sym_p(pe.hdr[pe.nbr[k]]) + pe.ghost_off[k])[bp.off[e]] = v;
      }
    }
    __threadfence_system();
  }
  for (long long i = gtid; i < n_plain; i += gsz) p[i] = r[i] + beta * p[i];
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(&st->ticket3, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {  // every CTA has read rs_old (and pushed its boundary rows) by now
    st->ticket3 = 0;
    st->rs_new = rs_new, st->beta = beta, st->rs_old = rs_new;
    st->it += 1;
    if (st->it >= max_iter) st->stop = 2, st->status = 2, st->iterations = max_iter;
    if (bp.ptr) {
      const long long e = st->epochA + 1;
      st->epochA = e;
      __threadfence_system();
      for (int k = 0; k < pe.nnbr; ++k) pe.hdr[pe.nbr[k]]->flagA[pe.rank] = e;
    }
    trace_stamp(st, 10);
  }
}

// =====================================================================================================================
// Merged-reduction iteration (default): TWO kernels and ONE waited all-reduce per iteration.
//   m1  SpMV as k1, but the CTA partials carry three sums: p.Ap, r.Ap and Ap.Ap (r is one more streamed vector)
//   m2  waits for that all-reduce, then alpha = rs/(p.Ap+eps) and, without a second global sum,
//         rs_new = rs - 2 alpha r.Ap + alpha^2 Ap.Ap        ( = |r - alpha Ap|^2 )
//       -> convergence test, beta, and ONE pass over the vectors: u += alpha p, r -= alpha Ap, p = r + beta p (boundary rows
//       are pushed to the neighbours' ghosts).  The same pass accumulates the TRUE r.r of the new residual; its all-reduce is
//       only consumed by m2 of the NEXT iteration (one SpMV later, so nobody waits for it) as the `rs` the recurrence starts
//       from -- rounding errors of the recurrence therefore never accumulate: each rs_new is one step away from an exact sum
//       (relative error ~ eps * rs/rs_new), and iteration counts match the three-kernel loop (tests: +-1).
// Against k1/k2/k3 this removes one launch boundary, one all-rank wait and two of the nine vector passes per iteration.
// Reduction slots are double-buffered by epoch parity: with a single all-rank wait per iteration a fast rank could
// otherwise overwrite a slot a slow rank has not read yet.
// =====================================================================================================================
// epilogue of the merged-reduction SpMV (scalar CSR and 3x3 block-CSR kernels): per-CTA partials of the three sums, the last
// CTA adds them in index order and sends the rank's sums to every rank as LL words (data + epoch in one 8-byte store)
template <int THREADS>
__device__ __forceinline__ void ll_reduce_send(const Peers& pe, double dot, double e0, double e1, double* __restrict__ partial, DistState* st) {
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
    double a[3] = {0.0, 0.0, 0.0};
    for (int k = threadIdx.x; k < G; k += THREADS)
      a[0] += ((volatile double*)partial)[k], a[1] += ((volatile double*)partial)[G + k], a[2] += ((volatile double*)partial)[2 * G + k];
    a[0] = block_sum<THREADS>(a[0]), a[1] = block_sum<THREADS>(a[1]), a[2] = block_sum<THREADS>(a[2]);
    __shared__ double sums[3];
    __shared__ long long eB;
    if (threadIdx.x == 0) {
      st->ticket1 = 0;
      eB = st->epochB + 1;
      st->epochB = eB;
      sums[0] = a[0], sums[1] = a[1], sums[2] = a[2];
    }
    __syncthreads();
    // 6 words to each of the P ranks (own included), one thread per word: data and epoch travel in the same 8-byte store
    const int par = (int)(eB & 1);
    for (int t = threadIdx.x; t < 6 * pe.P; t += THREADS) {
      const int q = t / 6, w = t - 6 * q;
      ll_store(&pe.hdr[q]->ll[par][pe.rank][w], sums[w >> 1], w & 1, eB);
    }
    if (threadIdx.x == 0) trace_stamp(st, 4);
  }
}

template <int LR, bool NC>
__global__ void __launch_bounds__(TMA_THREADS) dist_spmv3_kernel(Peers pe, long long n_owned, long long nnz, const int* __restrict__ crow,
                                                                 const int* __restrict__ col, const double* __restrict__ val,
                                                                 double* __restrict__ y, const unsigned char* __restrict__ mask,
                                                                 const double* __restrict__ rvec, const double* __restrict__ wvec,
                                                                 double* __restrict__ partial, DistState* st, long long n_interior, long long pin) {
  pdl_launch_dependents();
  SymHeader* me = pe.hdr[pe.rank];
  __shared__ int nbr[MAXP];
  if (threadIdx.x < MAXP) nbr[threadIdx.x] = pe.nbr[threadIdx.x];
  __syncthreads();
  const double* x = sym_p(me);
  // the halo epoch is read lazily (after the PDL wait inside spmv_tma_rows): st belongs to the previous kernel until then
  struct LazyHalo {
    SymHeader* me;
    const int* nbr;
    int nnbr;
    DistState* st;
    __device__ __forceinline__ void operator()() const { wait_flags(me->flagA, nbr, nnbr, st->epochA, st); }
  };
  const LazyHalo hw{me, nbr, pe.nnbr, st};
  double extra[2] = {0.0, 0.0};
  const double dot = spmv_tma_rows<LR, NC, TMA_THREADS, TMA_STAGES, TMA_CAP, LazyHalo, PdlWait>(
      n_owned, nnz, crow, col, val, x, y, mask, false, true, pe.nnbr > 0 ? n_interior : 0x7fffffffffffffffll, hw, rvec, extra, PdlWait(), &st->stop,
      pin, wvec);
  if (st->stop) return;  // set before this kernel (block-uniform) or by a spin timeout (status 3: the solve is lost anyway)
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 3);
  ll_reduce_send<TMA_THREADS>(pe, dot, extra[0], extra[1], partial, st);
}

// 3x3 block-CSR twin (3-dof operators: every elasticity solver of the reference): warp per block row as the single-GPU
// spmv_bsr3_vec_kernel (krylov.cu) -- lanes 0..26 = (block, position) of three consecutive blocks per step -- on the owned
// block rows, interior rows first; a warp waits for the halo flags when it reaches its first boundary row.  x = p in the
// symmetric buffer, dof-level numbering 3 * (local node) + component.
constexpr int DBSR_THREADS = 256;
template <int U>
__global__ void __launch_bounds__(DBSR_THREADS) dist_spmv3_bsr3_kernel(Peers pe, long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                                       const double* __restrict__ bval, double* __restrict__ y,
                                                                       const unsigned char* __restrict__ mask, const double* __restrict__ rvec,
                                                                       const double* __restrict__ wvec, double* __restrict__ partial, DistState* st,
                                                                       long long nb_interior) {
  pdl_launch_dependents();
  pdl_wait();
  if (st->stop) return;
  SymHeader* me = pe.hdr[pe.rank];
  const double* x = sym_p(me);
  const int lane = threadIdx.x & 31;
  const int boff = lane / 9, pos = lane - 9 * boff, cx = pos % 3;  // lanes 27..31: boff = 3 -> idle
  const bool active = lane < 27;
  const long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long epochA = st->epochA;
  bool waited = pe.nnbr == 0;
  double dot = 0.0, e0 = 0.0, e1 = 0.0;
  for (long long r = gw; r < nb; r += nw) {
    if (!waited && r >= nb_interior) {  // first boundary row of this warp: its columns may be ghosts
      if (lane < pe.nnbr) spin_until(me->flagA + pe.nbr[lane], epochA, st);
      __syncwarp();
      waited = true;
    }
    const int a = __ldg(brow + r), e = __ldg(brow + r + 1);
    double r_own = 0.0, w_own = 1.0;  // requested before the block loop (see spmv_bsr3_vec_kernel)
    if (lane == 0 || lane == 3 || lane == 6) {
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
    acc += __shfl_down_sync(0xffffffffu, acc, 9) + __shfl_down_sync(0xffffffffu, acc, 18);
    acc += __shfl_down_sync(0xffffffffu, acc, 1) + __shfl_down_sync(0xffffffffu, acc, 2);
    if (lane == 0 || lane == 3 || lane == 6) {
      const long long i = 3 * r + lane / 3;
      double sv = acc;
      if (mask && !mask[i]) sv = 0.0;
      dot += sv * __ldg(x + i);
      e0 += sv * (w_own * r_own), e1 += sv * (sv * w_own);
      y[i] = sv;
    }
  }
  if (st->stop == 3) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 3);
  ll_reduce_send<DBSR_THREADS>(pe, dot, e0, e1, partial, st);
}

__global__ void __launch_bounds__(DV_THREADS) dist_merged_vec_kernel(Peers pe, long long n, double* __restrict__ u, double* __restrict__ r,
                                                                     const double* __restrict__ Ap, const double* __restrict__ minv,
                                                                     double* __restrict__ partial, DistState* st, double tol, double eps,
                                                                     int guards, int max_iter, BoundaryPush bp) {
  // minv != nullptr: Jacobi-PCG (solver.py:766-812): z = minv .* r, the sums are r.z, p = z + beta p; the three sums of the
  // SpMV carry the same weights, so rs_new below is the recurrence of r.z
  pdl_launch_dependents();
  pdl_wait();
  if (st->stop) return;
  SymHeader* me = pe.hdr[pe.rank];
  __shared__ unsigned halves[MAXP * 8];
  __shared__ double sc[4];
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 5);
  const long long eB = st->epochB, eC = st->epochC;
  const int it = st->it;
  {  // all-reduce: wait for the 6 (+2 from the previous update, it > 0) words of every rank; one thread per word
    const int pb = (int)(eB & 1), pc = (int)(eC & 1);
    for (int t = threadIdx.x; t < 8 * pe.P; t += DV_THREADS) {
      const int q = t >> 3, w = t & 7;
      if (w < 6) halves[t] = ll_wait(&me->ll[pb][q][w], eB, st);
      else halves[t] = it > 0 ? ll_wait(&me->ll[pc][q][w], eC, st) : 0u;
    }
  }
  // block-uniform exit on a spin timeout (status 3): ONE read per CTA, broadcast through shared memory
  __shared__ int stop_now;
  if (threadIdx.x == 0) stop_now = st->stop;
  __syncthreads();
  if (stop_now) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) trace_stamp(st, 6);
  if (threadIdx.x < 4) {  // sums in rank order: identical on every rank and CTA
    double a = 0.0;
    for (int q = 0; q < pe.P; ++q)
      a += __longlong_as_double((long long)(((unsigned long long)halves[q * 8 + 2 * threadIdx.x + 1] << 32) | halves[q * 8 + 2 * threadIdx.x]));
    sc[threadIdx.x] = (threadIdx.x == 3 && it == 0) ? st->rs_old : a;
  }
  __syncthreads();
  const double pAp = sc[0], rAp = sc[1], ApAp = sc[2], rs_old = sc[3];
  // rs_old is the exactly summed r.r of the previous update (it arrived one SpMV ago): the reference's convergence test
  // (solver.py:208-212) is applied to IT, one SpMV late, before anything of this iteration is applied -- u and r are then
  // exactly the reference's state at its break.  The recurrence value below only feeds beta.
  // The stop flag is raised by the LAST CTA to take a ticket, never earlier: a CTA that is still on its way to the checks
  // above must not see it change under its feet (a flag set by the first CTA to get here split slower CTAs -- some warps left
  // at the check, the others went on without the scalars warp 0 computes and applied a garbage update to their rows).
  const bool converged = it > 0 && sqrt(rs_old) < tol;
  const double alpha = rs_old / (pAp + eps);
  const bool broke = !converged && guards && (fabs(pAp) < eps || pAp < 0.0 || !isfinite(alpha));  // solver.py:187-198, same verdict everywhere
  if (converged || broke) {
    if (threadIdx.x == 0 && atomicAdd(&st->ticket2, 1u) == gridDim.x - 1) {
      st->ticket2 = 0;
      st->rs_new = rs_old;
      if (converged) st->status = 0, st->iterations = it;
      else st->status = 1, st->iterations = it + 1, st->pAp = pAp;
      __threadfence();
      st->stop = 1;
    }
    return;
  }
  double rs_new = rs_old - 2.0 * alpha * rAp + alpha * alpha * ApAp;
  if (!(rs_new > 0.0)) rs_new = 0.0;                      // cancellation: beta = 0 restarts the direction, never a false "converged"
  const double beta = rs_new / (rs_old + eps);
  const bool bad = guards && !isfinite(beta);             // solver.py:216-218
  const bool move_p = !bad;
  double* p = sym_p(me);
  const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x, gsz = (long long)gridDim.x * blockDim.x;
  const long long n_plain = bp.ptr ? bp.n_interior : n;
  double dot = 0.0;
  if (bp.ptr) {  // boundary rows first: their new p has the longest way to go
    for (long long b = gtid; b < n - bp.n_interior; b += gsz) {
      const long long i = bp.n_interior + b;
      const double pi = p[i], ri = r[i] - alpha * Ap[i];
      const double zi = minv ? minv[i] * ri : ri;
      u[i] += alpha * pi;
      r[i] = ri;
      dot += ri * zi;
      if (move_p) {
        const double v = zi + beta * pi;
        p[i] = v;
        for (int e = bp.ptr[b]; e < bp.ptr[b + 1]; ++e) {
          const int k = bp.k[e];
          (sym_p(pe.hdr[pe.nbr[k]]) + pe.ghost_off[k])[bp.off[e]] = v;
        }
      }
    }
    // peer stores must be performed before this CTA's ticket (the halo flag follows the last ticket); CTAs whose threads all
    // lie beyond the boundary rows stored nothing remotely and skip the system-scope fence.  (Placing the fence after the
    // interior rows instead measured SLOWER at 4 and 8 GPUs, 26 -> 31 us and 16.5 -> 18.4 us for this kernel: a system fence
    // waits for every earlier write of the thread, and by then those are the whole u / r / p update.)
    if (blockIdx.x * (long long)blockDim.x < n - bp.n_interior) __threadfence_system();
  }
  for (long long i = gtid; i < n_plain; i += gsz) {
    const double pi = p[i], ri = r[i] - alpha * Ap[i];
    const double zi = minv ? minv[i] * ri : ri;
    u[i] += alpha * pi;
    r[i] = ri;
    dot += ri * zi;
    if (move_p) p[i] = zi + beta * pi;
  }
  const double t = block_sum<DV_THREADS>(dot);
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
    for (int k = threadIdx.x; k < (int)gridDim.x; k += DV_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<DV_THREADS>(a);
    __shared__ double rr;
    __shared__ long long eCn;
    if (threadIdx.x == 0) {
      trace_stamp(st, 7), trace_stamp(st, 8), trace_stamp(st, 9);
      st->ticket2 = 0;
      st->pAp = pAp, st->alpha = alpha, st->beta = beta, st->rs_new = rs_new, st->rs_old = rs_new;
      eCn = eC + 1;
      st->epochC = eCn;
      rr = a;
      if (!move_p) {
        st->stop = 1, st->status = 1, st->iterations = it + 1;
      } else {
        st->it = it + 1;
        if (it + 1 >= max_iter) st->stop = 2, st->status = 2, st->iterations = max_iter;
        if (bp.ptr) {  // every CTA fenced its pushes before taking a ticket: the halo is complete on the neighbours
          const long long ea = st->epochA + 1;
          st->epochA = ea;
          for (int k = 0; k < pe.nnbr; ++k) pe.hdr[pe.nbr[k]]->flagA[pe.rank] = ea;
        }
      }
    }
    __syncthreads();
    // exactly summed r.r of this update -> everyone (consumed by the next iteration's vector kernel / the final check)
    const int par = (int)(eCn & 1);
    for (int t2 = threadIdx.x; t2 < 2 * pe.P; t2 += DV_THREADS) {
      const int q = t2 >> 1, w = 6 + (t2 & 1);
      ll_store(&pe.hdr[q]->ll[par][pe.rank][w], rr, w & 1, eCn);
    }
    if (threadIdx.x == 0) trace_stamp(st, 10);
  }
}

// Cross-rank barrier in front of the iteration graph.  Capturing and instantiating the graph costs each rank's HOST a
// millisecond of jittery work during which its GPU idles; without this kernel the ranks would enter iteration 0 hundreds of
// microseconds apart and the early ones would spend that time inside their first all-reduce wait -- 5 us per iteration on a
// 20-iteration solve.  It is enqueued after the instantiation, right in front of the timing event and the first graph launch.
__global__ void dist_start_barrier(Peers pe, DistState* st) {
  SymHeader* me = pe.hdr[pe.rank];
  if (threadIdx.x < pe.P) pe.hdr[threadIdx.x]->flagS[pe.rank] = 1;
  if (threadIdx.x < pe.P) spin_until(me->flagS + threadIdx.x, 1, st);
}

// after the last graph: the loop tests convergence one SpMV late, so an update that converged in the very last iteration
// (status "maxiter") or right before a breakdown verdict is settled here from the r.r all-reduce that is still in flight
__global__ void dist_final_check(Peers pe, DistState* st, double tol) {
  SymHeader* me = pe.hdr[pe.rank];
  __shared__ unsigned halves[MAXP * 2];
  if (st->status == 3 || st->it == 0 || (st->stop == 1 && st->status == 0)) return;
  const long long eC = st->epochC;
  const int pc = (int)(eC & 1);
  for (int t = threadIdx.x; t < 2 * pe.P; t += blockDim.x) halves[t] = ll_wait(&me->ll[pc][t >> 1][6 + (t & 1)], eC, st);
  __syncthreads();
  if (threadIdx.x == 0 && st->status != 3) {
    double a = 0.0;
    for (int q = 0; q < pe.P; ++q) a += __longlong_as_double((long long)(((unsigned long long)halves[2 * q + 1] << 32) | halves[2 * q]));
    st->rs_new = a;  // the reported residual is the exactly summed one
    if (sqrt(a) < tol && st->status == 2) st->stop = 1, st->status = 0, st->iterations = st->it;
  }
}

// plain block-CSR product for the setup (Ap = A u): every warp waits for the neighbours' halo of this epoch first
__global__ void __launch_bounds__(DBSR_THREADS) dist_bsr3_plain_kernel(Peers pe, long long nb, const int* __restrict__ brow, const int* __restrict__ bcol,
                                                                       const double* __restrict__ bval, double* __restrict__ y, DistState* st) {
  SymHeader* me = pe.hdr[pe.rank];
  const double* x = sym_p(me);
  const int lane = threadIdx.x & 31;
  const int boff = lane / 9, pos = lane - 9 * boff, cx = pos % 3;
  const bool active = lane < 27;
  if (lane < pe.nnbr) spin_until(me->flagA + pe.nbr[lane], st->epochA, st);
  __syncwarp();
  const long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = gw; r < nb; r += nw) {
    const int a = __ldg(brow + r), e = __ldg(brow + r + 1);
    double acc = 0.0;
    if (active)
      for (int b = a + boff; b < e; b += 3) acc += ld_stream(bval + (size_t)b * 9 + pos) * __ldg(x + 3ll * ld_stream(bcol + b) + cx);
    acc += __shfl_down_sync(0xffffffffu, acc, 9) + __shfl_down_sync(0xffffffffu, acc, 18);
    acc += __shfl_down_sync(0xffffffffu, acc, 1) + __shfl_down_sync(0xffffffffu, acc, 2);
    if (lane == 0 || lane == 3 || lane == 6) y[3 * r + lane / 3] = acc;
  }
}

// ---- setup ------------------------------------------------------------------------------------------------------------
__global__ void dist_load_p(Peers pe, long long n, double* __restrict__ u, const unsigned char* __restrict__ mask) {
  double* p = sym_p(pe.hdr[pe.rank]);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) u[i] = 0.0;
    p[i] = u[i];
  }
}

__global__ void __launch_bounds__(DV_THREADS) dist_init_kernel(Peers pe, long long n, const double* __restrict__ F, const double* __restrict__ Au,
                                                               const unsigned char* __restrict__ mask, const double* __restrict__ minv,
                                                               double* __restrict__ r, double* __restrict__ partial, DistState* st) {
  double* p = sym_p(pe.hdr[pe.rank]);
  double dot = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double ri = F[i] - Au[i];
    if (mask && !mask[i]) ri = 0.0;
    const double z = minv ? minv[i] * ri : ri;
    r[i] = ri;
    p[i] = z;
    dot += ri * z;
  }
  const double t = block_sum<DV_THREADS>(dot);
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
    for (int k = threadIdx.x; k < (int)gridDim.x; k += DV_THREADS) a += ((volatile double*)partial)[k];
    a = block_sum<DV_THREADS>(a);
    if (threadIdx.x == 0) {
      st->ticket2 = 0;
      const long long e = st->epochC + 1;
      st->epochC = e;
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->redC[pe.rank] = a;
      __threadfence_system();
      for (int q = 0; q < pe.P; ++q) pe.hdr[q]->flagC[pe.rank] = e;
    }
  }
}

__global__ void dist_init_finish(Peers pe, DistState* st, int max_iter) {
  SymHeader* me = pe.hdr[pe.rank];
  if (threadIdx.x == 0) {
    bool ok = true;
    for (int q = 0; q < pe.P && ok; ++q) ok = spin_until(me->flagC + q, st->epochC, st);
    if (ok) {
      const double a = sum_slots_serial(me->redC, pe.P);
      st->rs_old = a, st->rs_new = a;
      if (max_iter <= 0) st->stop = 2, st->status = 2;
    }
  }
}

// ---- persistent variant: the whole solve is ONE cooperative kernel -------------------------------------------------------
// All CTAs are co-resident (cooperative launch) and walk the phases of every iteration together:
//   push (peer stores of the boundary of p; last CTA raises flag A on the neighbours)
//   SpMV (interior row tiles first; a CTA waits for flag A only when it reaches its first boundary tile) + p.Ap partial,
//        last CTA stores the rank's partial into every rank's slot and raises flag B
//   wait B -> alpha -> u, r update + r.r partial -> last CTA -> slots + flag C
//   wait C -> convergence / beta -> p update -> local grid barrier
// Iteration scalars live in registers of every thread (identical everywhere: they are functions of the rank-ordered sums),
// so there is no launch boundary, no graph and no host round trip inside the solve.  Because the kernel never ends between
// iterations the L1 is not flushed for us: every wait is followed by a fence (acquire side of the message-passing pattern)
// and x is read with plain loads, never through the non-coherent path.
struct PersistArgs {
  Peers pe;
  long long n, n_interior;
  const int *crow, *col;
  const double *val, *F, *minv;
  const unsigned char* mask;
  double *u, *r, *Ap, *partial;
  const int* send_idx;
  DistState* st;
  unsigned long long* counters;  // [4] monotonic: push tickets, k1 tickets, k2 tickets, grid barrier
  double tol, eps;
  int max_iter, guards;
};

__device__ __forceinline__ void wait_then_fence(volatile long long* flags, const int* ranks, int count, long long expect, DistState* st) {
  if (threadIdx.x < count) spin_until(flags + ranks[threadIdx.x], expect, st);
  if (threadIdx.x < 32) __threadfence_system();
  __syncthreads();
}

struct HaloWaiter {
  SymHeader* me;
  const int* nbr;
  int nnbr;
  long long epoch;
  DistState* st;
  __device__ __forceinline__ void operator()() const { wait_then_fence(me->flagA, nbr, nnbr, epoch, st); }
};

template <int LR>
__global__ void __launch_bounds__(SPMV_THREADS) dist_cg_persistent_kernel(const PersistArgs a) {
  const Peers& pe = a.pe;
  SymHeader* me = pe.hdr[pe.rank];
  double* p = sym_p(me);
  DistState* st = a.st;
  const unsigned long long G = gridDim.x;
  const int tid = threadIdx.x;
  const long long gtid = blockIdx.x * (long long)blockDim.x + tid, gsz = (long long)gridDim.x * blockDim.x;
  __shared__ int all[MAXP], nbr[MAXP];
  __shared__ bool last;
  if (tid < MAXP) all[tid] = tid, nbr[tid] = pe.nbr[tid];
  __syncthreads();
  const bool pre = a.minv != nullptr;
  double rs_old = st->rs_old;      // set by the setup kernels
  long long eA = st->epochA, eB = st->epochB, eC = st->epochC;
  unsigned long long round = 0;    // iterations done by this launch (tickets are monotonic: last CTA sees G*(round+1))
  int it = 0, stop = a.max_iter <= 0 ? 2 : 0, status = 2, iterations = a.max_iter;
  double rs_new = rs_old, pAp = 0.0;
  const int total_send = pe.send_ptr[pe.nnbr];
  while (!stop) {
    // ---- push
    for (long long t = gtid; t < total_send; t += gsz) {
      int k = 0;
      while (t >= pe.send_ptr[k + 1]) ++k;
      (sym_p(pe.hdr[pe.nbr[k]]) + pe.ghost_off[k])[t - pe.send_ptr[k]] = p[a.send_idx[t]];
    }
    ++eA;
    if (pe.nnbr > 0) {
      __threadfence_system();
      __syncthreads();
      if (tid == 0 && atomicAdd(&a.counters[0], 1ull) + 1 == G * (round + 1)) {
        __threadfence_system();
        for (int k = 0; k < pe.nnbr; ++k) pe.hdr[pe.nbr[k]]->flagA[pe.rank] = eA;
      }
    }
    // ---- SpMV + p.Ap
    const HaloWaiter hw{me, nbr, pe.nnbr, eA, st};
    double dot = spmv_stream_rows<LR, false, HaloWaiter>(a.n, a.crow, a.col, a.val, p, a.Ap, a.mask, false, true,
                                                          pe.nnbr > 0 ? a.n_interior : 0x7fffffffffffffffll, hw);
    double t = block_sum<SPMV_THREADS>(dot);
    if (tid == 0) {
      a.partial[blockIdx.x] = t;
      __threadfence();
      last = atomicAdd(&a.counters[1], 1ull) + 1 == G * (round + 1);
    }
    __syncthreads();
    ++eB;
    if (last) {
      __threadfence();
      double s = 0.0;
      for (int k = tid; k < (int)G; k += SPMV_THREADS) s += ((volatile double*)a.partial)[k];
      s = block_sum<SPMV_THREADS>(s);
      if (tid == 0) {
        for (int q = 0; q < pe.P; ++q) pe.hdr[q]->redB[pe.rank] = s;
        __threadfence_system();
        for (int q = 0; q < pe.P; ++q) pe.hdr[q]->flagB[pe.rank] = eB;
      }
    }
    // ---- alpha, u/r update, r.z
    wait_then_fence(me->flagB, all, pe.P, eB, st);
    if (st->stop == 3) break;
    pAp = sum_slots(me->redB, pe.P);
    const double alpha = rs_old / (pAp + a.eps);
    if (a.guards && (fabs(pAp) < a.eps || pAp < 0.0 || !isfinite(alpha))) {  // solver.py:187-198
      stop = 1, status = 1, iterations = it + 1;
      break;
    }
    dot = 0.0;
    for (long long i = gtid; i < a.n; i += gsz) {
      const double ri = a.r[i] - alpha * a.Ap[i];
      a.u[i] += alpha * p[i];
      a.r[i] = ri;
      dot += pre ? ri * (a.minv[i] * ri) : ri * ri;
    }
    t = block_sum<SPMV_THREADS>(dot);
    if (tid == 0) {
      a.partial[blockIdx.x] = t;
      __threadfence();
      last = atomicAdd(&a.counters[2], 1ull) + 1 == G * (round + 1);
    }
    __syncthreads();
    ++eC;
    if (last) {
      __threadfence();
      double s = 0.0;
      for (int k = tid; k < (int)G; k += SPMV_THREADS) s += ((volatile double*)a.partial)[k];
      s = block_sum<SPMV_THREADS>(s);
      if (tid == 0) {
        for (int q = 0; q < pe.P; ++q) pe.hdr[q]->redC[pe.rank] = s;
        __threadfence_system();
        for (int q = 0; q < pe.P; ++q) pe.hdr[q]->flagC[pe.rank] = eC;
      }
    }
    // ---- convergence, beta, direction
    wait_then_fence(me->flagC, all, pe.P, eC, st);
    if (st->stop == 3) break;
    rs_new = sum_slots(me->redC, pe.P);
    if (sqrt(rs_new) < a.tol) {  // solver.py:210-212 / :804-806
      stop = 1, status = 0, iterations = it + 1;
      break;
    }
    const double beta = rs_new / (rs_old + a.eps);
    if (a.guards && !isfinite(beta)) {  // solver.py:216-218
      stop = 1, status = 1, iterations = it + 1;
      break;
    }
    for (long long i = gtid; i < a.n; i += gsz) p[i] = (pre ? a.minv[i] * a.r[i] : a.r[i]) + beta * p[i];
    rs_old = rs_new;
    ++it;
    ++round;
    if (it >= a.max_iter) stop = 2, status = 2, iterations = a.max_iter;
    // ---- local grid barrier: p is complete before anyone pushes or gathers it again
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      atomicAdd(&a.counters[3], 1ull);
      const long long t0 = clock64();
      while (*((volatile unsigned long long*)&a.counters[3]) < G * round) {
        if (clock64() - t0 > SPIN_TIMEOUT_CYCLES) {
          st->stop = 3, st->status = 3;
          break;
        }
      }
      __threadfence();
    }
    __syncthreads();
    if (st->stop == 3) break;
  }
  if (blockIdx.x == 0 && tid == 0 && st->stop != 3) {
    st->it = it, st->stop = stop ? stop : 2, st->status = status, st->iterations = iterations;
    st->rs_new = rs_new, st->rs_old = rs_old, st->pAp = pAp;
    st->epochA = eA, st->epochB = eB, st->epochC = eC;
  }
}

static int pick_lr(long long n, long long nnz) {
  const double avg = n > 0 ? (double)nnz / (double)n : 1.0;
  for (int lr = 1; lr <= 32; lr *= 2)
    if ((SPMV_THREADS / lr) * avg * 1.25 <= STREAM_CAP) return lr;
  return 32;
}

template <bool FUSED>
static void launch_dist_spmv(int lr, int grid, cudaStream_t s, const Peers& pe, long long n, long long nnz, const int* crow, const int* col,
                             const double* val, double* y, const unsigned char* mask, double* partial, DistState* st, long long n_interior) {
  static const bool nc = getenv("FEMB_DIST_PLAIN_X") == nullptr;  // read-only path for x: 17 % faster than plain loads; safe because
  // ghosts start on their own 128-byte line and are first touched after the halo flag (L1 is flushed at every launch)
#define FEMB_DSPMV(LRV)                                                                                                         \
  {                                                                                                                             \
    if (nc) {                                                                                                                   \
      cudaFuncSetAttribute(dist_spmv_kernel<LRV, FUSED, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TMA_SMEM);     \
      dist_spmv_kernel<LRV, FUSED, true><<<grid, TMA_THREADS, TMA_SMEM, s>>>(pe, n, nnz, crow, col, val, y, mask, partial, st, n_interior); \
    } else {                                                                                                                    \
      cudaFuncSetAttribute(dist_spmv_kernel<LRV, FUSED, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TMA_SMEM);    \
      dist_spmv_kernel<LRV, FUSED, false><<<grid, TMA_THREADS, TMA_SMEM, s>>>(pe, n, nnz, crow, col, val, y, mask, partial, st, n_interior); \
    }                                                                                                                           \
  }
  switch (lr) {
    case 1: FEMB_DSPMV(1) break;
    case 2: FEMB_DSPMV(2) break;
    case 4: FEMB_DSPMV(4) break;
    case 8: FEMB_DSPMV(8) break;
    case 16: FEMB_DSPMV(16) break;
    default: FEMB_DSPMV(32) break;
  }
#undef FEMB_DSPMV
}

static void launch_dist_spmv3(int lr, int grid, cudaStream_t s, bool pdl, const Peers& pe, long long n, long long nnz, const int* crow,
                              const int* col, const double* val, double* y, const unsigned char* mask, const double* rvec, const double* wvec,
                              double* partial, DistState* st, long long n_interior, long long pin) {
#define FEMB_DSPMV3(LRV)                                                                                                    \
  {                                                                                                                         \
    cudaFuncSetAttribute(dist_spmv3_kernel<LRV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TMA_SMEM);         \
    launch_pdl(dist_spmv3_kernel<LRV, true>, grid, TMA_THREADS, TMA_SMEM, s, pdl, pe, n, nnz, crow, col, val, y, mask, rvec, wvec, partial, \
               st, n_interior, pin);                                                                                        \
  }
  switch (lr) {
    case 1: FEMB_DSPMV3(1) break;
    case 2: FEMB_DSPMV3(2) break;
    case 4: FEMB_DSPMV3(4) break;
    case 8: FEMB_DSPMV3(8) break;
    case 16: FEMB_DSPMV3(16) break;
    default: FEMB_DSPMV3(32) break;
  }
#undef FEMB_DSPMV3
}

}  // namespace femb

using namespace femb;

extern "C" int femb_dist_header_bytes(void) { return (int)sizeof(SymHeader); }

extern "C" int femb_dist_alloc(int64_t bytes, void** ptr, void* ipc_handle64) {
  FEMB_CHECK_ARG(bytes > 0 && ptr && ipc_handle64, "bytes/ptr/handle");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
  FEMB_CUDA(cudaMalloc(ptr, (size_t)bytes));
  FEMB_CUDA(cudaMemset(*ptr, 0, (size_t)bytes));
  FEMB_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle64), *ptr));
  return FEMB_OK;
}

extern "C" int femb_dist_open(const void* ipc_handle64, void** ptr) {
  FEMB_CHECK_ARG(ptr && ipc_handle64, "ptr/handle");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle64, sizeof(h));
  FEMB_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return FEMB_OK;
}

extern "C" int femb_dist_close(void* ptr) {
  FEMB_CUDA(cudaIpcCloseMemHandle(ptr));
  return FEMB_OK;
}

extern "C" int femb_dist_free(void* ptr) {
  FEMB_CUDA(cudaFree(ptr));
  return FEMB_OK;
}

extern "C" int femb_dist_reset(void* own_sym, femb_stream stream) {
  FEMB_CUDA(cudaMemsetAsync(own_sym, 0, sizeof(SymHeader), as_stream(stream)));
  FEMB_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return FEMB_OK;
}

extern "C" int femb_dist_cg_solve(int rank, int nranks, int64_t n_owned, int64_t n_interior, int64_t nnz, const int32_t* crow,
                                  const int32_t* col, const double* val, const double* F, const uint8_t* mask, const double* minv,
                                  double* u, double* work, void* const* sym_host, int nnbr,
                                  const int32_t* nbr_host, const int32_t* send_ptr_host, const int32_t* send_idx,
                                  const int64_t* ghost_off_host, const int32_t* bptr, const uint8_t* bk, const int32_t* boff, double tol,
                                  int max_iter, double eps, int check_every, int block, femb_cg_result* result_host, femb_stream stream) {
  FEMB_CHECK_ARG(nranks >= 1 && nranks <= MAXP && rank >= 0 && rank < nranks && nnbr >= 0 && nnbr < MAXP, "rank/nranks/nnbr");
  FEMB_CHECK_ARG(block == 1 || (block == 3 && n_owned % 3 == 0 && n_interior % 3 == 0), "block in {1,3}; block 3 needs 3 rows per node");
  FEMB_CHECK_ARG(n_owned > 0 && crow && col && val && F && u && work && sym_host && result_host, "null pointer / n_owned <= 0");
  if (check_every < 1) check_every = 16;
  spmv_apply_env_once();
  SolveCtx* ctx = solve_ctx(as_stream(stream));  // private capture-capable stream of the current device, ordered after the caller's
  if (!ctx) return FEMB_ERR_CUDA;
  cudaStream_t s = ctx->stream;
  Peers pe;
  memset(&pe, 0, sizeof(pe));
  pe.rank = rank, pe.P = nranks, pe.nnbr = nnbr;
  for (int q = 0; q < nranks; ++q) pe.hdr[q] = static_cast<SymHeader*>(sym_host[q]);
  for (int k = 0; k < nnbr; ++k) pe.nbr[k] = nbr_host[k], pe.ghost_off[k] = ghost_off_host[k];
  for (int k = 0; k <= nnbr; ++k) pe.send_ptr[k] = send_ptr_host[k];
  const long long n = n_owned;
  double *r = work, *Ap = work + n;
  const int lr = tma_pick_lr(n, nnz);
  int g1 = tma_grid(n, lr);
  if (block == 3) {  // warp per block row, persistent: every CTA that fits on the device
    int per_sm = 0;
    FEMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dist_spmv3_bsr3_kernel<4>, DBSR_THREADS, 0));
    g1 = (int)std::max<long long>(1, std::min<long long>((n / 3 + DBSR_THREADS / 32 - 1) / (DBSR_THREADS / 32), (long long)SMS * std::max(per_sm, 1)));
  }
  const int g2 = grid_for(n, DV_THREADS, 8);
  const int gp = std::max(1, std::min(64, (pe.send_ptr[nnbr] + 255) / 256));
  Scratch scr(s);
  double* partial;
  DistState* st;
  FEMB_CUDA(scr.alloc(&partial, (size_t)std::max(3 * g1, g2)));
  FEMB_CUDA(scr.alloc(&st, 1));
  FEMB_CUDA(cudaMemsetAsync(st, 0, sizeof(DistState), s));
  long long* trace = nullptr;
  if (getenv("FEMB_DIST_TRACE")) {
    FEMB_CUDA(scr.alloc(&trace, (size_t)TRACE_ITERS * 12));
    FEMB_CUDA(cudaMemsetAsync(trace, 0, sizeof(long long) * TRACE_ITERS * 12, s));
    FEMB_CUDA(cudaMemcpyAsync(&st->trace, &trace, sizeof(trace), cudaMemcpyHostToDevice, s));
  }
  const int guards = minv ? 0 : 1;  // the reference's PCG loop has no guards and no eps (solver.py:795-810)
  if (minv) eps = 0.0;
  if (n_interior < 0 || n_interior > n_owned) n_interior = 0;
  // ---- setup: p <- mask.*u, halo, Ap = A u, r = mask.*(F - Ap), p = r, rs_old = allreduce(r.r)   (solver.py:163-181)
  dist_load_p<<<g2, DV_THREADS, 0, s>>>(pe, n, u, mask);
  dist_push_kernel<<<gp, 256, 0, s>>>(pe, send_idx, st);
  if (block == 3) dist_bsr3_plain_kernel<<<g1, DBSR_THREADS, 0, s>>>(pe, n / 3, crow, col, val, Ap, st);
  else launch_dist_spmv<false>(lr, g1, s, pe, n, nnz, crow, col, val, Ap, nullptr, nullptr, st, 0);
  dist_init_kernel<<<g2, DV_THREADS, 0, s>>>(pe, n, F, Ap, mask, minv, r, partial, st);
  dist_init_finish<<<1, 32, 0, s>>>(pe, st, max_iter);
  FEMB_LAUNCH_CHECK();
  // default: three kernels per iteration in a CUDA graph.  FEMB_DIST_PERSISTENT=1 (and PCG) selects the single persistent
  // cooperative kernel, which measured slower so far (grid-wide software barriers cost more than launch boundaries)
  static const bool use_persistent = getenv("FEMB_DIST_PERSISTENT") != nullptr;
  if (use_persistent && block == 1) {
    // ---- iterations: one persistent cooperative kernel
    PersistArgs pa;
    pa.pe = pe, pa.n = n, pa.n_interior = n_interior, pa.crow = crow, pa.col = col, pa.val = val, pa.F = F, pa.minv = minv, pa.mask = mask;
    pa.u = u, pa.r = r, pa.Ap = Ap, pa.send_idx = send_idx, pa.st = st, pa.tol = tol, pa.eps = eps, pa.max_iter = max_iter, pa.guards = guards;
    const void* kern = nullptr;
    switch (pick_lr(n, nnz)) {
      case 1: kern = (const void*)dist_cg_persistent_kernel<1>; break;
      case 2: kern = (const void*)dist_cg_persistent_kernel<2>; break;
      case 4: kern = (const void*)dist_cg_persistent_kernel<4>; break;
      case 8: kern = (const void*)dist_cg_persistent_kernel<8>; break;
      case 16: kern = (const void*)dist_cg_persistent_kernel<16>; break;
      default: kern = (const void*)dist_cg_persistent_kernel<32>; break;
    }
    int per_sm = 0, dev = 0, sms = SMS;
    FEMB_CUDA(cudaGetDevice(&dev));
    FEMB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    FEMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SPMV_THREADS, 0));
    FEMB_CHECK_ARG(per_sm >= 1, "persistent CG kernel does not fit on an SM");
    const int G = per_sm * sms;
    unsigned long long* counters;
    FEMB_CUDA(scr.alloc(&pa.partial, (size_t)G));
    FEMB_CUDA(scr.alloc(&counters, 4));
    FEMB_CUDA(cudaMemsetAsync(counters, 0, 4 * sizeof(unsigned long long), s));
    pa.counters = counters;
    static_assert(2 * sizeof(DistState) <= SOLVE_PINNED_BYTES, "pinned status buffer");
    DistState* hfin = static_cast<DistState*>(ctx->pinned);
    cudaEvent_t* pev = ctx->time_ev;
    void* kargs[] = {(void*)&pa};
    FEMB_CUDA(cudaEventRecord(pev[0], s));
    FEMB_CUDA(cudaLaunchCooperativeKernel(kern, dim3(G), dim3(SPMV_THREADS), kargs, 0, s));
    FEMB_CUDA(cudaEventRecord(pev[1], s));
    FEMB_CUDA(cudaMemcpyAsync(hfin, st, sizeof(DistState), cudaMemcpyDeviceToHost, s));
    FEMB_CUDA(cudaStreamSynchronize(s));
    float pms = 0.f;
    cudaEventElapsedTime(&pms, pev[0], pev[1]);
    if (hfin->status == 3 || hfin->stop == 3) {
      set_error("distributed CG: timed out waiting for a peer rank (flag never arrived)");
      return FEMB_ERR_NCCL;
    }
    result_host->iterations = hfin->iterations;
    result_host->status = hfin->status;
    result_host->rs = hfin->rs_new;
    result_host->loop_ms = pms;
    result_host->index_bytes = 4;
    return FEMB_OK;
  }
  if (bptr != nullptr && nnbr > 0 && n_interior > 0 && !getenv("FEMB_DIST_SEPARATE_PUSH")) dist_push_kernel<<<gp, 256, 0, s>>>(pe, send_idx, st);
  // ---- iterations: CUDA graph (k1, k2, k3 with the halo push folded into k3)
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  FEMB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  const bool folded = bptr != nullptr && nnbr > 0 && n_interior > 0 && !getenv("FEMB_DIST_SEPARATE_PUSH");
  BoundaryPush bp{folded ? bptr : nullptr, bk, boff, n_interior};
  // FEMB_DIST_CLASSIC=1: the three-kernel loop k1/k2/k3 (two waited all-reduces); default: merged reduction m1/m2
  static const bool classic_env = getenv("FEMB_DIST_CLASSIC") != nullptr;
  const bool classic = classic_env && block == 1 && !minv;  // the three-kernel loop exists for scalar CSR without a preconditioner
  const bool pdl = pdl_enabled() && !classic;
  const long long pin = classic ? 0 : spmv_pin_entries(nnz);
  // with PDL the next SpMV's CTAs (4 x 128 threads per SM) become resident beside the vector kernel: leave them room
  static const int vec_waves = getenv("FEMB_DIST_VEC_WAVES") ? atoi(getenv("FEMB_DIST_VEC_WAVES")) : 8;
  const int g2m = pdl ? grid_for(n, DV_THREADS, vec_waves) : g2;
  for (int k = 0; k < check_every; ++k) {
    if (!folded && nnbr > 0) dist_push_kernel<<<gp, 256, 0, s>>>(pe, send_idx, st);
    if (classic) {
      launch_dist_spmv<true>(lr, g1, s, pe, n, nnz, crow, col, val, Ap, mask, partial, st, n_interior);
      dist_update_kernel<<<g2, DV_THREADS, 0, s>>>(pe, n, u, r, Ap, partial, st, eps, guards);
      dist_direction_kernel<<<g2, DV_THREADS, 0, s>>>(pe, n, r, st, tol, eps, guards, max_iter, bp);
    } else {
      const bool pdl_s = pdl && k > 0 && (pdl_mode() & 2);
      if (block == 3)
        launch_pdl(dist_spmv3_bsr3_kernel<4>, g1, DBSR_THREADS, 0, s, pdl_s, pe, n / 3, crow, col, val, Ap, mask, (const double*)r, minv, partial, st,
                   n_interior / 3);
      else
        launch_dist_spmv3(lr, g1, s, pdl_s, pe, n, nnz, crow, col, val, Ap, mask, r, minv, partial, st, n_interior, pin);
      launch_pdl(dist_merged_vec_kernel, g2m, DV_THREADS, 0, s, pdl && (pdl_mode() & 1), pe, n, u, r, Ap, minv, partial, st, tol, eps, guards, max_iter,
                 bp);
    }
  }
  cudaError_t ce = cudaStreamEndCapture(s, &graph);
  if (ce != cudaSuccess) {
    set_error(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
    return FEMB_ERR_CUDA;
  }
  FEMB_CUDA(cudaGraphInstantiate(&exec, graph, 0));
  if (!getenv("FEMB_DIST_NO_UPLOAD")) FEMB_CUDA(cudaGraphUpload(exec, s));  // the first launch must not pay for the upload inside the loop
  if (!getenv("FEMB_DIST_NO_START_BARRIER")) dist_start_barrier<<<1, 32, 0, s>>>(pe, st);
  DistState* hst = static_cast<DistState*>(ctx->pinned);  // [2] pinned
  cudaEvent_t* ev = ctx->poll_ev;
  cudaEvent_t* tev = ctx->time_ev;
  int rc = FEMB_OK;
  const int launches = (max_iter + check_every - 1) / check_every;
  hst[0].stop = hst[1].stop = 0;
  bool stopped = false;
  cudaEventRecord(tev[0], s);
  for (int l = 0; l < launches && !stopped; ++l) {
    if (cudaGraphLaunch(exec, s) != cudaSuccess || cudaMemcpyAsync(&hst[l & 1], st, sizeof(DistState), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaEventRecord(ev[l & 1], s) != cudaSuccess) {
      set_error(std::string("distributed CG graph launch: ") + cudaGetErrorString(cudaGetLastError()));
      rc = FEMB_ERR_CUDA;
      break;
    }
    if (l >= 1) {
      cudaEventSynchronize(ev[(l - 1) & 1]);
      stopped = hst[(l - 1) & 1].stop != 0;
    }
  }
  cudaEventRecord(tev[1], s);
  if (!classic) dist_final_check<<<1, 64, 0, s>>>(pe, st, tol);
  DistState* fin = &hst[0];
  if (rc == FEMB_OK && (cudaMemcpyAsync(fin, st, sizeof(DistState), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess)) {
    set_error(std::string("distributed CG final state: ") + cudaGetErrorString(cudaGetLastError()));
    rc = FEMB_ERR_CUDA;
  }
  float ms = 0.f;
  if (rc == FEMB_OK) cudaEventElapsedTime(&ms, tev[0], tev[1]);
  cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  if (rc != FEMB_OK) return rc;
  if (fin->status == 3) {
    set_error("distributed CG: timed out waiting for a peer rank (flag never arrived)");
    return FEMB_ERR_NCCL;
  }
  result_host->iterations = fin->stop ? fin->iterations : max_iter;
  result_host->status = fin->stop ? fin->status : 2;
  result_host->rs = fin->rs_new;
  result_host->loop_ms = ms;
  result_host->index_bytes = 4;
  if (trace && fin->it > 20) {  // average phase times over iterations 10..min(it,TRACE_ITERS)-1 (microseconds)
    static long long h[TRACE_ITERS * 12];
    cudaMemcpy(h, trace, sizeof(h), cudaMemcpyDeviceToHost);
    const int i1 = std::min(fin->it, TRACE_ITERS) - 2;
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 10; i < i1; ++i) {
      const long long* t = h + i * 12;
      if (classic) {
        acc[0] += t[1] - t[0];                 // push
        acc[1] += t[3] - t[2];                 // k1 wait for halo
        acc[2] += t[4] - t[3];                 // k1 body + reduction + remote stores
        acc[3] += t[6] - t[5];                 // k2 wait for all-reduce B
        acc[4] += t[7] - t[6];                 // k2 body
        acc[5] += t[9] - t[8];                 // k3 wait for all-reduce C
        acc[6] += t[10] - t[9];                // k3 body
        acc[7] += (h + (i + 1) * 12)[0] - t[0];  // whole iteration
      } else {
        // slot 10 is stamped after st->it was advanced: row i holds the END of iteration i-1's vector kernel there
        const long long* tn = h + (i + 1) * 12;
        acc[0] += t[3] - t[10];                // SpMV: end of the previous vector kernel -> rows done on CTA 0 (launch gap included)
        acc[1] += t[4] - t[3];                 // SpMV tail of the other CTAs + last CTA: reduction + LL stores to all ranks
        acc[2] += t[5] - t[4];                 // gap until the vector kernel runs
        acc[3] += t[6] - t[5];                 // vector kernel: wait for the all-reduce words of every rank
        acc[4] += tn[10] - t[6];               // vector kernel body + r.r reduction + halo flag
        acc[7] += tn[10] - t[10];              // whole iteration
      }
    }
    const double m = 1e-3 / (i1 - 10);
    if (classic)
      fprintf(stderr, "[femb dist trace] rank %d: push %.1f | k1 wait %.1f body %.1f | k2 wait %.1f body %.1f | k3 wait %.1f body %.1f | iteration %.1f us\n",
              rank, acc[0] * m, acc[1] * m, acc[2] * m, acc[3] * m, acc[4] * m, acc[5] * m, acc[6] * m, acc[7] * m);
    else
      fprintf(stderr, "[femb dist trace] rank %d: spmv %.1f | reduce+send %.1f | gap %.1f | allreduce wait %.1f | vector body %.1f | iteration %.1f us\n",
              rank, acc[0] * m, acc[1] * m, acc[2] * m, acc[3] * m, acc[4] * m, acc[7] * m);
  }
  return FEMB_OK;
}
