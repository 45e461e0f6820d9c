// linalg.cuh -- CSR SpMM (multi-RHS SpMV), the fused "matrix-vector strategy" kernels of
// fracstep.py:438-472, rectangular P2xP1 products, vector kernels and the Krylov recurrences
// (PCG / BiCGStab on up to 3 systems that share one matrix) that replace PETSc Mat/Vec/KSP
// (SURVEY.md N4-N9).
#pragma once
#include "common.cuh"

// ---- Krylov state, device resident ------------------------------------------------------
// One instance per solve; scalars are produced by the last block of the reducing kernel
// (grid_reduce) and consumed by the next kernel on the stream: no host round trip per iteration.
struct KryState {
  double rho[B2_MAXK], alpha[B2_MAXK], beta[B2_MAXK], omega[B2_MAXK];
  double rz[B2_MAXK], bb[B2_MAXK], rr[B2_MAXK], tol2[B2_MAXK];
  int active[B2_MAXK], reason[B2_MAXK], its[B2_MAXK];
  int restart[B2_MAXK];  // BiCGStab: shadow residual became orthogonal to r -> restart with rhat = r
  double rh2[B2_MAXK];   // |rhat|^2
  double rr0[B2_MAXK];   // initial |r|^2 (diagnostics: quality of the initial guess)
  int done, maxit, K, block_rtol;  // block_rtol: tolerance relative to max_k |b_k| (one vector system)
  double rtol, atol;
};

enum {
  FIN_NONE = 0,
  FIN_CG_INIT,
  FIN_CG_PQ,
  FIN_CG_UPDATE,
  FIN_BCGS_INIT,
  FIN_BCGS_V,
  FIN_BCGS_T,
  FIN_BCGS_UPDATE,
  FIN_STORE  // just store totals into st->rr[0..] (generic sums read back by the host)
};

__device__ __forceinline__ bool b2_bad(double v) { return !(fabs(v) <= 1.79e308); }

__device__ inline void kry_check_done(KryState* st) {
  int any = 0;
  for (int k = 0; k < st->K; ++k) any |= st->active[k];
  st->done = !any;
}

__device__ inline void kry_converge_test(KryState* st, int k) {
  if (!st->active[k]) return;
  double rr = st->rr[k];
  if (b2_bad(rr)) {
    st->reason[k] = -9;  // KSP_DIVERGED_NANORINF
    st->active[k] = 0;
  } else if (rr <= st->tol2[k]) {
    st->reason[k] = (rr <= st->atol * st->atol && st->atol * st->atol >= st->rtol * st->rtol * st->bb[k]) ? 3 : 2;
    st->active[k] = 0;
  } else if (st->its[k] >= st->maxit) {
    st->reason[k] = -3;  // KSP_DIVERGED_ITS
    st->active[k] = 0;
  }
}

// Runs in thread 0 of the last block.  `t` holds the reduced sums in the order documented at
// each case.
__device__ inline void kry_finalize(int fin, KryState* st, const double* t) {
  const int K = st->K;
  switch (fin) {
    case FIN_CG_INIT:  // t = rz[K], bb[K], rr[K]
      for (int k = 0; k < K; ++k) {
        st->rz[k] = t[k];
        st->bb[k] = t[K + k];
        st->rr[k] = t[2 * K + k];
        st->rr0[k] = t[2 * K + k];
      }
      for (int k = 0; k < K; ++k) {
        double bref = st->bb[k];
        if (st->block_rtol)
          for (int j = 0; j < K; ++j) bref = bref > t[K + j] ? bref : t[K + j];
        double a2 = st->atol * st->atol, r2 = st->rtol * st->rtol * bref;
        st->tol2[k] = r2 > a2 ? r2 : a2;
        st->its[k] = 0;
        st->reason[k] = 0;
        st->active[k] = 1;
        st->beta[k] = 0.0;
        kry_converge_test(st, k);
      }
      kry_check_done(st);
      break;
    case FIN_CG_PQ:  // t = pq[K]
      for (int k = 0; k < K; ++k) {
        if (!st->active[k]) continue;
        double pq = t[k];
        if (b2_bad(pq)) { st->reason[k] = -9; st->active[k] = 0; }
        else if (pq == 0.0) { st->reason[k] = -5; st->active[k] = 0; }  // KSP_DIVERGED_BREAKDOWN
        else if (pq < 0.0) { st->reason[k] = -8; st->active[k] = 0; }   // KSP_DIVERGED_INDEFINITE_PC/MAT
        else st->alpha[k] = st->rz[k] / pq;
      }
      kry_check_done(st);
      break;
    case FIN_CG_UPDATE:  // t = rz_new[K], rr[K]
      for (int k = 0; k < K; ++k) {
        if (!st->active[k]) continue;
        st->beta[k] = t[k] / st->rz[k];
        st->rz[k] = t[k];
        st->rr[k] = t[K + k];
        st->its[k] += 1;
        kry_converge_test(st, k);
      }
      kry_check_done(st);
      break;
    case FIN_BCGS_INIT:  // t = bb[K], rr[K]
      for (int k = 0; k < K; ++k) {
        st->bb[k] = t[k];
        st->rr[k] = t[K + k];
        st->rr0[k] = t[K + k];
        st->rho[k] = t[K + k];  // rhat = r0
        st->rh2[k] = t[K + k];
        st->restart[k] = 0;
        st->alpha[k] = 1.0;
        st->omega[k] = 1.0;
        st->beta[k] = 0.0;
      }
      for (int k = 0; k < K; ++k) {
        double bref = st->bb[k];
        if (st->block_rtol)
          for (int j = 0; j < K; ++j) bref = bref > t[j] ? bref : t[j];
        double a2 = st->atol * st->atol, r2 = st->rtol * st->rtol * bref;
        st->tol2[k] = r2 > a2 ? r2 : a2;
        st->its[k] = 0;
        st->reason[k] = 0;
        st->active[k] = 1;
        kry_converge_test(st, k);
      }
      kry_check_done(st);
      break;
    case FIN_BCGS_V:  // t = (rhat . v)[K]
      for (int k = 0; k < K; ++k) {
        if (!st->active[k]) continue;
        double d = t[k];
        if (b2_bad(d)) { st->reason[k] = -9; st->active[k] = 0; }
        else if (d == 0.0) { st->reason[k] = -5; st->active[k] = 0; }
        else st->alpha[k] = st->rho[k] / d;
      }
      kry_check_done(st);
      break;
    case FIN_BCGS_T:  // t = (t . s)[K], (t . t)[K]
      for (int k = 0; k < K; ++k) {
        if (!st->active[k]) continue;
        double tt = t[K + k];
        st->omega[k] = tt > 0.0 ? t[k] / tt : 0.0;
      }
      break;
    case FIN_BCGS_UPDATE:  // t = rr[K], rho_new[K]
      for (int k = 0; k < K; ++k) {
        if (!st->active[k]) continue;
        st->rr[k] = t[k];
        st->its[k] += 1;
        kry_converge_test(st, k);
        if (!st->active[k]) continue;
        double rn = t[K + k];
        if (b2_bad(rn)) {
          st->reason[k] = -9;
          st->active[k] = 0;
          continue;
        }
        // (near) breakdown: rhat orthogonal to r, or a vanishing omega -- restart from the current
        // residual (rhat = p = r) instead of giving up (PETSc would return KSP_DIVERGED_BREAKDOWN)
        if (st->omega[k] == 0.0 || st->rho[k] == 0.0 || rn * rn <= 1e-24 * st->rr[k] * st->rh2[k]) {
          st->restart[k] = 1;
          st->rho[k] = st->rr[k];
          st->rh2[k] = st->rr[k];
          st->beta[k] = 0.0;
          continue;
        }
        st->restart[k] = 0;
        st->beta[k] = (rn / st->rho[k]) * (st->alpha[k] / st->omega[k]);
        st->rho[k] = rn;
      }
      kry_check_done(st);
      break;
    case FIN_STORE:
    default:
      break;
  }
}

// Grid-wide sum of N per-thread values followed by the fused scalar update in the last block.  Several ranks:
//   peer path  -- the last block's first warp all-reduces the totals over the ranks through peer memory
//                 (common.cuh: peer_allreduce_warp) and then runs the same scalar update: no extra launch;
//   NCCL path  -- the raw totals are stored and the host enqueues ncclAllReduce + k_kry_finalize next.
struct RedCtl {
  double* out;          // NCCL path: where the raw totals go (nullptr otherwise)
  const PeerDev* peer;  // peer path (nullptr otherwise)
};

template <int N>
__device__ __forceinline__ void reduce_finish(double (&v)[N], double* partials, unsigned* counter, int fin,
                                              KryState* st, RedCtl red_out) {
  static_assert(N <= B2_RED_MAX, "fused reductions carry at most B2_RED_MAX values");
  double total[N];
  if (!grid_reduce<N>(v, partials, counter, total)) return;
  if (red_out.peer != nullptr) {
    __shared__ double sh[N];
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < N; ++i) sh[i] = total[i];
    }
    __syncthreads();
    if (threadIdx.x < 32) peer_allreduce_warp(red_out.peer, sh, N);
    if (threadIdx.x == 0) kry_finalize(fin, st, sh);
  } else if (threadIdx.x == 0) {
    if (red_out.out != nullptr) {
#pragma unroll
      for (int i = 0; i < N; ++i) red_out.out[i] = total[i];
    } else {
      kry_finalize(fin, st, total);
    }
  }
}

__global__ void k_kry_finalize(int fin, KryState* st, const double* __restrict__ totals, int is_init) {
  if (!is_init && st->done) return;
  kry_finalize(fin, st, totals);
}

// ---- halo exchange helpers (multi rank): pack owned entries per neighbour, unpack into ghost slots --
// send buffer layout: neighbour j owns [K*send_off[j], K*send_off[j+1]) as [k][i]
__global__ void k_halo_pack(int n_neighbors, const int64_t* __restrict__ send_off, const int* __restrict__ send_idx,
                            int K, int ld, const double* __restrict__ v, double* __restrict__ buf) {
  const int64_t total = send_off[n_neighbors];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total * K; t += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(t / total);
    const int64_t i = t - (int64_t)k * total;
    int j = 0;
    while (j + 1 < n_neighbors && i >= send_off[j + 1]) ++j;
    const int64_t cnt = send_off[j + 1] - send_off[j];
    buf[K * send_off[j] + k * cnt + (i - send_off[j])] = v[(size_t)k * ld + send_idx[i]];
  }
}
__global__ void k_halo_unpack(int n_neighbors, const int64_t* __restrict__ recv_off, int K, int ld, int n_owned,
                              const double* __restrict__ buf, double* __restrict__ v) {
  const int64_t total = recv_off[n_neighbors];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total * K; t += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(t / total);
    const int64_t i = t - (int64_t)k * total;
    int j = 0;
    while (j + 1 < n_neighbors && i >= recv_off[j + 1]) ++j;
    const int64_t cnt = recv_off[j + 1] - recv_off[j];
    v[(size_t)k * ld + n_owned + i] = buf[K * recv_off[j] + k * cnt + (i - recv_off[j])];
  }
}

// ---- storage ------------------------------------------------------------------------------------
// Vectors: component-major (SoA): component k of a velocity-space vector lives at v + k*ld, ld = dofs
// of the space incl. ghosts.  Square operators (M, K, A on VxV; Ap, MQ on QxQ) and P_i, G_i on VxQ (the
// directions one after the other, vals + i*slots): sliced ELLPACK with 32-row slices ("SELL-32"): entry t
// of row r is at slice_ptr[r/32] + 32*t + r%32, rows padded to the longest row of their slice with
// (col = r, or 0 past the last column, val = 0).  D_i (QxV) is CSR with [nnz][K] values.  One thread
// owns one row; at step t the 32 lanes of a warp read 32 consecutive values and 32 consecutive column
// indices (2 + 1 L1 wavefronts) and, because the host numbers dofs by stencil class (fem._class_order),
// their 32 gathered vector entries are (nearly) consecutive too.  No cross-lane reduction is needed.
// The CSR pattern of create_matrix stays the public face (b2_get_pattern); CSR position p of row r maps
// to the SELL slot slice_ptr[r/32] + 32*(p - rowptr[r]) + r%32 (sell_slot, common.cuh).
// ld_stream (common.cuh): streaming loads for the matrix stream (values, columns)

__global__ void k_sell_slice_len(int n_rows, const int* __restrict__ rowptr, int* __restrict__ slice_entries) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  int n_slices = (n_rows + 31) >> 5;
  if (s >= n_slices) return;
  int mx = 0;
  for (int r = s << 5; r < min(n_rows, (s + 1) << 5); ++r) mx = max(mx, rowptr[r + 1] - rowptr[r]);
  slice_entries[s] = mx << 5;
}

__global__ void k_sell_fill_cols(int n_rows, const int* __restrict__ rowptr, const int* __restrict__ cols,
                                 const int* __restrict__ slice_ptr, int* __restrict__ scols,
                                 int* __restrict__ diag_t, int n_cols) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const int s = row >> 5;
  const int len = (slice_ptr[s + 1] - slice_ptr[s]) >> 5;
  const int start = rowptr[row], n = rowptr[row + 1] - start;
  int dt = -1;
  for (int t = 0; t < len; ++t) {
    int c = t < n ? cols[start + t] : (row < n_cols ? row : 0);  // pads: (a valid column, value 0)
    if (t < n && c == row) dt = t;
    scols[(size_t)slice_ptr[s] + ((size_t)t << 5) + (row & 31)] = c;
  }
  if (diag_t != nullptr) diag_t[row] = dt;
}

// values between CSR order and SELL slots (to_sell: pads are left untouched = 0)
__global__ void k_sell_convert(int n_rows, const int* __restrict__ rowptr, const int* __restrict__ slice_ptr,
                               int to_sell, const double* __restrict__ in, double* __restrict__ out,
                               const double* __restrict__ row_scale) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const int start = rowptr[row], n = rowptr[row + 1] - start;
  const size_t base = (size_t)slice_ptr[row >> 5] + (row & 31);
  const double f = row_scale != nullptr ? 1.0 / row_scale[row] : 1.0;  // undo a row scaling on the way out
  for (int t = 0; t < n; ++t) {
    if (to_sell) out[base + ((size_t)t << 5)] = in[start + t];
    else out[start + t] = in[base + ((size_t)t << 5)] * f;
  }
}

// ---- SELL SpMM: y_k[row] = sum_t vals[slot] * x_k[cols[slot]], k < K ------------------------------
//   DOT == 0: no reduction          DOT == 1: sums[k] = y_k . w_k
//   DOT == 2: sums[k] = y_k . w_k , sums[K+k] = y_k . y_k
// Persistent grid: warp w of the grid walks slices w, w + nwarps, ...  The t-loop is unrolled by 8:
// eight independent (column -> gather) chains per thread keep enough loads in flight to cover HBM
// latency at < 100% occupancy.
// Scheduling: `order` lists the slices tile by tile (all stencil classes of one small spatial tile
// are adjacent in the list, fem.slice_order); a block takes blockDim/32 consecutive list entries at
// a time, so the warps of a block gather from the same neighbourhood of x concurrently and share
// those lines in L1 instead of each pulling them through the L2 fabric.
// MINB: resident blocks per SM the register allocation is bounded for (8 x 256 threads = 32 registers, 6 = 40).
template <int K, int DOT, int BLOCK, bool RS = false, int MINB = 2048 / BLOCK>
__global__ void __launch_bounds__(BLOCK, MINB)
k_spmm(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols,
       const double* __restrict__ vals, const int* __restrict__ order, const double* __restrict__ x, int ld,
       double* __restrict__ y, const double* __restrict__ w, KryState* st, int fin, double* partials,
       unsigned* counter, RedCtl red_out, const double* __restrict__ rscale) {
  if (st != nullptr && st->done) return;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  constexpr int WPB = BLOCK / 32;
  constexpr int UNROLL = 8;
  const int n_slices = (n_rows + 31) >> 5;
  constexpr int ND = DOT == 0 ? 1 : DOT * K;
  // the running dot products live in shared memory between slices: keeping them in registers across
  // the gather loop costs 8-16 registers, i.e. one to three resident blocks per SM on a kernel whose
  // speed is set by the number of loads in flight
  __shared__ double sdots[DOT == 0 ? 1 : ND][DOT == 0 ? 1 : BLOCK];
  if constexpr (DOT > 0) {
#pragma unroll
    for (int i = 0; i < ND; ++i) sdots[i][threadIdx.x] = 0.0;
  }
  for (int i = blockIdx.x * WPB + wib; i < n_slices; i += gridDim.x * WPB) {
    const int s = order != nullptr ? __ldg(order + i) : i;
    const int base = __ldg(slice_ptr + s);
    const int len = (__ldg(slice_ptr + s + 1) - base) >> 5;
    const int row = (s << 5) + lane;
    const int* cp = cols + base + lane;
    const double* vp = vals + base + lane;
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    int t = 0;
    for (; t + UNROLL <= len; t += UNROLL) {
      int c[UNROLL];
      double v[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        c[u] = ld_stream(cp + ((t + u) << 5));
        v[u] = ld_stream(vp + ((t + u) << 5));
      }
      double xv[UNROLL][K];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u)
#pragma unroll
        for (int k = 0; k < K; ++k) xv[u][k] = __ldg(x + (size_t)k * ld + c[u]);
#pragma unroll
      for (int u = 0; u < UNROLL; ++u)
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = fma(v[u], xv[u][k], acc[k]);
    }
    for (; t < len; ++t) {
      const int c = ld_stream(cp + (t << 5));
      const double v = ld_stream(vp + (t << 5));
#pragma unroll
      for (int k = 0; k < K; ++k) acc[k] = fma(v, __ldg(x + (size_t)k * ld + c), acc[k]);
    }
    if (row < n_rows) {
      // epilogue: every load is issued before the first use, so that one memory latency is exposed per slice, not
      // one per dependent step (the row scale alone cost +45 us of 565 when it was loaded, used, and only then w)
      double rs = 1.0, wv[DOT >= 1 ? K : 1];
      if constexpr (RS) rs = __ldg(rscale + row);  // y = D^-1 (A x): left Jacobi preconditioning of BiCGStab, A stored as assembled
      if constexpr (DOT >= 1) {
#pragma unroll
        for (int k = 0; k < K; ++k) wv[k] = __ldg(w + (size_t)k * ld + row);
      }
      if constexpr (RS) {
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] *= rs;
      }
#pragma unroll
      for (int k = 0; k < K; ++k) y[(size_t)k * ld + row] = acc[k];
      if constexpr (DOT >= 1) {
#pragma unroll
        for (int k = 0; k < K; ++k) sdots[k][threadIdx.x] = fma(acc[k], wv[k], sdots[k][threadIdx.x]);
      }
      if constexpr (DOT == 2) {
#pragma unroll
        for (int k = 0; k < K; ++k) sdots[K + k][threadIdx.x] = fma(acc[k], acc[k], sdots[K + k][threadIdx.x]);
      }
    }
  }
  if constexpr (DOT > 0) {
    double dots[ND];
#pragma unroll
    for (int i = 0; i < ND; ++i) dots[i] = sdots[i][threadIdx.x];
    reduce_finish<ND>(dots, partials, counter, fin, st, red_out);
  }
}

// ---- the "matrix-vector strategy" right-hand side in ONE pass (fracstep.py:438-452; the timed block of
// demo/assembly_strategies.py:128-133: A.scale(-0.5); A.axpy(1/dt, M); A.axpy(-nu/2, K); A.mult(u_1, b)) ------------
//   out_k[row] = sum_t (inv_dt M - half_nu K - Ch)[slot] * u_k[cols[slot]] (+ add_k[row]),   Ch = 1/2 C(uab) as
// assembled by k_first_cells with 1/dt = nu = 0.  Three value streams + the column stream are read once; nothing is
// written back to a matrix (the reference rewrites A three times).  The IPCS step itself uses the matrix-free
// action (k_first_cells, MODE & 2); this kernel is the other arm of the micro-benchmark and of its allclose test.
template <int K, int U = 4>
__global__ void __launch_bounds__(256, 4)
k_matvec_rhs(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols, const double* __restrict__ Ch,
             const double* __restrict__ M, const double* __restrict__ Kst, const int* __restrict__ order, double inv_dt,
             double half_nu, const double* __restrict__ u, int ld, const double* __restrict__ add,
             double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int n_slices = (n_rows + 31) >> 5;
  for (int i = blockIdx.x * wpb + wib; i < n_slices; i += gridDim.x * wpb) {
    const int s = order != nullptr ? __ldg(order + i) : i;
    const int base = __ldg(slice_ptr + s);
    const int len = (__ldg(slice_ptr + s + 1) - base) >> 5;
    const int row = (s << 5) + lane;
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    int t = 0;
    for (; t + U <= len; t += U) {
      int cc[U];
      double r[U], xu[U][K];
#pragma unroll
      for (int q = 0; q < U; ++q) {
        const size_t p = (size_t)base + ((size_t)(t + q) << 5) + lane;
        cc[q] = ld_stream(cols + p);
        r[q] = (inv_dt * ld_stream(M + p) - ld_stream(Ch + p)) - half_nu * ld_stream(Kst + p);
      }
#pragma unroll
      for (int q = 0; q < U; ++q)
#pragma unroll
        for (int k = 0; k < K; ++k) xu[q][k] = __ldg(u + (size_t)k * ld + cc[q]);
#pragma unroll
      for (int q = 0; q < U; ++q)
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = fma(r[q], xu[q][k], acc[k]);
    }
    for (; t < len; ++t) {
      const size_t p = (size_t)base + ((size_t)t << 5) + lane;
      const int c = ld_stream(cols + p);
      const double r = (inv_dt * ld_stream(M + p) - ld_stream(Ch + p)) - half_nu * ld_stream(Kst + p);
#pragma unroll
      for (int k = 0; k < K; ++k) acc[k] = fma(r, __ldg(u + (size_t)k * ld + c), acc[k]);
    }
    if (row < n_rows) {
#pragma unroll
      for (int k = 0; k < K; ++k) out[(size_t)k * ld + row] = acc[k] + (add != nullptr ? add[(size_t)k * ld + row] : 0.0);
    }
  }
}

// ---- rectangular products -------------------------------------------------------------------------
// out_k[row] = add_k[row] + scale * sum_t vals[k * slots + slot] * xq[cols[slot]]   (P_i ps, G_i dp)
// on the sliced-ELL form of the V x Q pattern with COMPONENT-MAJOR values (vals + k * slots): the P2 rows have only
// 4-14 entries, so a CSR kernel (4-8 lanes per row, [nnz][K] values) ran at 0.56 of the HBM peak; one thread per row
// over coalesced streams reads (8 K + 4) bytes per slot and nothing else.
template <int K>
__global__ void __launch_bounds__(256, 4)
k_rect_vq_sell(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols, const double* __restrict__ vals,
               int64_t slots, const double* __restrict__ xq, const double* add, int ld, double scale, double* out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n_slices = (n_rows + 31) >> 5;
  for (int s = warp; s < n_slices; s += nwarps) {
    const int base = __ldg(slice_ptr + s);
    const int len = (__ldg(slice_ptr + s + 1) - base) >> 5;
    const int row = (s << 5) + lane;
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
#pragma unroll 4
    for (int t = 0; t < len; ++t) {
      const size_t p = (size_t)base + ((size_t)t << 5) + lane;
      const double xv = __ldg(xq + ld_stream(cols + p));
#pragma unroll
      for (int k = 0; k < K; ++k) acc[k] = fma(ld_stream(vals + (size_t)k * slots + p), xv, acc[k]);
    }
    if (row < n_rows) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const double a = add != nullptr ? add[(size_t)k * ld + row] : 0.0;
        out[(size_t)k * ld + row] = fma(scale, acc[k], a);
      }
    }
  }
}

// out[q] = scale * sum_p sum_k vals[p][k] * xv_k[cols[p]]            (sum_i D_i u_i, CSR [nnz][K] values)
template <int K, int LPR>
__global__ void __launch_bounds__(256)
k_rect_qv(int n_rows, const int* __restrict__ rowptr, const int* __restrict__ cols,
          const double* __restrict__ vals, const double* __restrict__ xv, int ld, double scale,
          const uint8_t* __restrict__ zero_row, double* __restrict__ out) {
  const int lane = threadIdx.x % LPR;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  double acc = 0.0;
  if (row < n_rows) {
    const int end = __ldg(rowptr + row + 1);
    for (int p = __ldg(rowptr + row) + lane; p < end; p += LPR) {
      const int c = __ldg(cols + p);
#pragma unroll
      for (int k = 0; k < K; ++k) acc = fma(__ldg(vals + (size_t)p * K + k), __ldg(xv + (size_t)k * ld + c), acc);
    }
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (row < n_rows && lane == 0) out[row] = (zero_row != nullptr && zero_row[row]) ? 0.0 : scale * acc;
}

// ---- small vector kernels ----------------------------------------------------------------
__global__ void k_lincomb2(int64_t n, double a, const double* x, double b, const double* y, double* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = a * x[i] + b * y[i];
}

// out = a x + b y + c z (+ add)
__global__ void k_lincomb4(int64_t n, double a, const double* x, double b, const double* y, double c, const double* z,
                           const double* add, double* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double v = fma(a, x[i], fma(b, y[i], c * z[i]));
    out[i] = add != nullptr ? v + add[i] : v;
  }
}

__global__ void k_fill(int64_t n, double v, double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = v;
}

// vec[dofs[i]] = values[i]   (set_bc, bcs.py:135-139) on one component
__global__ void k_set_bc(int64_t n, const int* __restrict__ dofs, const double* __restrict__ values,
                         double* __restrict__ vec) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) vec[dofs[i]] = values[i];
}

__global__ void k_mark(int64_t n, const int* __restrict__ dofs, uint8_t* __restrict__ mask) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) mask[dofs[i]] = 1;
}

// strided copies: one direction value family out of [nnz][K] matrix values
__global__ void k_extract(int64_t n, int stride, int comp, const double* __restrict__ src, double* __restrict__ dst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[i * stride + comp];
}
// component-major [K][ld] <-> blocked [n][K] (the layout of solver.u, fracstep.py:698-705)
__global__ void k_to_blocked(int64_t n, int K, int ld, const double* __restrict__ src, double* __restrict__ dst) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n * K; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = t / K;
    int k = (int)(t - i * K);
    dst[t] = src[(size_t)k * ld + i];
  }
}
__global__ void k_from_blocked(int64_t n, int K, int ld, const double* __restrict__ src, double* __restrict__ dst) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n * K; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = t / K;
    int k = (int)(t - i * K);
    dst[(size_t)k * ld + i] = src[t];
  }
}

// dinv[row] = 1 / (diagonal entry of a SELL matrix)
__global__ void k_inv_diag(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ diag_t,
                           const double* __restrict__ vals, double* __restrict__ dinv) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  dinv[row] = 1.0 / vals[sell_slot(slice_ptr, row, diag_t[row])];
}

// assemble_matrix(..., bcs=) semantics on a square SELL matrix (fracstep.py:379, Appendix D): BC rows
// and columns zeroed, unit diagonal.
__global__ void k_apply_bc_rows_cols(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols,
                                     const int* __restrict__ diag_t, const uint8_t* __restrict__ is_bc,
                                     double* __restrict__ vals) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const int s = row >> 5;
  const int len = (slice_ptr[s + 1] - slice_ptr[s]) >> 5;
  const bool rb = is_bc[row];
  for (int t = 0; t < len; ++t) {
    const size_t p = (size_t)slice_ptr[s] + ((size_t)t << 5) + (row & 31);
    const int c = cols[p];
    if (rb || is_bc[c]) vals[p] = (t == diag_t[row]) ? 1.0 : 0.0;
  }
}

// out[k] = sum_i (a_k[i] - b_k[i])^2  (b may be null)
template <int K>
__global__ void __launch_bounds__(256)
k_sqdiff(int64_t n, int ld, const double* __restrict__ a, const double* __restrict__ b, double* out,
         double* partials, unsigned* counter) {
  double s[K];
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double d = a[(size_t)k * ld + i] - (b != nullptr ? b[(size_t)k * ld + i] : 0.0);
      s[k] = fma(d, d, s[k]);
    }
  }
  double total[K];
  if (grid_reduce<K>(s, partials, counter, total) && threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) out[k] = total[k];
  }
}

// out[0] = sum_i x[i] ; out[1] = sum_i w[i]*x[i] (w may be null)
__global__ void __launch_bounds__(256)
k_sums(int64_t n, const double* __restrict__ x, const double* __restrict__ w, double* out,
       double* partials, unsigned* counter) {
  double s[2] = {0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double v = x[i];
    s[0] += v;
    if (w != nullptr) s[1] = fma(w[i], v, s[1]);
  }
  double total[2];
  if (grid_reduce<2>(s, partials, counter, total) && threadIdx.x == 0) {
    out[0] = total[0];
    out[1] = total[1];
  }
}

// out[0] = sum_k sum_i a_k[i] * b_k[i]
__global__ void __launch_bounds__(256)
k_dot_all(int64_t n, int K, int ld, const double* __restrict__ a, const double* __restrict__ b, double* out,
          double* partials, unsigned* counter) {
  double s[1] = {0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    for (int k = 0; k < K; ++k) s[0] = fma(a[(size_t)k * ld + i], b[(size_t)k * ld + i], s[0]);
  double total[1];
  if (grid_reduce<1>(s, partials, counter, total) && threadIdx.x == 0) out[0] = total[0];
}

// x[i] -= sums[which] * inv_norm   (null-space removal :573-574 with which=0, inv_norm = 1/n;
// mass-mean removal :579-591 with which=1, inv_norm = 1/vol); optionally y = z + x (ps = p + dp, :604)
__global__ void k_shift(int64_t n, double* __restrict__ x, const double* __restrict__ sums, int which,
                        double inv_norm, const double* __restrict__ z, double* __restrict__ y) {
  const double s = sums[which] * inv_norm;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double v = x[i] - s;
    x[i] = v;
    if (y != nullptr) y[i] = z[i] + v;
  }
}

// ---- PCG (Jacobi) on K systems sharing one matrix ---------------------------------------------
// init: r = b - q (q = A x0, or r = b and x = 0 when no initial guess), p = dinv r;
//       sums rz, bb, rr
template <int K>
__global__ void __launch_bounds__(256)
k_cg_init(int64_t n, int ld, const double* __restrict__ b, const double* __restrict__ q,
          const double* __restrict__ dinv, double* __restrict__ x, double* __restrict__ r,
          double* __restrict__ p, KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  double s[3 * K];
#pragma unroll
  for (int i = 0; i < 3 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const size_t j = (size_t)k * ld + i;
      const double bv = b[j];
      double rv = bv;
      if (q != nullptr) rv -= q[j];
      else x[j] = 0.0;
      const double zv = di * rv;
      r[j] = rv;
      p[j] = zv;
      s[k] = fma(rv, zv, s[k]);
      s[K + k] = fma(bv, bv, s[K + k]);
      s[2 * K + k] = fma(rv, rv, s[2 * K + k]);
    }
  }
  reduce_finish<3 * K>(s, partials, counter, FIN_CG_INIT, st, red_out);
}

// x += alpha p ; r -= alpha q ; sums rz' = r.dinv r , rr = r.r
template <int K>
__global__ void __launch_bounds__(256)
k_cg_update(int64_t n, int ld, const double* __restrict__ p, const double* __restrict__ q,
            const double* __restrict__ dinv, double* __restrict__ x, double* __restrict__ r,
            KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  if (st->done) return;
  double alpha[K];
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    alpha[k] = st->alpha[k];
  }
  double s[2 * K];
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t j = (size_t)k * ld + i;
      x[j] = fma(alpha[k], p[j], x[j]);
      const double rv = fma(-alpha[k], q[j], r[j]);
      r[j] = rv;
      s[k] = fma(rv * di, rv, s[k]);
      s[K + k] = fma(rv, rv, s[K + k]);
    }
  }
  reduce_finish<2 * K>(s, partials, counter, FIN_CG_UPDATE, st, red_out);
}

// p = dinv r + beta p
template <int K>
__global__ void __launch_bounds__(256)
k_cg_p(int64_t n, int ld, const double* __restrict__ r, const double* __restrict__ dinv,
       double* __restrict__ p, const KryState* st) {
  if (st->done) return;
  double beta[K];
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    beta[k] = st->beta[k];
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t j = (size_t)k * ld + i;
      p[j] = fma(beta[k], p[j], di * r[j]);
    }
  }
}

// ---- BiCGStab on K systems sharing one (already left-preconditioned, row-scaled) matrix ----------
// init: r = dinv b - q (or r = dinv b, x = 0); rhat = r; p = r; sums bb = |dinv b|^2, rr
template <int K>
__global__ void __launch_bounds__(256)
k_bcgs_init(int64_t n, int ld, const double* __restrict__ b, const double* __restrict__ q,
            const double* __restrict__ dinv, double* __restrict__ x, double* __restrict__ r,
            double* __restrict__ rhat, double* __restrict__ p, KryState* st, double* partials,
            unsigned* counter, RedCtl red_out) {
  double s[2 * K];
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const size_t j = (size_t)k * ld + i;
      const double bv = di * b[j];
      double rv = bv;
      if (q != nullptr) rv -= q[j];
      else x[j] = 0.0;
      r[j] = rv;
      rhat[j] = rv;
      p[j] = rv;
      s[k] = fma(bv, bv, s[k]);
      s[K + k] = fma(rv, rv, s[K + k]);
    }
  }
  reduce_finish<2 * K>(s, partials, counter, FIN_BCGS_INIT, st, red_out);
}

// s = r - alpha v   (in place in r)
template <int K>
__global__ void __launch_bounds__(256)
k_bcgs_s(int64_t n, int ld, const double* __restrict__ v, double* __restrict__ r, const KryState* st) {
  if (st->done) return;
  double alpha[K];
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    alpha[k] = st->alpha[k];
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t j = (size_t)k * ld + i;
      r[j] = fma(-alpha[k], v[j], r[j]);
    }
  }
}

// x += alpha p + omega s ; r = s - omega t ; sums rr, rho' = rhat . r
template <int K>
__global__ void __launch_bounds__(256)
k_bcgs_update(int64_t n, int ld, const double* __restrict__ p, const double* __restrict__ t,
              const double* __restrict__ rhat, double* __restrict__ x, double* __restrict__ r,
              KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  if (st->done) return;
  double alpha[K], omega[K];
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    alpha[k] = st->alpha[k];
    omega[k] = st->omega[k];
  }
  double s[2 * K];
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t j = (size_t)k * ld + i;
      const double sv = r[j];
      x[j] = fma(alpha[k], p[j], fma(omega[k], sv, x[j]));
      const double rv = fma(-omega[k], t[j], sv);
      r[j] = rv;
      s[k] = fma(rv, rv, s[k]);
      s[K + k] = fma(rhat[j], rv, s[K + k]);
    }
  }
  reduce_finish<2 * K>(s, partials, counter, FIN_BCGS_UPDATE, st, red_out);
}

// p = r + beta (p - omega v);  on a restart: rhat = p = r
template <int K>
__global__ void __launch_bounds__(256)
k_bcgs_p(int64_t n, int ld, const double* __restrict__ r, const double* __restrict__ v,
         double* __restrict__ p, double* __restrict__ rhat, const KryState* st) {
  if (st->done) return;
  double beta[K], omega[K];
  bool act[K], rst[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    rst[k] = st->restart[k];
    beta[k] = st->beta[k];
    omega[k] = st->omega[k];
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t j = (size_t)k * ld + i;
      if (rst[k]) {
        const double rv = r[j];
        rhat[j] = rv;
        p[j] = rv;
      } else {
        p[j] = fma(beta[k], fma(-omega[k], v[j], p[j]), r[j]);
      }
    }
  }
}

// ---- Chebyshev iteration (Jacobi-preconditioned) on K systems sharing one SPD matrix -----------------
// The spectrum of D^-1 M of a mass matrix is bounded by the element-level generalised eigenvalues
// (Wathen 1987), which the host computes once from the reference tables: the recurrence scalars are
// data independent, so an iteration needs NO reduction (multi-GPU: no all-reduce).
// init: r = b - q (or b), d = dinv r / theta ; sums bb, rr (stored to out[0..2K))
template <int K>
__global__ void __launch_bounds__(256)
k_cheb_init(int64_t n, int ld, const double* __restrict__ b, const double* __restrict__ q,
            const double* __restrict__ dinv, double inv_theta, double* __restrict__ x, double* __restrict__ r,
            double* __restrict__ d, double* out, double* partials, unsigned* counter) {
  double s[2 * K];
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i] * inv_theta;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const size_t j = (size_t)k * ld + i;
      const double bv = b[j];
      double rv = bv;
      if (q != nullptr) rv -= q[j];
      else x[j] = 0.0;
      r[j] = rv;
      d[j] = di * rv;
      s[k] = fma(bv, bv, s[k]);
      s[K + k] = fma(rv, rv, s[K + k]);
    }
  }
  double total[2 * K];
  if (grid_reduce<2 * K>(s, partials, counter, total) && threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < 2 * K; ++i) out[i] = total[i];
  }
}

// x += d ; r -= q ; d = c1 d + c2 dinv r ; NORM: out[k] = |r_k|^2
template <int K, bool NORM>
__global__ void __launch_bounds__(256)
k_cheb_update(int64_t n, int ld, const double* __restrict__ q, const double* __restrict__ dinv, double c1, double c2,
              double* __restrict__ x, double* __restrict__ r, double* __restrict__ d, double* out, double* partials,
              unsigned* counter) {
  double s[K];
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = c2 * dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const size_t j = (size_t)k * ld + i;
      const double dv = d[j];
      x[j] += dv;
      const double rv = r[j] - q[j];
      r[j] = rv;
      d[j] = fma(c1, dv, di * rv);
      if (NORM) s[k] = fma(rv, rv, s[k]);
    }
  }
  if constexpr (NORM) {
    double total[K];
    if (grid_reduce<K>(s, partials, counter, total) && threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) out[k] = total[k];
    }
  }
}
