// gmres.cuh -- restarted, left-preconditioned GMRES(m) (PETSc KSPGMRES with classical Gram-Schmidt) on up to 3
// systems that share one matrix.  The components advance in lockstep: one SpMM per Arnoldi step for all of them
// (k_spmm with the D^-1 row-scale epilogue), then
//   k_gmres_dots   h_{i,j} = v_i . w   for i <= j, every component, one launch, deterministic reduction;
//   k_gmres_orth   w -= sum_i h_{i,j} v_i and |w|^2 in the same pass; the last block runs the Givens update of
//                  column j, the residual estimate |g_{j+1}| and the convergence test (gmres_fin_orth);
//   k_gmres_scale  v_{j+1} = w / h_{j+1,j};
// and at the end of a cycle k_gmres_backsolve (H y = g, one thread per component) and k_gmres_update_x
// (x += V y).  Each component keeps its own Hessenberg matrix, rotations, g and number of steps: one that stops
// inside a cycle is updated with its own length when the cycle closes.  Reasons, iteration counts and the
// tolerance live in KryState, shared with CG and BiCGStab.
#pragma once
#include "linalg.cuh"

#define B2_GMRES_MAXM 100  // largest restart length (ksp_gmres_restart)
#define B2_GMRES_HAPTOL 1e-30  // PETSc's gmres->haptol

struct GmresState {
  double H[B2_MAXK][B2_GMRES_MAXM + 1][B2_GMRES_MAXM];  // Hessenberg columns, rotated in place: R of H = Q R
  double cs[B2_MAXK][B2_GMRES_MAXM], sn[B2_MAXK][B2_GMRES_MAXM];
  double g[B2_MAXK][B2_GMRES_MAXM + 1];  // rotated right-hand side |r_0| e_1
  double y[B2_MAXK][B2_GMRES_MAXM];
  double hcol[(B2_GMRES_MAXM + 1) * B2_MAXK];  // totals of k_gmres_dots, [i * K + k]
  double tot[2 * B2_MAXK];                     // totals of the norm reductions
  double nrm[B2_MAXK];                         // divisor of the newest basis vector
  int steps[B2_MAXK];                          // Arnoldi steps of the current cycle
  int ny[B2_MAXK];                             // length of y for k_gmres_update_x (0: nothing to add)
};

enum { GM_FIN_INIT = 0, GM_FIN_RESTART = 1, GM_FIN_ORTH = 2 };

// Totals t = |D^-1 b|^2[K], |r|^2[K] of k_gmres_residual: tolerance and state (init) or the convergence test of the
// true residual (restart); g_0 = |r| and the divisor of v_0 for every active component
__device__ inline void gmres_fin_residual(GmresState* gs, KryState* st, const double* t, int init) {
  const int K = st->K;
  if (init) {
    kry_finalize(FIN_BCGS_INIT, st, t);  // bb, rr, rr0, tol2 (b200_block_rtol), its = 0, reason, active, done
  } else {
    for (int k = 0; k < K; ++k) {
      if (!st->active[k]) continue;
      st->rr[k] = t[K + k];
      kry_converge_test(st, k);
    }
    kry_check_done(st);
  }
  for (int k = 0; k < K; ++k) {
    gs->steps[k] = 0;
    const double beta = sqrt(st->rr[k]);
    gs->g[k][0] = beta;
    gs->nrm[k] = beta;
  }
}

// Column j of every active component: H[:, j] (+)= hcol; on the last Gram-Schmidt pass also h_{j+1,j} = |w| (t[k]),
// the earlier rotations, the new rotation, g and the convergence test.  PETSc's happy-breakdown test (tt < min(|tt /
// g_j|, haptol)) stops the component: converged when the estimate meets the tolerance, KSP_DIVERGED_BREAKDOWN
// otherwise.
__device__ inline void gmres_fin_orth(GmresState* gs, KryState* st, const double* t, int j, int first, int last) {
  const int K = st->K;
  for (int k = 0; k < K; ++k) {
    if (!st->active[k]) continue;
    double(*H)[B2_GMRES_MAXM] = gs->H[k];
    for (int i = 0; i <= j; ++i) H[i][j] = (first ? 0.0 : H[i][j]) + gs->hcol[i * K + k];
    if (!last) continue;
    const double tt = sqrt(t[k]);
    double hapbnd = fabs(tt / gs->g[k][j]);
    if (hapbnd > B2_GMRES_HAPTOL) hapbnd = B2_GMRES_HAPTOL;
    const bool happy = tt < hapbnd;
    for (int i = 0; i < j; ++i) {
      const double a = H[i][j], b = H[i + 1][j];
      H[i][j] = gs->cs[k][i] * a + gs->sn[k][i] * b;
      H[i + 1][j] = gs->cs[k][i] * b - gs->sn[k][i] * a;
    }
    const double hjj = H[j][j];
    const double d = sqrt(hjj * hjj + tt * tt);
    st->its[k] += 1;
    gs->nrm[k] = tt;
    if (d == 0.0) {  // column j is zero: it cannot enter the solution
      gs->steps[k] = j;
      st->reason[k] = -5;
      st->active[k] = 0;
      continue;
    }
    gs->steps[k] = j + 1;
    const double cj = hjj / d, sj = tt / d;
    gs->cs[k][j] = cj;
    gs->sn[k][j] = sj;
    H[j][j] = d;
    gs->g[k][j + 1] = -sj * gs->g[k][j];
    gs->g[k][j] = cj * gs->g[k][j];
    st->rr[k] = gs->g[k][j + 1] * gs->g[k][j + 1];
    kry_converge_test(st, k);
    if (st->active[k] && happy) {
      st->reason[k] = -5;
      st->active[k] = 0;
    }
  }
  kry_check_done(st);
}

// finalize of the several-rank path, after the host all-reduced the totals
__global__ void k_gmres_fin(int fin, GmresState* gs, KryState* st, int j, int first, int last) {
  if (fin != GM_FIN_INIT && st->done) return;
  if (fin == GM_FIN_ORTH) gmres_fin_orth(gs, st, gs->tot, j, first, last);
  else gmres_fin_residual(gs, st, gs->tot, fin == GM_FIN_INIT);
}

// v0 = D^-1 b - q (q = D^-1 A x), or v0 = D^-1 b and x = 0 without an initial guess; sums |D^-1 b|^2, |v0|^2.
// init = 0 (restart): only the active components.
template <int K>
__global__ void __launch_bounds__(256)
k_gmres_residual(int64_t n, int ld, const double* __restrict__ b, const double* __restrict__ q,
                 const double* __restrict__ dinv, double* __restrict__ x, double* __restrict__ v0, int init,
                 int fin_here, GmresState* gs, KryState* st, double* partials, unsigned* counter) {
  if (!init && st->done) return;
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) act[k] = init || st->active[k];
  double s[2 * K];
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) s[i] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double di = dinv[i];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t jj = (size_t)k * ld + i;
      const double bv = di * b[jj];
      double rv = bv;
      if (q != nullptr) rv -= q[jj];
      else x[jj] = 0.0;
      v0[jj] = rv;
      s[k] = fma(bv, bv, s[k]);
      s[K + k] = fma(rv, rv, s[K + k]);
    }
  }
  double total[2 * K];
  if (grid_reduce<2 * K>(s, partials, counter, total) && threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < 2 * K; ++i) gs->tot[i] = total[i];
    if (fin_here) gmres_fin_residual(gs, st, total, init);
  }
}

// h_{i,j} = v_i . w (i <= j) for every active component.  Basis vectors are taken CH at a time (CH * K running sums
// per thread, w re-read once per chunk); each block leaves its (j+1) K sums in `partials`, and the last block adds
// them up in block order (no floating-point atomics: the same bits on every run).
template <int K, int CH>
__global__ void __launch_bounds__(512)
k_gmres_dots(int64_t n, int ld, const double* __restrict__ V, int j, const double* __restrict__ w, GmresState* gs,
             const KryState* st, double* partials, unsigned* counter) {
  if (st->done) return;
  __shared__ double swarp[CH * K][16];
  __shared__ double sblk[(B2_GMRES_MAXM + 1) * B2_MAXK];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) act[k] = st->active[k];
  const int nb = j + 1, N = nb * K;
  for (int c0 = 0; c0 < nb; c0 += CH) {
    double acc[CH][K];
#pragma unroll
    for (int u = 0; u < CH; ++u)
#pragma unroll
      for (int k = 0; k < K; ++k) acc[u][k] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (!act[k]) continue;
        const double wv = w[(size_t)k * ld + i];
#pragma unroll
        for (int u = 0; u < CH; ++u)
          if (c0 + u < nb) acc[u][k] = fma(V[((size_t)(c0 + u) * K + k) * ld + i], wv, acc[u][k]);
      }
    }
#pragma unroll
    for (int u = 0; u < CH; ++u)
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const double s = warp_sum(acc[u][k]);
        if (lane == 0) swarp[u * K + k][warp] = s;
      }
    __syncthreads();
    if (threadIdx.x < CH * K && c0 * K + (int)threadIdx.x < N) {
      double s = 0.0;
      for (int q = 0; q < nwarp; ++q) s += swarp[threadIdx.x][q];
      const int u = threadIdx.x / K, k = threadIdx.x - u * K;
      sblk[(c0 + u) * K + k] = s;
    }
    __syncthreads();
  }
  for (int t = threadIdx.x; t < N; t += blockDim.x) partials[(size_t)blockIdx.x * N + t] = sblk[t];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int t = threadIdx.x; t < N; t += blockDim.x) {
    // four interleaved running sums keep loads in flight; combined in a fixed order
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    unsigned bk = 0;
    for (; bk + 4 <= gridDim.x; bk += 4) {
      a0 += __ldcg(&partials[(size_t)bk * N + t]);
      a1 += __ldcg(&partials[(size_t)(bk + 1) * N + t]);
      a2 += __ldcg(&partials[(size_t)(bk + 2) * N + t]);
      a3 += __ldcg(&partials[(size_t)(bk + 3) * N + t]);
    }
    for (; bk < gridDim.x; ++bk) a0 += __ldcg(&partials[(size_t)bk * N + t]);
    gs->hcol[t] = (a0 + a1) + (a2 + a3);
  }
  if (threadIdx.x == 0) *counter = 0u;
}

// w -= sum_{i<=j} h_{i,j} v_i and |w|^2, active components; last block: gmres_fin_orth (one rank) or the raw totals
template <int K>
__global__ void __launch_bounds__(256)
k_gmres_orth(int64_t n, int ld, const double* __restrict__ V, int j, double* __restrict__ w, int first, int last,
             int fin_here, GmresState* gs, KryState* st, double* partials, unsigned* counter) {
  if (st->done) return;
  __shared__ double sh[B2_MAXK][B2_GMRES_MAXM + 1];
  bool act[K];
#pragma unroll
  for (int k = 0; k < K; ++k) act[k] = st->active[k];
  for (int t = threadIdx.x; t < (j + 1) * K; t += blockDim.x) sh[t % K][t / K] = gs->hcol[t];
  __syncthreads();
  double s[K];
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = 0.0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (!act[k]) continue;
      const size_t jj = (size_t)k * ld + r;
      double wv = w[jj];
#pragma unroll 4
      for (int i = 0; i <= j; ++i) wv = fma(-sh[k][i], V[((size_t)i * K + k) * ld + r], wv);
      w[jj] = wv;
      s[k] = fma(wv, wv, s[k]);
    }
  }
  double total[K];
  if (grid_reduce<K>(s, partials, counter, total) && threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) gs->tot[k] = total[k];
    if (fin_here) gmres_fin_orth(gs, st, total, j, first, last);
  }
}

// v /= nrm, active components
template <int K>
__global__ void __launch_bounds__(256)
k_gmres_scale(int64_t n, int ld, double* __restrict__ v, const GmresState* gs, const KryState* st) {
  if (st->done) return;
  bool act[K];
  double inv[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    act[k] = st->active[k];
    inv[k] = 1.0 / gs->nrm[k];
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (act[k]) v[(size_t)k * ld + i] *= inv[k];
  }
}

// R y = g over the steps of the cycle, one thread per component; the steps are consumed (a second call adds nothing)
__global__ void k_gmres_backsolve(GmresState* gs, int K) {
  const int k = threadIdx.x;
  if (k >= K) return;
  const int s = gs->steps[k];
  for (int i = s - 1; i >= 0; --i) {
    double t = gs->g[k][i];
    for (int l = i + 1; l < s; ++l) t -= gs->H[k][i][l] * gs->y[k][l];
    gs->y[k][i] = t / gs->H[k][i][i];
  }
  gs->ny[k] = s;
  gs->steps[k] = 0;
}

// x += sum_{i < ny} y_i v_i per component
template <int K>
__global__ void __launch_bounds__(256)
k_gmres_update_x(int64_t n, int ld, const double* __restrict__ V, double* __restrict__ x, const GmresState* gs) {
  __shared__ double sy[B2_MAXK][B2_GMRES_MAXM];
  int ny[K];
#pragma unroll
  for (int k = 0; k < K; ++k) ny[k] = gs->ny[k];
  for (int t = threadIdx.x; t < K * B2_GMRES_MAXM; t += blockDim.x) {
    const int k = t / B2_GMRES_MAXM, i = t - k * B2_GMRES_MAXM;
    if (i < ny[k]) sy[k][i] = gs->y[k][i];
  }
  __syncthreads();
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (ny[k] == 0) continue;
      const size_t jj = (size_t)k * ld + r;
      double xv = x[jj];
#pragma unroll 4
      for (int i = 0; i < ny[k]; ++i) xv = fma(sy[k][i], V[((size_t)i * K + k) * ld + r], xv);
      x[jj] = xv;
    }
  }
}
