// mg.cuh -- kernels of the geometric multigrid preconditioner for the pressure Poisson problem
// (the device-side answer to the reference's forced direct solve of the singular system,
// /root/reference/src/oasisx/fracstep.py:562-578, which cannot scale to 10^6 unknowns), and the
// PCG recurrences with an explicit preconditioned residual z = V(r).
#pragma once
#include "linalg.cuh"

// one damped-Jacobi sweep on a SELL-32 operator: x_out = x_in + omega * dinv * (b - A x_in);
// RESID: r_out = b - A x_in instead (x_out unused)
template <bool RESID>
__global__ void __launch_bounds__(256)
k_mg_sweep(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols,
           const double* __restrict__ vals, const double* __restrict__ dinv, const double* __restrict__ b,
           const double* __restrict__ x_in, double omega, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n_slices = (n_rows + 31) >> 5;
  for (int s = warp; s < n_slices; s += nwarps) {
    const int base = __ldg(slice_ptr + s);
    const int len = (__ldg(slice_ptr + s + 1) - base) >> 5;
    const int row = (s << 5) + lane;
    double acc = 0.0;
#pragma unroll 4
    for (int t = 0; t < len; ++t) {
      const int c = ld_stream(cols + base + lane + (t << 5));
      acc = fma(ld_stream(vals + base + lane + (t << 5)), __ldg(x_in + c), acc);
    }
    if (row < n_rows) {
      const double r = b[row] - acc;
      out[row] = RESID ? r : fma(omega * dinv[row], r, x_in[row]);
    }
  }
}

// the LAST post-smoothing sweep of the fine level with the PCG scalar product fused in: z = x_in + omega D^-1 (r - A x_in)
// and sum r.z (fin = FIN_CGZ_RZ0 / FIN_CGZ_RZ) -- one launch and one pass over r and z less per iteration
__global__ void __launch_bounds__(256)
k_mg_sweep_rz(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols, const double* __restrict__ vals,
              const double* __restrict__ dinv, const double* __restrict__ b, const double* __restrict__ x_in, double omega,
              double* __restrict__ out, int fin, KryState* st, double* partials, unsigned* counter, RedCtl red_out);

// x = omega * dinv * b  (first sweep from a zero initial guess)
__global__ void k_mg_first(int64_t n, const double* __restrict__ dinv, const double* __restrict__ b, double omega,
                           double* __restrict__ x) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] = omega * dinv[i] * b[i];
}

// restriction with the first smoothing sweep of the coarse level fused in: b_c = R r_f, x_c = omega D_c^-1 b_c
// (PARTIAL: on several ranks b_c is a partial sum -- the caller then all-reduces b_c and launches k_mg_first)
__global__ void __launch_bounds__(256)
k_mg_restrict(int n_rows, const int* __restrict__ rowptr, const int* __restrict__ cols, const double* __restrict__ vals,
              const double* __restrict__ rf, const double* __restrict__ dinv, double omega, double* __restrict__ bc,
              double* __restrict__ xc) {
  constexpr int LPR = 8;
  const int lane = threadIdx.x % LPR;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  double acc = 0.0;
  if (row < n_rows) {
    const int end = __ldg(rowptr + row + 1);
    for (int p = __ldg(rowptr + row) + lane; p < end; p += LPR) acc = fma(__ldg(vals + p), __ldg(rf + __ldg(cols + p)), acc);
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (row < n_rows && lane == 0) {
    bc[row] = acc;
    if (xc != nullptr) xc[row] = omega * dinv[row] * acc;
  }
}

// x_f += P x_c: nested P1 prolongations have at most d + 1 entries per row -- one thread per row
__global__ void __launch_bounds__(256)
k_mg_prolong(int n_rows, const int* __restrict__ rowptr, const int* __restrict__ cols, const double* __restrict__ vals,
             const double* __restrict__ xc, double* __restrict__ xf) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  double acc = xf[row];
  const int end = __ldg(rowptr + row + 1);
  for (int p = __ldg(rowptr + row); p < end; ++p) acc = fma(__ldg(vals + p), __ldg(xc + __ldg(cols + p)), acc);
  xf[row] = acc;
}

// ---- the small end of the hierarchy in one kernel ------------------------------------------------
// Levels with a few thousand unknowns are pure launch latency when every sweep is its own kernel
// (~60 launches per cycle).  One 1024-thread block runs the whole sub-cycle from level l0 down to the
// coarsest level and back, with block barriers between the phases.
struct MgDev {
  int n, n_fine;
  const int *slice_ptr, *cols;
  const double *A, *dinv;
  double *x, *b, *tmp;
  const int *Pptr, *Pcol;
  const double* Pval;  // rows: dofs of the finer level, cols: this level
  const int *Rptr, *Rcol;
  const double* Rval;  // rows: this level, cols: dofs of the finer level
  double omega;        // damping of an algebraic level; 0: the kernel's omega argument (geometric levels)
};

__device__ __forceinline__ double mg_row_dot(const MgDev& L, int row, const double* x) {
  const int s = row >> 5;
  const int base = L.slice_ptr[s];
  const int len = (L.slice_ptr[s + 1] - base) >> 5;
  double acc = 0.0;
  for (int t = 0; t < len; ++t) {
    const size_t p = (size_t)base + ((size_t)t << 5) + (row & 31);
    acc = fma(L.A[p], x[L.cols[p]], acc);
  }
  return acc;
}

// n_sweeps damped-Jacobi sweeps on level L for L.b, result pointer returned (x and tmp ping-pong)
__device__ double* mg_block_sweeps(const MgDev& L, double* x, double* tmp, int n_sweeps, bool from_zero, double omega) {
  int s = 0;
  if (from_zero && n_sweeps > 0) {
    for (int r = threadIdx.x; r < L.n; r += blockDim.x) x[r] = omega * L.dinv[r] * L.b[r];
    __syncthreads();
    s = 1;
  }
  for (; s < n_sweeps; ++s) {
    for (int r = threadIdx.x; r < L.n; r += blockDim.x) tmp[r] = fma(omega * L.dinv[r], L.b[r] - mg_row_dot(L, r, x), x[r]);
    __syncthreads();
    double* t = x;
    x = tmp;
    tmp = t;
  }
  return x;
}

__global__ void __launch_bounds__(1024)
k_mg_small_cycle(const MgDev* __restrict__ lv, int l0, int l_last, int pre, int post, int coarse, double omega,
                 double** result) {
  __shared__ double* xs[16];
  __shared__ double* ts[16];
  // down
  for (int l = l0; l <= l_last; ++l) {
    const MgDev L = lv[l];
    double* x = mg_block_sweeps(L, L.x, L.tmp, l == l_last ? coarse : pre, true, L.omega > 0.0 ? L.omega : omega);
    double* tmp = (x == L.x) ? L.tmp : L.x;
    if (threadIdx.x == 0) { xs[l - l0] = x; ts[l - l0] = tmp; }
    if (l < l_last) {
      for (int r = threadIdx.x; r < L.n; r += blockDim.x) tmp[r] = L.b[r] - mg_row_dot(L, r, x);  // residual
      __syncthreads();
      const MgDev C = lv[l + 1];
      for (int r = threadIdx.x; r < C.n; r += blockDim.x) {  // b_{l+1} = R r
        double acc = 0.0;
        for (int p = C.Rptr[r]; p < C.Rptr[r + 1]; ++p) acc = fma(C.Rval[p], tmp[C.Rcol[p]], acc);
        C.b[r] = acc;
      }
    }
    __syncthreads();
  }
  // up
  for (int l = l_last - 1; l >= l0; --l) {
    const MgDev L = lv[l];
    const MgDev C = lv[l + 1];
    double* x = xs[l - l0];
    double* tmp = ts[l - l0];
    const double* xc = xs[l + 1 - l0];
    for (int r = threadIdx.x; r < L.n; r += blockDim.x) {  // x += P xc
      double acc = x[r];
      for (int p = C.Pptr[r]; p < C.Pptr[r + 1]; ++p) acc = fma(C.Pval[p], xc[C.Pcol[p]], acc);
      x[r] = acc;
    }
    __syncthreads();
    x = mg_block_sweeps(L, x, tmp, post, false, L.omega > 0.0 ? L.omega : omega);
    if (threadIdx.x == 0) xs[l - l0] = x;
    __syncthreads();
  }
  if (threadIdx.x == 0) *result = xs[0];
}

// ---- exact solve on the coarsest used level -------------------------------------------------------
// A level with a few thousand unknowns is solved exactly by ONE dense mat-vec with the precomputed
// inverse of (A_l + alpha e e^T) (A_l is the singular Neumann stiffness, e = ones; the shift makes it
// SPD and leaves the action on mean-free right-hand sides unchanged).  2197^2 doubles = 39 MB read by
// the whole machine (~10 us) replaces ~30 block-synchronised phases of the single-block sub-cycle
// (~190 us), and the V-cycle stays a symmetric positive definite preconditioner.
__global__ void k_dense_from_sell(int n, const int* __restrict__ slice_ptr, const int* __restrict__ cols,
                                  const double* __restrict__ vals, double alpha, double* __restrict__ a) {
  const int row = blockIdx.x;
  for (int j = threadIdx.x; j < n; j += blockDim.x) a[(size_t)row * n + j] = alpha;
  __syncthreads();
  const int base = slice_ptr[row >> 5];
  const int len = (slice_ptr[(row >> 5) + 1] - base) >> 5;
  for (int t = threadIdx.x; t < len; t += blockDim.x) {
    const size_t p = (size_t)base + ((size_t)t << 5) + (row & 31);
    if (vals[p] != 0.0) atomicAdd(&a[(size_t)row * n + cols[p]], vals[p]);  // pads: (col = row, val = 0)
  }
}

// in-place Gauss-Jordan inversion of an SPD matrix (no pivoting needed), step k in two launches
__global__ void k_gj_pivot(int n, int k, const double* __restrict__ a, double* __restrict__ rowk, double* __restrict__ colk) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rowk[i] = a[(size_t)k * n + i];
  colk[i] = a[(size_t)i * n + k];
}

__global__ void k_gj_update(int n, int k, double* __restrict__ a, const double* __restrict__ rowk, const double* __restrict__ colk) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j >= n) return;
  const double p = 1.0 / rowk[k];
  double* e = a + (size_t)i * n + j;
  if (i == k) *e = (j == k) ? p : rowk[j] * p;
  else if (j == k) *e = -colk[i] * p;
  else *e = fma(-colk[i] * p, rowk[j], *e);
}

// y = B b, B dense n x n row-major: one warp per row
__global__ void __launch_bounds__(256)
k_dense_matvec(int n, const double* __restrict__ B, const double* __restrict__ b, double* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const double* r = B + (size_t)row * n;
  double acc0 = 0.0, acc1 = 0.0;
  int j = lane;
  for (; j + 32 < n; j += 64) {
    acc0 = fma(ld_stream(r + j), __ldg(b + j), acc0);
    acc1 = fma(ld_stream(r + j + 32), __ldg(b + j + 32), acc1);
  }
  if (j < n) acc0 = fma(ld_stream(r + j), __ldg(b + j), acc0);
  double acc = acc0 + acc1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) y[row] = acc;
}

// ---- PCG with explicit z (K = 1) ----------------------------------------------------------------
enum { FIN_CGZ_INIT = 32, FIN_CGZ_RZ0, FIN_CGZ_RZ, FIN_CGZ_UPDATE };

__device__ inline void cgz_finalize(int fin, KryState* st, const double* t) {
  switch (fin) {
    case FIN_CGZ_INIT: {  // t = bb, rr
      st->bb[0] = t[0];
      st->rr[0] = t[1];
      st->rr0[0] = t[1];
      double a2 = st->atol * st->atol, r2 = st->rtol * st->rtol * st->bb[0];
      st->tol2[0] = r2 > a2 ? r2 : a2;
      st->its[0] = 0;
      st->reason[0] = 0;
      st->active[0] = 1;
      st->beta[0] = 0.0;
      kry_converge_test(st, 0);
      kry_check_done(st);
    } break;
    case FIN_CGZ_RZ0:
      st->rz[0] = t[0];
      st->beta[0] = 0.0;
      break;
    case FIN_CGZ_RZ:
      st->beta[0] = t[0] / st->rz[0];
      st->rz[0] = t[0];
      break;
    case FIN_CGZ_UPDATE:  // t = rr
      if (st->active[0]) {
        st->rr[0] = t[0];
        st->its[0] += 1;
        kry_converge_test(st, 0);
      }
      kry_check_done(st);
      break;
  }
}

template <int N>
__device__ __forceinline__ void cgz_reduce_finish(double (&v)[N], double* partials, unsigned* counter, int fin,
                                                  KryState* st, RedCtl red_out) {
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
    if (threadIdx.x == 0) cgz_finalize(fin, st, sh);
  } else if (threadIdx.x == 0) {
    if (red_out.out != nullptr) {
#pragma unroll
      for (int i = 0; i < N; ++i) red_out.out[i] = total[i];
    } else {
      cgz_finalize(fin, st, total);
    }
  }
}

__global__ void k_cgz_finalize(int fin, KryState* st, const double* __restrict__ totals) { cgz_finalize(fin, st, totals); }

// r = b - q (or r = b, x = 0); sums bb, rr
__global__ void __launch_bounds__(256)
k_cgz_init(int64_t n, const double* __restrict__ b, const double* __restrict__ q, double* __restrict__ x,
           double* __restrict__ r, KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  double s[2] = {0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double bv = b[i];
    double rv = bv;
    if (q != nullptr) rv -= q[i];
    else x[i] = 0.0;
    r[i] = rv;
    s[0] = fma(bv, bv, s[0]);
    s[1] = fma(rv, rv, s[1]);
  }
  cgz_reduce_finish<2>(s, partials, counter, FIN_CGZ_INIT, st, red_out);
}

// sum r.z -> rz (first: beta = 0) / beta = rz'/rz
__global__ void __launch_bounds__(256)
k_cgz_rz(int64_t n, const double* __restrict__ r, const double* __restrict__ z, int fin, KryState* st,
         double* partials, unsigned* counter, RedCtl red_out) {
  double s[1] = {0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    s[0] = fma(r[i], z[i], s[0]);
  cgz_reduce_finish<1>(s, partials, counter, fin, st, red_out);
}

// p = z + beta p
__global__ void k_cgz_p(int64_t n, const double* __restrict__ z, double* __restrict__ p, const KryState* st) {
  const double beta = st->beta[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = fma(beta, p[i], z[i]);
}

// x += alpha p ; r -= alpha q ; sum rr
__global__ void __launch_bounds__(256)
k_cgz_update(int64_t n, const double* __restrict__ p, const double* __restrict__ q, double* __restrict__ x,
             double* __restrict__ r, KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  if (st->done) return;
  const double alpha = st->alpha[0];
  double s[1] = {0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double rv = fma(-alpha, q[i], r[i]);
    r[i] = rv;
    s[0] = fma(rv, rv, s[0]);
  }
  cgz_reduce_finish<1>(s, partials, counter, FIN_CGZ_UPDATE, st, red_out);
}

__global__ void __launch_bounds__(256)
k_mg_sweep_rz(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ cols, const double* __restrict__ vals,
              const double* __restrict__ dinv, const double* __restrict__ b, const double* __restrict__ x_in, double omega,
              double* __restrict__ out, int fin, KryState* st, double* partials, unsigned* counter, RedCtl red_out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n_slices = (n_rows + 31) >> 5;
  double s[1] = {0.0};
  for (int sl = warp; sl < n_slices; sl += nwarps) {
    const int base = __ldg(slice_ptr + sl);
    const int len = (__ldg(slice_ptr + sl + 1) - base) >> 5;
    const int row = (sl << 5) + lane;
    double acc = 0.0;
#pragma unroll 4
    for (int t = 0; t < len; ++t) {
      const int c = ld_stream(cols + base + lane + (t << 5));
      acc = fma(ld_stream(vals + base + lane + (t << 5)), __ldg(x_in + c), acc);
    }
    if (row < n_rows) {
      const double r = b[row];
      const double z = fma(omega * dinv[row], r - acc, x_in[row]);
      out[row] = z;
      s[0] = fma(r, z, s[0]);
    }
  }
  cgz_reduce_finish<1>(s, partials, counter, fin, st, red_out);
}

// k_cgz_init / k_cgz_update with the first smoothing sweep of the next V-cycle fused in: x0 = omega D^-1 r
__global__ void __launch_bounds__(256)
k_cgz_init_x0(int64_t n, const double* __restrict__ b, const double* __restrict__ q, double* __restrict__ x,
              double* __restrict__ r, const double* __restrict__ dinv, double omega, double* __restrict__ x0, KryState* st,
              double* partials, unsigned* counter, RedCtl red_out) {
  double s[2] = {0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double bv = b[i];
    double rv = bv;
    if (q != nullptr) rv -= q[i];
    else x[i] = 0.0;
    r[i] = rv;
    x0[i] = omega * dinv[i] * rv;
    s[0] = fma(bv, bv, s[0]);
    s[1] = fma(rv, rv, s[1]);
  }
  cgz_reduce_finish<2>(s, partials, counter, FIN_CGZ_INIT, st, red_out);
}

__global__ void __launch_bounds__(256)
k_cgz_update_x0(int64_t n, const double* __restrict__ p, const double* __restrict__ q, double* __restrict__ x,
                double* __restrict__ r, const double* __restrict__ dinv, double omega, double* __restrict__ x0, KryState* st,
                double* partials, unsigned* counter, RedCtl red_out) {
  if (st->done) return;
  const double alpha = st->alpha[0];
  double s[1] = {0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double rv = fma(-alpha, q[i], r[i]);
    r[i] = rv;
    x0[i] = omega * dinv[i] * rv;
    s[0] = fma(rv, rv, s[0]);
  }
  cgz_reduce_finish<1>(s, partials, counter, FIN_CGZ_UPDATE, st, red_out);
}
