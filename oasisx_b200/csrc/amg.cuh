// amg.cuh -- kernels of the smoothed-aggregation algebraic multigrid set-up (b2_pressure_amg_build): strength graph,
// MIS(2) aggregation (Bell, Dalton and Olson 2012) that keeps the pressure Dirichlet dofs out of every aggregate, power
// iteration for rho(D^-1 A), and the expand-sort-reduce sparse
// products behind P = (I - omega D^-1 A) T, R = P^T and A_c = R (A P), and on several ranks the gather of the global
// fine matrix and the cut of level 1 back to each rank's owned rows.  Every step is deterministic: no floating-point
// atomics, sums are taken sequentially in an order fixed by a stable sort, and the reductions of the power iteration
// run in one block in a fixed order (k_amg_sum).  The V-cycle that uses the hierarchy is mg.cuh's.
#pragma once
#include "linalg.cuh"

enum { AMG_OUT = 0, AMG_UNDECIDED = 1, AMG_ROOT = 2 };

// murmur3 finaliser: the random key of node i is (amg_fmix32(i ^ 0x9E3779B9), i)
__host__ __device__ __forceinline__ uint32_t amg_fmix32(uint32_t h) {
  h ^= h >> 16;
  h *= 0x85ebca6bu;
  h ^= h >> 13;
  h *= 0xc2b2ae35u;
  h ^= h >> 16;
  return h;
}

// (key_hash, i) packed so that integer order is lexicographic order; i < 2^30
__device__ __forceinline__ unsigned long long amg_key(int i) {
  return ((unsigned long long)amg_fmix32((uint32_t)i ^ 0x9E3779B9u) << 30) | (unsigned)i;
}

// j is a strong neighbour of i when j != i and a_ij != 0 (threshold 0)
__device__ __forceinline__ bool amg_strong(int i, int j, double a) { return j != i && a != 0.0; }

// excl (nullptr: none): nodes kept out of every aggregate (pressure Dirichlet dofs of the fine level); they start out
// of the MIS and are never roots
__global__ void k_amg_init(int n, const uint8_t* __restrict__ excl, int* __restrict__ state) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) state[i] = excl != nullptr && excl[i] ? AMG_OUT : AMG_UNDECIDED;
}

// an excluded row must be isolated in the strength graph (no nonzero off-diagonal entry): *err = 1 otherwise
__global__ void k_amg_check_excluded(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                                     const uint8_t* __restrict__ excl, int* __restrict__ err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !excl[i]) return;
  for (int p = rp[i]; p < rp[i + 1]; ++p)
    if (amg_strong(i, ci[p], va[p])) atomicOr(err, 1);
}

// t[i] = (state_i, key_i): the MIS(2) tuple, state in the top two bits
__global__ void k_amg_tuples(int n, const int* __restrict__ state, unsigned long long* __restrict__ t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) t[i] = ((unsigned long long)state[i] << 62) | amg_key(i);
}

// one hop of the 2-hop maximum: out_i = max(in_i, in_j over the strong neighbours j of i)
__global__ void k_amg_max_hop(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                              const unsigned long long* __restrict__ in, unsigned long long* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long m = in[i];
  for (int p = rp[i]; p < rp[i + 1]; ++p) {
    const int j = ci[p];
    if (amg_strong(i, j, va[p])) m = max(m, in[j]);
  }
  out[i] = m;
}

// end of a synchronous round: an undecided node that is the 2-hop maximum becomes a root, one that sees a root within
// two hops drops out; *undecided counts those left
__global__ void k_amg_mis_update(int n, int* __restrict__ state, const unsigned long long* __restrict__ t0,
                                 const unsigned long long* __restrict__ m2, int* __restrict__ undecided) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || state[i] != AMG_UNDECIDED) return;
  if (m2[i] == t0[i]) state[i] = AMG_ROOT;
  else if ((int)(m2[i] >> 62) == AMG_ROOT) state[i] = AMG_OUT;
  else atomicAdd(undecided, 1);
}

__global__ void k_amg_root_flags(int n, const int* __restrict__ state, int* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = state[i] == AMG_ROOT;
}

// pass 1: roots take their number (exclusive scan of the root flags), their neighbours join them (roots are >= 3 apart,
// so at most one root is adjacent); -1: not assigned yet
__global__ void k_amg_pass1(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                            const int* __restrict__ state, const int* __restrict__ id, int* __restrict__ agg1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int a = -1;
  if (state[i] == AMG_ROOT) {
    a = id[i];
  } else {
    for (int p = rp[i]; p < rp[i + 1]; ++p) {
      const int j = ci[p];
      if (amg_strong(i, j, va[p]) && state[j] == AMG_ROOT) a = id[j];
    }
  }
  agg1[i] = a;
}

// pass 2: a node left over joins the aggregate of its pass-1 neighbour with the largest key; MIS(2) maximality
// guarantees one exists -- a node without one sets *err.  An excluded node keeps -1.
__global__ void k_amg_pass2(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                            const uint8_t* __restrict__ excl, const int* __restrict__ agg1, int* __restrict__ agg,
                            int* __restrict__ err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int a = agg1[i];
  if (a < 0 && !(excl != nullptr && excl[i])) {
    unsigned long long best = 0;
    for (int p = rp[i]; p < rp[i + 1]; ++p) {
      const int j = ci[p];
      if (amg_strong(i, j, va[p]) && agg1[j] >= 0) {
        const unsigned long long k = amg_key(j) + 1;
        if (k > best) { best = k; a = agg1[j]; }
      }
    }
    if (a < 0) atomicOr(err, 1);
  }
  agg[i] = a;
}

// hash-seeded start vector of the power iteration, entries in [-0.5, 0.5)
__global__ void k_amg_seed(int n, double* __restrict__ x) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = amg_fmix32((uint32_t)i ^ 0x2545F491u) * (1.0 / 4294967296.0) - 0.5;
}

// one power step y = D^-1 A (x / |x|), |x|^2 = *nrm2 (nullptr: 1); y2 = y^2 for the next norm
__global__ void k_amg_power(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                            const double* __restrict__ dinv, const double* __restrict__ x, const double* __restrict__ nrm2,
                            double* __restrict__ y, double* __restrict__ y2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double s = nrm2 != nullptr ? rsqrt(*nrm2) : 1.0;
  double acc = 0.0;
  for (int p = rp[i]; p < rp[i + 1]; ++p) acc = fma(va[p], x[ci[p]], acc);
  const double v = dinv[i] * acc * s;
  y[i] = v;
  y2[i] = v * v;
}

// *out = sum of in[0..n) by ONE 1024-thread block in a fixed order (strided partial sums, then a fixed tree): the
// same bits on every run, whatever the scheduling.  Set-up only; a few microseconds per 10^6 entries.
__global__ void __launch_bounds__(1024) k_amg_sum(int n, const double* __restrict__ in, double* __restrict__ out) {
  __shared__ double sm[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += in[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
    acc = warp_sum(acc);
    if (threadIdx.x == 0) *out = acc;
  }
}

// terms of the Rayleigh quotient of D^-1 A in the D inner product: num_i = x_i (A x)_i, den_i = x_i^2 / dinv_i
__global__ void k_amg_rayleigh(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                               const double* __restrict__ dinv, const double* __restrict__ x, double* __restrict__ num,
                               double* __restrict__ den) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double acc = 0.0;
  for (int p = rp[i]; p < rp[i + 1]; ++p) acc = fma(va[p], x[ci[p]], acc);
  num[i] = x[i] * acc;
  den[i] = x[i] * x[i] / dinv[i];
}

// values of the prolongator smoother S = I - omega D^-1 A on A's pattern
__global__ void k_amg_smoother(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                               const double* __restrict__ dinv, double omega, double* __restrict__ s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double w = omega * dinv[i];
  for (int p = rp[i]; p < rp[i + 1]; ++p) s[p] = (ci[p] == i ? 1.0 : 0.0) - w * va[p];
}

// flag[i] = 1 where node i has an aggregate: the row lengths of T, whose exclusive scan is T's row pointer (rp[i] = i
// when no node is excluded)
__global__ void k_amg_kept_flags(int n, const int* __restrict__ agg, int* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = agg[i] >= 0;
}

// tentative prolongator T[i, agg(i)] = 1 as CSR; the row of an excluded node (agg -1) is empty
__global__ void k_amg_tentative(int n, const int* __restrict__ agg, const int* __restrict__ rp, int* __restrict__ ci,
                                double* __restrict__ va) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || agg[i] < 0) return;
  ci[rp[i]] = agg[i];
  va[rp[i]] = 1.0;
}

// row index of every stored entry of a CSR matrix
__global__ void k_amg_entry_rows(int n, const int* __restrict__ rp, int* __restrict__ row) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int p = rp[i]; p < rp[i + 1]; ++p) row[p] = i;
}

// ---- C = A B by expansion: one (key = row << 32 | col, product) pair per A_ij B_jk -------------------------------
__global__ void k_amg_product_counts(int64_t nnz_a, const int* __restrict__ ca, const int* __restrict__ rpb,
                                     int64_t* __restrict__ cnt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < nnz_a) cnt[e] = rpb[ca[e] + 1] - rpb[ca[e]];
}

__global__ void k_amg_expand(int64_t nnz_a, const int* __restrict__ row_a, const int* __restrict__ ca,
                             const double* __restrict__ va, const int* __restrict__ rpb, const int* __restrict__ cb,
                             const double* __restrict__ vb, const int64_t* __restrict__ off,
                             unsigned long long* __restrict__ keys, double* __restrict__ vals) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz_a) return;
  const unsigned long long r = (unsigned long long)(unsigned)row_a[e] << 32;
  const double a = va[e];
  int64_t o = off[e];
  const int j = ca[e];
  for (int p = rpb[j]; p < rpb[j + 1]; ++p, ++o) {
    keys[o] = r | (unsigned)cb[p];
    vals[o] = a * vb[p];
  }
}

// (key, value) pairs of a transpose: (col << 32 | row, value)
__global__ void k_amg_transpose_keys(int64_t nnz, const int* __restrict__ row, const int* __restrict__ col,
                                     const double* __restrict__ v, unsigned long long* __restrict__ keys,
                                     double* __restrict__ vals) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  keys[e] = ((unsigned long long)(unsigned)col[e] << 32) | (unsigned)row[e];
  vals[e] = v[e];
}

// head[t] = 1 where a run of equal sorted keys starts (head[n] = 0 closes the scan)
__global__ void k_amg_heads(int64_t n, const unsigned long long* __restrict__ keys, int* __restrict__ head) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n) return;
  head[t] = t < n && (t == 0 || keys[t] != keys[t - 1]);
}

// ---- several ranks: the global matrix gathered from every rank's owned rows, level 1 cut back to the owned rows -----
// (global row << 32 | global col, a_ij) for every entry of this rank's owned rows; gid = global id of every local dof
__global__ void k_amg_global_pairs(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                                   const int* __restrict__ gid, unsigned long long* __restrict__ keys, double* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long r = (unsigned long long)(unsigned)gid[i] << 32;
  for (int p = rp[i]; p < rp[i + 1]; ++p) {
    keys[p] = r | (unsigned)gid[ci[p]];
    vals[p] = va[p];
  }
}

// mask[gid] = flag of an owned row, from the gathered (global id << 8 | flag) of every rank
__global__ void k_amg_scatter_mask(int64_t n, const unsigned long long* __restrict__ keys, uint8_t* __restrict__ mask) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) mask[keys[t] >> 8] = (uint8_t)(keys[t] & 0xff);
}

// (global id << 8 | flag) of this rank's owned rows
__global__ void k_amg_flag_keys(int n, const int* __restrict__ gid, const uint8_t* __restrict__ flag,
                                unsigned long long* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = ((unsigned long long)(unsigned)gid[i] << 8) | (flag[i] ? 1u : 0u);
}

// dinv_i = 1 / a_ii of a CSR matrix (every row of the gathered Ap holds its diagonal)
__global__ void k_amg_inv_diag(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                               double* __restrict__ dinv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int p = rp[i]; p < rp[i + 1]; ++p)
    if (ci[p] == i) dinv[i] = 1.0 / va[p];
}

// len[i] = length of row gid[i] of a CSR matrix
__global__ void k_amg_row_lengths(int n, const int* __restrict__ rp, const int* __restrict__ gid, int* __restrict__ len) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) len[i] = rp[gid[i] + 1] - rp[gid[i]];
}

// row i of the output = row gid[i] of (rp, ci, va), and agg_out[i] = agg[gid[i]]: the rows of the global P_1 and the
// aggregates of this rank's owned dofs, in local order
__global__ void k_amg_gather_rows(int n, const int* __restrict__ rp, const int* __restrict__ ci, const double* __restrict__ va,
                                  const int* __restrict__ agg, const int* __restrict__ gid, const int* __restrict__ rp_out,
                                  int* __restrict__ ci_out, double* __restrict__ va_out, int* __restrict__ agg_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int g = gid[i];
  int o = rp_out[i];
  for (int p = rp[g]; p < rp[g + 1]; ++p, ++o) {
    ci_out[o] = ci[p];
    va_out[o] = va[p];
  }
  agg_out[i] = agg[g];
}

// one thread per run: the run's key and the sequential sum of its values, in sorted (= stable generation) order
__global__ void k_amg_reduce_runs(int64_t n, const unsigned long long* __restrict__ keys, const double* __restrict__ vals,
                                  const int* __restrict__ head, const int* __restrict__ run,
                                  unsigned long long* __restrict__ ukeys, double* __restrict__ uvals) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n || !head[t]) return;
  const unsigned long long k = keys[t];
  double acc = vals[t];
  for (int64_t u = t + 1; u < n && keys[u] == k; ++u) acc += vals[u];
  ukeys[run[t]] = k;
  uvals[run[t]] = acc;
}
