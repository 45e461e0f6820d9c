// elem.cuh -- affine simplex geometry, reference tensors in constant memory, and the cell
// (element) kernels that replace the FFCx tabulate_tensor + DOLFINx assemble_matrix /
// assemble_vector pairs of /root/reference/src/oasisx/fracstep.py:289-404,435-437.
#pragma once
#include "common.cuh"

#define B2_TABLE_QUAL static __constant__ const
#include "ref_tables.h"

// ---- element traits: (gdim, velocity degree) -> table accessors ----------------------------
template <int D, int DEG>
struct El;

#define B2_DEFINE_EL(D_, DEG_, NV_)                                                            \
  template <>                                                                                  \
  struct El<D_, DEG_> {                                                                        \
    static constexpr int D = D_, DEG = DEG_, NV = NV_, NQ = D_ + 1;                                        \
    __device__ static __forceinline__ double MV(int i, int j) { return REF_D##D_##P##DEG_##_MV[i][j]; } \
    __device__ static __forceinline__ double SV(int a, int b, int i, int j) { return REF_D##D_##P##DEG_##_SV[a][b][i][j]; } \
    __device__ static __forceinline__ double T(int a, int dl, int i, int j) { return REF_D##D_##P##DEG_##_T[a][dl][i][j]; } \
    __device__ static __forceinline__ double PX(int dl, int j, int q) { return REF_D##D_##P##DEG_##_PX[dl][j][q]; } \
    __device__ static __forceinline__ double GX(int dl, int j, int q) { return REF_D##D_##P##DEG_##_GX[dl][j][q]; } \
    __device__ static __forceinline__ double SQ(int a, int b, int q, int r) { return REF_D##D_##P##DEG_##_SQ[a][b][q][r]; } \
    __device__ static __forceinline__ double MQ(int q, int r) { return REF_D##D_##P##DEG_##_MQ[q][r]; } \
    __device__ static __forceinline__ double LV(int j) { return REF_D##D_##P##DEG_##_LV[j]; }   \
    __device__ static __forceinline__ double LQ(int q) { return REF_D##D_##P##DEG_##_LQ[q]; }   \
  };

B2_DEFINE_EL(2, 1, 3)
B2_DEFINE_EL(2, 2, 6)
B2_DEFINE_EL(3, 1, 4)
B2_DEFINE_EL(3, 2, 10)

// ---- geometry --------------------------------------------------------------------------------
// J[k][dl] = d x_k / d xi_dl ;  Kinv = J^{-1}  (Kinv[dl][k]) ;  physical gradient
// d/dx_k = sum_dl Kinv[dl][k] d/dxi_dl   (SURVEY.md Appendix C)
template <int D>
struct Geo {
  double Kinv[D][D];
  double detJ;  // |det J|
};

template <int D>
__device__ __forceinline__ Geo<D> cell_geometry(const double* __restrict__ x,
                                                const int* __restrict__ nodes) {
  Geo<D> g;
  double X[D + 1][D];
#pragma unroll
  for (int v = 0; v <= D; ++v) {
    const double* p = x + 3 * (size_t)nodes[v];
#pragma unroll
    for (int k = 0; k < D; ++k) X[v][k] = p[k];
  }
  double J[D][D];
#pragma unroll
  for (int k = 0; k < D; ++k)
#pragma unroll
    for (int dl = 0; dl < D; ++dl) J[k][dl] = X[dl + 1][k] - X[0][k];
  if constexpr (D == 2) {
    double det = J[0][0] * J[1][1] - J[0][1] * J[1][0];
    double id = 1.0 / det;
    g.Kinv[0][0] = J[1][1] * id;
    g.Kinv[0][1] = -J[0][1] * id;
    g.Kinv[1][0] = -J[1][0] * id;
    g.Kinv[1][1] = J[0][0] * id;
    g.detJ = fabs(det);
  } else {
    double c00 = J[1][1] * J[2][2] - J[1][2] * J[2][1];
    double c01 = J[1][2] * J[2][0] - J[1][0] * J[2][2];
    double c02 = J[1][0] * J[2][1] - J[1][1] * J[2][0];
    double det = J[0][0] * c00 + J[0][1] * c01 + J[0][2] * c02;
    double id = 1.0 / det;
    g.Kinv[0][0] = c00 * id;
    g.Kinv[0][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * id;
    g.Kinv[0][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * id;
    g.Kinv[1][0] = c01 * id;
    g.Kinv[1][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * id;
    g.Kinv[1][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * id;
    g.Kinv[2][0] = c02 * id;
    g.Kinv[2][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * id;
    g.Kinv[2][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * id;
    g.detJ = fabs(det);
  }
  return g;
}

// position of column `col` in CSR row [lo, hi) (columns sorted); -1 if absent
__device__ __forceinline__ int csr_find(const int* __restrict__ cols, int lo, int hi, int col) {
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    int c = __ldg(cols + mid);
    if (c < col)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// ---- one-off (pre)assembly kernels: one thread per (cell, local row) -----------------------
enum { B2_FORM_MASS_V = 0, B2_FORM_STIFF_V = 1, B2_FORM_MASS_Q = 2, B2_FORM_STIFF_Q = 3 };

// pair_slot != nullptr: instead of adding into vals, entry (cell, i, j) writes its SELL slot and value to
// pair_slot/pair_val[(cell * ND + i) * ND + j] (sum_slot_pairs adds them up in a fixed order)
template <int D, int DEG, int FORM>
__global__ void k_assemble_square(int64_t n_cells, const double* __restrict__ x,
                                  const int* __restrict__ cell_nodes, const int* __restrict__ cdofs,
                                  int n_rows_owned, const int* __restrict__ rowptr,
                                  const int* __restrict__ cols, const int* __restrict__ slice_ptr,
                                  double* __restrict__ vals, unsigned* __restrict__ pair_slot = nullptr,
                                  double* __restrict__ pair_val = nullptr) {
  using E = El<D, DEG>;
  constexpr bool onV = (FORM == B2_FORM_MASS_V || FORM == B2_FORM_STIFF_V);
  constexpr int ND = onV ? E::NV : E::NQ;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cells * ND) return;
  int64_t c = t / ND;
  int i = (int)(t - c * ND);
  const int* dofs = cdofs + c * ND;
  int row = dofs[i];
  if (row >= n_rows_owned) return;
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  double G[D][D];
  if constexpr (FORM == B2_FORM_STIFF_V || FORM == B2_FORM_STIFF_Q) {
#pragma unroll
    for (int a = 0; a < D; ++a)
#pragma unroll
      for (int b = 0; b < D; ++b) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < D; ++k) s += g.Kinv[a][k] * g.Kinv[b][k];
        G[a][b] = s * g.detJ;
      }
  }
  int lo = rowptr[row], hi = rowptr[row + 1];
  for (int j = 0; j < ND; ++j) {
    double v = 0;
    if constexpr (FORM == B2_FORM_MASS_V) v = g.detJ * E::MV(i, j);
    if constexpr (FORM == B2_FORM_MASS_Q) v = g.detJ * E::MQ(i, j);
    if constexpr (FORM == B2_FORM_STIFF_V) {
#pragma unroll
      for (int a = 0; a < D; ++a)
#pragma unroll
        for (int b = 0; b < D; ++b) v += G[a][b] * E::SV(a, b, i, j);
    }
    if constexpr (FORM == B2_FORM_STIFF_Q) {
#pragma unroll
      for (int a = 0; a < D; ++a)
#pragma unroll
        for (int b = 0; b < D; ++b) v += G[a][b] * E::SQ(a, b, i, j);
    }
    int pos = csr_find(cols, lo, hi, dofs[j]);
    if (pair_slot != nullptr) {
      pair_slot[t * ND + j] = (unsigned)sell_slot(slice_ptr, row, pos - lo);
      pair_val[t * ND + j] = v;
    } else {
      atomicAdd(vals + sell_slot(slice_ptr, row, pos - lo), v);
    }
  }
}

// after a stable sort of the (slot, value) pairs by slot: the first pair of every slot adds up its run sequentially
// and stores the sum; slot 0xffffffff marks pairs nobody wrote (rows owned by another rank)
__global__ void k_sum_slot_runs(int64_t n, const unsigned* __restrict__ slot, const double* __restrict__ v,
                                double* __restrict__ vals) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n || slot[t] == 0xffffffffu || (t > 0 && slot[t] == slot[t - 1])) return;
  double acc = v[t];
  for (int64_t u = t + 1; u < n && slot[u] == slot[t]; ++u) acc += v[u];
  vals[slot[t]] = acc;
}

// P_c[j,q] = int psi_q d_c phi_j and G_c[j,q] = int d_c psi_q phi_j in the SELL-32 slots of the V x Q
// pattern, component-major: direction c at vals + c * slots (the form k_rect_vq_sell reads; pads stay 0).
template <int D, int DEG>
__global__ void k_assemble_PG(int64_t n_cells, const double* __restrict__ x,
                              const int* __restrict__ cell_nodes, const int* __restrict__ vdofs,
                              const int* __restrict__ qdofs, int n_rows_owned,
                              const int* __restrict__ rowptr, const int* __restrict__ cols,
                              const int* __restrict__ slice_ptr, int64_t slots,
                              double* __restrict__ Pvals, double* __restrict__ Gvals) {
  using E = El<D, DEG>;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cells * E::NV) return;
  int64_t c = t / E::NV;
  int j = (int)(t - c * E::NV);
  int row = vdofs[c * E::NV + j];
  if (row >= n_rows_owned) return;
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  int lo = rowptr[row], hi = rowptr[row + 1];
  for (int q = 0; q < E::NQ; ++q) {
    const size_t s = sell_slot(slice_ptr, row, csr_find(cols, lo, hi, qdofs[c * E::NQ + q]) - lo);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      double p = 0, gg = 0;
#pragma unroll
      for (int dl = 0; dl < D; ++dl) {
        p += g.Kinv[dl][k] * E::PX(dl, j, q);
        gg += g.Kinv[dl][k] * E::GX(dl, j, q);
      }
      atomicAdd(Pvals + (size_t)k * slots + s, g.detJ * p);
      atomicAdd(Gvals + (size_t)k * slots + s, g.detJ * gg);
    }
  }
}

// D_c[q,j] = int d_c phi_j psi_q on the Q x V pattern ([nnz][D])
template <int D, int DEG>
__global__ void k_assemble_D(int64_t n_cells, const double* __restrict__ x,
                             const int* __restrict__ cell_nodes, const int* __restrict__ vdofs,
                             const int* __restrict__ qdofs, int n_rows_owned,
                             const int* __restrict__ rowptr, const int* __restrict__ cols,
                             double* __restrict__ Dvals) {
  using E = El<D, DEG>;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cells * E::NQ) return;
  int64_t c = t / E::NQ;
  int q = (int)(t - c * E::NQ);
  int row = qdofs[c * E::NQ + q];
  if (row >= n_rows_owned) return;
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  int lo = rowptr[row], hi = rowptr[row + 1];
  for (int j = 0; j < E::NV; ++j) {
    int pos = csr_find(cols, lo, hi, vdofs[c * E::NV + j]);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      double p = 0;
#pragma unroll
      for (int dl = 0; dl < D; ++dl) p += g.Kinv[dl][k] * E::PX(dl, j, q);
      atomicAdd(Dvals + (size_t)pos * D + k, g.detJ * p);
    }
  }
}

// b0[j][c] = int f_c phi_j (fracstep.py:387-390), mQ[q] = int psi_q (the measure for :581-591)
template <int D, int DEG>
__global__ void k_assemble_loads(int64_t n_cells, const double* __restrict__ x,
                                 const int* __restrict__ cell_nodes, const int* __restrict__ vdofs,
                                 const int* __restrict__ qdofs, int nV_owned, int nQ_owned, int ld,
                                 double f0, double f1, double f2, double* __restrict__ b0,
                                 double* __restrict__ mQ) {
  using E = El<D, DEG>;
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  const double f[3] = {f0, f1, f2};
  for (int j = 0; j < E::NV; ++j) {
    int row = vdofs[c * E::NV + j];
    if (row >= nV_owned) continue;
    double l = g.detJ * E::LV(j);
#pragma unroll
    for (int k = 0; k < D; ++k)
      if (f[k] != 0.0) atomicAdd(b0 + (size_t)k * ld + row, f[k] * l);
  }
  for (int q = 0; q < E::NQ; ++q) {
    int row = qdofs[c * E::NQ + q];
    if (row < nQ_owned) atomicAdd(mQ + row, g.detJ * E::LQ(q));
  }
}

// ---- per-step convection assembly (fracstep.py:435-437) --------------------------------------
// Scatter table, built once: pos8[(c*NV + i)*NVP + j] = index t of column dofs[j] within row dofs[i]
// (t < 256; the host checks the longest row), NVP = NV rounded up to a multiple of 4 so that a row of
// the table is read with 32-bit loads.  It replaces 100 binary searches per P2 tetrahedron and step by
// 120 bytes of streamed table.
template <int NV>
__global__ void k_build_pos8(int64_t n_cells, const int* __restrict__ vdofs, int n_rows_owned,
                             const int* __restrict__ rowptr, const int* __restrict__ cols,
                             uint8_t* __restrict__ pos8) {
  constexpr int NVP = (NV + 3) / 4 * 4;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cells * NV) return;
  int64_t c = t / NV;
  int i = (int)(t - c * NV);
  const int* dofs = vdofs + c * NV;
  int row = dofs[i];
  uint8_t* out = pos8 + (size_t)t * NVP;
  if (row >= n_rows_owned) {
    for (int j = 0; j < NVP; ++j) out[j] = 0;
    return;
  }
  int lo = rowptr[row], hi = rowptr[row + 1];
  for (int j = 0; j < NVP; ++j) out[j] = j < NV ? (uint8_t)(csr_find(cols, lo, hi, dofs[j]) - lo) : 0;
}

// ---- assemble_first, cell-parallel (fracstep.py:432-472 in one pass over the cells) -----------------------------
// One thread per cell forms, row by row, the COMPLETE element operators of the step
//     A_e = M_e/dt + nu/2 K_e + 1/2 C_e(uab)      (left-hand side, :468-469)
//     R_e = M_e/dt - nu/2 K_e - 1/2 C_e(uab)      (right-hand side operator, :438-442)
// from the exact reference tensors (every tensor entry a compile-time operand of its DFMA; M and K are never read
// from memory) and, matrix-free, the action  b_first += R_e u1_e  (the "action strategy" of
// demo/assembly_strategies.py:83-88,137-140): no separate CSR-value passes, no SpMV, A written by FP64 reductions
// into zero-filled slots and finished (Dirichlet rows -> identity, dinv = 1/diagonal) by k_first_finalize.
//
// COALESCED SCATTER.  The kernel is bound by the number of 32-byte sectors its reductions touch (one LSU wavefront
// each), not by bytes or flops: with cells in mesh order the 32 lanes of a RED hit 32 sectors.  `cell_order` (host:
// build_first_plan) lists the cells by congruence class -- cells that are translates of each other -- and, inside a
// class, along x: consecutive lanes then hold the same local dof of consecutive dofs of one stencil class, the
// scatter position t is the same for all of them, and a RED instruction covers 32 CONSECUTIVE doubles of one
// sliced-ELL column (8 sectors instead of 32); the gathers of uab / u1 coalesce the same way.  Classes are
// interleaved slab by slab so that the rows being accumulated stay resident in L2.  Meshes without congruent cells
// simply keep their order (nothing assumes a lattice).  Summation order inside an entry is not fixed (L2
// reductions): reproducible to rounding, like PETSc's ADD_VALUES over ranks.
//   MODE & 1: matrix,  MODE & 2: vector (b_first, preloaded with b0 + p_surf by k_first_init).
template <int D, int DEG, int MODE>
__global__ void __launch_bounds__(128, 3)
k_first_cells(int64_t n_cells, const int* __restrict__ cell_order, const double* __restrict__ x,
              const int* __restrict__ cell_nodes, const int* __restrict__ vdofs, int n_rows_owned,
              const double* __restrict__ uab, const double* __restrict__ u1, int ld, const int* __restrict__ slice_ptr,
              const uint8_t* __restrict__ pos8, const uint8_t* __restrict__ is_bc_row, double inv_dt, double half_nu,
              double* __restrict__ Avals, double* __restrict__ bfirst) {
  using E = El<D, DEG>;
  constexpr int NV = E::NV, K = D;
  constexpr int NVP = (NV + 3) / 4 * 4;
  constexpr bool MAT = (MODE & 1) != 0, VEC = (MODE & 2) != 0;
  const int64_t ci = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ci >= n_cells) return;
  const int64_t c = cell_order != nullptr ? (int64_t)__ldg(cell_order + ci) : ci;
  const Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  int dofs[NV];
#pragma unroll
  for (int a = 0; a < NV; ++a) dofs[a] = vdofs[c * NV + a];
  double w[NV][D], u1e[NV][K];
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double u[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      u[k] = __ldg(uab + (size_t)k * ld + dofs[a]);
      if (VEC) u1e[a][k] = __ldg(u1 + (size_t)k * ld + dofs[a]);
    }
#pragma unroll
    for (int dl = 0; dl < D; ++dl) {
      double sacc = 0;
#pragma unroll
      for (int k = 0; k < D; ++k) sacc += g.Kinv[dl][k] * u[k];
      w[a][dl] = sacc * (0.5 * g.detJ);  // 1/2 C_e
    }
  }
  // Gh = nu/2 |detJ| Kinv Kinv^T (symmetric): nu/2 K_e[i][j] = sum_ab Gh[a][b] SV[a][b][i][j]
  double Gh[D][D];
#pragma unroll
  for (int a = 0; a < D; ++a)
#pragma unroll
    for (int b = a; b < D; ++b) {
      double sacc = 0;
#pragma unroll
      for (int k = 0; k < D; ++k) sacc += g.Kinv[a][k] * g.Kinv[b][k];
      Gh[a][b] = Gh[b][a] = sacc * (half_nu * g.detJ);
    }
  const double mdt = inv_dt * g.detJ;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int row = dofs[i];
    if (row >= n_rows_owned) continue;
    double cv[NV], kv[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) { cv[j] = 0.0; kv[j] = 0.0; }
#pragma unroll
    for (int a = 0; a < NV; ++a)
#pragma unroll
      for (int dl = 0; dl < D; ++dl) {
        const double wv = w[a][dl];
#pragma unroll
        for (int j = 0; j < NV; ++j)
          if (E::T(a, dl, i, j) != 0.0) cv[j] = fma(wv, E::T(a, dl, i, j), cv[j]);
      }
#pragma unroll
    for (int a = 0; a < D; ++a)
#pragma unroll
      for (int b = a; b < D; ++b) {
        const double gv = Gh[a][b];
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          const double sv = (a == b) ? E::SV(a, b, i, j) : (E::SV(a, b, i, j) + E::SV(b, a, i, j));
          if (sv != 0.0) kv[j] = fma(gv, sv, kv[j]);
        }
      }
    double dot[K];
#pragma unroll
    for (int k = 0; k < K; ++k) dot[k] = 0.0;
    double av[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const double m = mdt * E::MV(i, j);
      av[j] = (m + cv[j]) + kv[j];
      if (VEC) {
        const double rr = (m - cv[j]) - kv[j];
#pragma unroll
        for (int k = 0; k < K; ++k) dot[k] = fma(rr, u1e[j][k], dot[k]);
      }
    }
    if (MAT && !is_bc_row[row]) {
      const uint32_t* pw = reinterpret_cast<const uint32_t*>(pos8 + ((size_t)c * NV + i) * NVP);
      double* rowbase = Avals + (size_t)__ldg(slice_ptr + (row >> 5)) + (row & 31);
      uint32_t word = 0;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        if ((j & 3) == 0) word = __ldg(pw + (j >> 2));
        atomicAdd(rowbase + ((size_t)((word >> (8 * (j & 3))) & 0xff) << 5), av[j]);
      }
    }
    if (VEC) {
#pragma unroll
      for (int k = 0; k < K; ++k) atomicAdd(bfirst + (size_t)k * ld + row, dot[k]);
    }
  }
}

// b_first <- b0 (+ p_surf) before the cell kernel adds R u1 (:449-465)
__global__ void k_first_init(int64_t n, const double* __restrict__ b0, const double* __restrict__ psurf,
                             double* __restrict__ bfirst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    bfirst[i] = psurf != nullptr ? b0[i] + psurf[i] : b0[i];
}

// after the cell kernel: Dirichlet rows -> identity (:470-472; their slots still hold the zero-fill), dinv = 1 / diagonal
__global__ void k_first_finalize(int n_rows, const int* __restrict__ slice_ptr, const int* __restrict__ diag_t,
                                 const uint8_t* __restrict__ is_bc_row, int scale, double* __restrict__ Avals,
                                 double* __restrict__ dinv) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  double* d = Avals + (size_t)slice_ptr[row >> 5] + (row & 31) + ((size_t)diag_t[row] << 5);
  if (is_bc_row[row]) {
    *d = 1.0;
    dinv[row] = 1.0;
  } else {
    dinv[row] = scale ? 1.0 / *d : 1.0;
  }
}

// ---- natural pressure boundary term (PressureBC, bcs.py:233-242; fracstep.py:461-465) --------------
// psurf_i[j] += int_F h n_i d(phi_j)/dx_i ds over the tagged exterior facets F (one thread per facet).
// h is a P1 function (nodal values in Q); the integrand is at most quadratic on the facet: 2-point
// Gauss on edges, the 3-point degree-2 rule on triangles.
template <int D, int DEG>
__global__ void k_pressure_surface(int64_t n_facets, const int* __restrict__ facet_cells,
                                   const int* __restrict__ facet_local, const double* __restrict__ x,
                                   const int* __restrict__ cell_nodes, const int* __restrict__ vdofs,
                                   const int* __restrict__ qdofs, int nV_owned, int ld,
                                   const double* __restrict__ h, double* __restrict__ psurf) {
  using E = El<D, DEG>;
  constexpr int NV = E::NV;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets) return;
  const int64_t c = facet_cells[t];
  const int f = facet_local[t];
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  // reference gradients of the barycentrics and their physical images
  double dl[D + 1][D], gl[D + 1][D];
#pragma unroll
  for (int a = 0; a <= D; ++a)
#pragma unroll
    for (int k = 0; k < D; ++k) dl[a][k] = a == 0 ? -1.0 : (a - 1 == k ? 1.0 : 0.0);
#pragma unroll
  for (int a = 0; a <= D; ++a)
#pragma unroll
    for (int k = 0; k < D; ++k) {
      double s = 0;
#pragma unroll
      for (int d2 = 0; d2 < D; ++d2) s += g.Kinv[d2][k] * dl[a][d2];
      gl[a][k] = s;
    }
  // outward normal times facet measure: -grad(lambda_f) * detJ / (D-1)!
  double nA[D];
#pragma unroll
  for (int k = 0; k < D; ++k) nA[k] = -gl[f][k] * g.detJ / (D == 3 ? 2.0 : 1.0);
  double hq[D + 1];
#pragma unroll
  for (int a = 0; a <= D; ++a) hq[a] = h[qdofs[c * (D + 1) + a]];
  constexpr int NQP = D == 3 ? 3 : 2;
  double acc[NV][D];
#pragma unroll
  for (int j = 0; j < NV; ++j)
#pragma unroll
    for (int k = 0; k < D; ++k) acc[j][k] = 0.0;
  for (int q = 0; q < NQP; ++q) {
    // barycentric coordinates of the quadrature point in the cell: zero on vertex f
    double lam[D + 1];
    int m = 0;
#pragma unroll
    for (int a = 0; a <= D; ++a) {
      if (a == f) { lam[a] = 0.0; continue; }
      if (D == 3) lam[a] = (m == q) ? 2.0 / 3.0 : 1.0 / 6.0;
      else lam[a] = (m == q) ? 0.5 + 0.28867513459481287 : 0.5 - 0.28867513459481287;
      ++m;
    }
    const double wq = 1.0 / NQP;
    double hv = 0;
#pragma unroll
    for (int a = 0; a <= D; ++a) hv += lam[a] * hq[a];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      double gphi[D];
      if (DEG == 1 || j <= D) {
        const double cf = DEG == 1 ? 1.0 : 4.0 * lam[j] - 1.0;
#pragma unroll
        for (int k = 0; k < D; ++k) gphi[k] = cf * gl[j][k];
      } else {
        // edge dof: basix order e0=(2,3), e1=(1,3), e2=(1,2), e3=(0,3), e4=(0,2), e5=(0,1) / e0=(1,2), e1=(0,2), e2=(0,1)
        const int e = j - (D + 1);
        int a, b;
        if (D == 3) {
          const int ea[6] = {2, 1, 1, 0, 0, 0}, eb[6] = {3, 3, 2, 3, 2, 1};
          a = ea[e];
          b = eb[e];
        } else {
          const int ea[3] = {1, 0, 0}, eb[3] = {2, 2, 1};
          a = ea[e];
          b = eb[e];
        }
#pragma unroll
        for (int k = 0; k < D; ++k) gphi[k] = 4.0 * (lam[a] * gl[b][k] + lam[b] * gl[a][k]);
      }
#pragma unroll
      for (int k = 0; k < D; ++k) acc[j][k] = fma(wq * hv * nA[k], gphi[k], acc[j][k]);
    }
  }
  for (int j = 0; j < NV; ++j) {
    const int row = vdofs[c * NV + j];
    if (row >= nV_owned) continue;
#pragma unroll
    for (int k = 0; k < D; ++k) atomicAdd(psurf + (size_t)k * ld + row, acc[j][k]);
  }
}

// ---- functionals (assemble_scalar, demo/taylor_green.py:186-207) ----------------------------------
// out += sum over cells, quadrature points and components of |detJ| w_q (u_h,k(x_q) - exact[c][q][k])^2.
// The exact field is evaluated by the host at the physical quadrature points (it is a Python callable).
// SPACE_V: vec is component-major with K comps of the velocity element; !SPACE_V: P1, K = 1.
template <int D, int DEG, bool SPACE_V>
__global__ void __launch_bounds__(128)
k_l2_error(int64_t n_cells, const double* __restrict__ x, const int* __restrict__ cell_nodes,
           const int* __restrict__ cdofs, int K, int ld, const double* __restrict__ vec, int n_q,
           const double* __restrict__ ref_pts, const double* __restrict__ weights,
           const double* __restrict__ exact, double* out, double* partials, unsigned* counter) {
  using E = El<D, DEG>;
  constexpr int ND = SPACE_V ? E::NV : E::NQ;
  constexpr bool P2 = SPACE_V && DEG == 2;
  double s[1] = {0.0};
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cells; c += (int64_t)gridDim.x * blockDim.x) {
    Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
    int dofs[ND];
#pragma unroll
    for (int j = 0; j < ND; ++j) dofs[j] = cdofs[c * ND + j];
    for (int q = 0; q < n_q; ++q) {
      double lam[D + 1];
      lam[0] = 1.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        lam[k + 1] = ref_pts[q * D + k];
        lam[0] -= lam[k + 1];
      }
      double phi[ND];
      if (!P2) {
#pragma unroll
        for (int j = 0; j < ND; ++j) phi[j] = lam[j];
      } else {
#pragma unroll
        for (int j = 0; j <= D; ++j) phi[j] = lam[j] * (2.0 * lam[j] - 1.0);
        if (D == 3) {
          const int ea[6] = {2, 1, 1, 0, 0, 0}, eb[6] = {3, 3, 2, 3, 2, 1};
#pragma unroll
          for (int e = 0; e < 6; ++e) phi[(D + 1 + e) < ND ? (D + 1 + e) : 0] = 4.0 * lam[ea[e]] * lam[eb[e]];
        } else {
          const int ea[3] = {1, 0, 0}, eb[3] = {2, 2, 1};
#pragma unroll
          for (int e = 0; e < 3; ++e) phi[(D + 1 + e) < ND ? (D + 1 + e) : 0] = 4.0 * lam[ea[e]] * lam[eb[e]];
        }
      }
      for (int k = 0; k < K; ++k) {
        double uh = 0.0;
#pragma unroll
        for (int j = 0; j < ND; ++j) uh = fma(phi[j], vec[(size_t)k * ld + dofs[j]], uh);
        const double e = uh - exact[((size_t)c * n_q + q) * K + k];
        s[0] = fma(g.detJ * weights[q], e * e, s[0]);
      }
    }
  }
  double total[1];
  if (grid_reduce<1>(s, partials, counter, total) && threadIdx.x == 0) out[0] = total[0];
}

// The same functional with the exact field evaluated ON THE DEVICE from a short list of trigonometric product terms
//   exact_k(x) = sum_m c_m F(f1_m, a_m . x + a0_m) F(f2_m, b_m . x + b0_m),   F(0, s) = 1, F(1, s) = sin s, F(2, s) = cos s
// (terms[m] = {c, a[3], a0, b[3], b0, f1, f2, component}: 12 doubles) -- the Taylor-Green fields of
// demo/taylor_green.py:41-53,176-191, also rotated, are sums of two such terms per component.  A call moves a few
// hundred bytes to the device instead of cells x points x components doubles (27 GB at 96^3 with a degree-10 rule).
template <int D, int DEG, bool SPACE_V>
__global__ void __launch_bounds__(128)
k_l2_error_trig(int64_t n_cells, const double* __restrict__ x, const int* __restrict__ cell_nodes,
                const int* __restrict__ cdofs, int K, int ld, const double* __restrict__ vec, int n_q,
                const double* __restrict__ ref_pts, const double* __restrict__ weights, int n_terms,
                const double* __restrict__ terms, double* out, double* partials, unsigned* counter) {
  using E = El<D, DEG>;
  constexpr int ND = SPACE_V ? E::NV : E::NQ;
  constexpr bool P2 = SPACE_V && DEG == 2;
  double s[1] = {0.0};
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cells; c += (int64_t)gridDim.x * blockDim.x) {
    Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
    double X[D + 1][3];
    for (int v = 0; v <= D; ++v)
      for (int k = 0; k < 3; ++k) X[v][k] = x[3 * (size_t)cell_nodes[c * (D + 1) + v] + k];
    int dofs[ND];
#pragma unroll
    for (int j = 0; j < ND; ++j) dofs[j] = cdofs[c * ND + j];
    for (int q = 0; q < n_q; ++q) {
      double lam[D + 1];
      lam[0] = 1.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        lam[k + 1] = ref_pts[q * D + k];
        lam[0] -= lam[k + 1];
      }
      double xq[3] = {0.0, 0.0, 0.0};
      for (int v = 0; v <= D; ++v)
        for (int k = 0; k < 3; ++k) xq[k] = fma(lam[v], X[v][k], xq[k]);
      double phi[ND];
      if (!P2) {
#pragma unroll
        for (int j = 0; j < ND; ++j) phi[j] = lam[j];
      } else {
#pragma unroll
        for (int j = 0; j <= D; ++j) phi[j] = lam[j] * (2.0 * lam[j] - 1.0);
        if (D == 3) {
          const int ea[6] = {2, 1, 1, 0, 0, 0}, eb[6] = {3, 3, 2, 3, 2, 1};
#pragma unroll
          for (int e = 0; e < 6; ++e) phi[(D + 1 + e) < ND ? (D + 1 + e) : 0] = 4.0 * lam[ea[e]] * lam[eb[e]];
        } else {
          const int ea[3] = {1, 0, 0}, eb[3] = {2, 2, 1};
#pragma unroll
          for (int e = 0; e < 3; ++e) phi[(D + 1 + e) < ND ? (D + 1 + e) : 0] = 4.0 * lam[ea[e]] * lam[eb[e]];
        }
      }
      double ex[3] = {0.0, 0.0, 0.0};
      for (int m = 0; m < n_terms; ++m) {
        const double* t = terms + 12 * m;
        const double sa = t[1] * xq[0] + t[2] * xq[1] + t[3] * xq[2] + t[4];
        const double sb = t[5] * xq[0] + t[6] * xq[1] + t[7] * xq[2] + t[8];
        const int f1 = (int)t[9], f2 = (int)t[10], comp = (int)t[11];
        const double v1 = f1 == 0 ? 1.0 : (f1 == 1 ? sin(sa) : cos(sa));
        const double v2 = f2 == 0 ? 1.0 : (f2 == 1 ? sin(sb) : cos(sb));
        if (comp < 3) ex[comp] = fma(t[0], v1 * v2, ex[comp]);
      }
      for (int k = 0; k < K; ++k) {
        double uh = 0.0;
#pragma unroll
        for (int j = 0; j < ND; ++j) uh = fma(phi[j], vec[(size_t)k * ld + dofs[j]], uh);
        const double e = uh - ex[k];
        s[0] = fma(g.detJ * weights[q], e * e, s[0]);
      }
    }
  }
  double total[1];
  if (grid_reduce<1>(s, partials, counter, total) && threadIdx.x == 0) out[0] = total[0];
}

// ---- right-hand side of an L2 projection (Projector, function.py:108-119): out_k[i] += int f_k phi_i dx -----------
// The source f is sampled at the quadrature points of each cell either by the host (a Python callable: `fq`,
// [cell][q][n_comp]) or on the device from the nodal values of a Lagrange function on the same mesh (`src`,
// n_src_comp components, component-major with leading dimension ld_src): its value (DERIV < 0) or its derivative
// along x_DERIV, or -- GRAD -- all gdim derivatives of ONE scalar function as the gdim components of f (grad(u) into
// a vector space, test/test_projector.py:33).  TDEG / SDEG: degree of the target / source space.
template <int D, int TDEG, int SDEG>
__global__ void __launch_bounds__(128)
k_project_rhs(int64_t n_cells, const double* __restrict__ x, const int* __restrict__ cell_nodes,
              const int* __restrict__ tdofs, int n_t_owned, int ld_t, const int* __restrict__ sdofs, int ld_src,
              const double* __restrict__ src, const double* __restrict__ fq, int n_comp, int deriv, int grad, int n_q,
              const double* __restrict__ ref_pts, const double* __restrict__ weights, double* __restrict__ out) {
  constexpr int NT = TDEG == 1 ? D + 1 : (D == 2 ? 6 : 10);
  constexpr int NS = SDEG == 1 ? D + 1 : (D == 2 ? 6 : 10);
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  const Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  auto basis = [](const double (&lam)[D + 1], int deg, double* phi, double (*dphi)[D]) {
    // values and REFERENCE gradients (d/dxi_dl) of the Lagrange basis in the basix dof order (SURVEY.md Appendix C)
    double dl[D + 1][D];
    for (int a = 0; a <= D; ++a)
      for (int k = 0; k < D; ++k) dl[a][k] = a == 0 ? -1.0 : (a - 1 == k ? 1.0 : 0.0);
    if (deg == 1) {
      for (int a = 0; a <= D; ++a) {
        phi[a] = lam[a];
        for (int k = 0; k < D; ++k) dphi[a][k] = dl[a][k];
      }
      return;
    }
    for (int a = 0; a <= D; ++a) {
      phi[a] = lam[a] * (2.0 * lam[a] - 1.0);
      for (int k = 0; k < D; ++k) dphi[a][k] = (4.0 * lam[a] - 1.0) * dl[a][k];
    }
    const int ea3[6] = {2, 1, 1, 0, 0, 0}, eb3[6] = {3, 3, 2, 3, 2, 1}, ea2[3] = {1, 0, 0}, eb2[3] = {2, 2, 1};
    const int ne = D == 3 ? 6 : 3;
    for (int e = 0; e < ne; ++e) {
      const int a = D == 3 ? ea3[e] : ea2[e], b = D == 3 ? eb3[e] : eb2[e];
      phi[D + 1 + e] = 4.0 * lam[a] * lam[b];
      for (int k = 0; k < D; ++k) dphi[D + 1 + e][k] = 4.0 * (lam[a] * dl[b][k] + lam[b] * dl[a][k]);
    }
  };
  double acc[NT][3];
  for (int i = 0; i < NT; ++i)
    for (int k = 0; k < 3; ++k) acc[i][k] = 0.0;
  for (int q = 0; q < n_q; ++q) {
    double lam[D + 1];
    lam[0] = 1.0;
    for (int k = 0; k < D; ++k) {
      lam[k + 1] = ref_pts[q * D + k];
      lam[0] -= lam[k + 1];
    }
    double f[3] = {0.0, 0.0, 0.0};
    if (fq != nullptr) {
      for (int k = 0; k < n_comp; ++k) f[k] = fq[((size_t)c * n_q + q) * n_comp + k];
    } else {
      double sphi[NS], sdphi[NS][D];
      basis(lam, SDEG, sphi, sdphi);
      if (grad) {  // f_k = d u / d x_k of the scalar source
        double gr[D];
        for (int dd = 0; dd < D; ++dd) gr[dd] = 0.0;
        for (int j = 0; j < NS; ++j) {
          const double uj = src[sdofs[c * NS + j]];
          for (int dd = 0; dd < D; ++dd) gr[dd] = fma(uj, sdphi[j][dd], gr[dd]);
        }
        for (int k = 0; k < D; ++k) {
          double v = 0.0;
          for (int dd = 0; dd < D; ++dd) v = fma(g.Kinv[dd][k], gr[dd], v);
          f[k] = v;
        }
      } else {
        for (int k = 0; k < n_comp; ++k) {
          double v = 0.0;
          for (int j = 0; j < NS; ++j) {
            const double uj = src[(size_t)k * ld_src + sdofs[c * NS + j]];
            double b = sphi[j];
            if (deriv >= 0) {
              b = 0.0;
              for (int dd = 0; dd < D; ++dd) b = fma(g.Kinv[dd][deriv], sdphi[j][dd], b);
            }
            v = fma(uj, b, v);
          }
          f[k] = v;
        }
      }
    }
    double tphi[NT], tdphi[NT][D];
    basis(lam, TDEG, tphi, tdphi);
    const double wq = g.detJ * weights[q];
    for (int i = 0; i < NT; ++i)
      for (int k = 0; k < n_comp; ++k) acc[i][k] = fma(wq * tphi[i], f[k], acc[i][k]);
  }
  for (int i = 0; i < NT; ++i) {
    const int row = tdofs[c * NT + i];
    if (row >= n_t_owned) continue;
    for (int k = 0; k < n_comp; ++k) atomicAdd(out + (size_t)k * ld_t + row, acc[i][k]);
  }
}

// ---- low_memory_version=True: matrix-free element vectors (fracstep.py:305-309,327-330,342-346) -----
// MODE 0: out_k[j] += int s dphi_j/dx_k          (s in Q: p* for :485-497, out = rhs1 preloaded with b_first)
// MODE 1: out_k[j] += int ds/dx_k phi_j          (s in Q: dp for :612-622)
// MODE 2: outq[q]  += int (sum_k du_k/dx_k) psi_q (u in V: div(u) q for :537-538)
// One thread per local cell; rows beyond the owned range are skipped (the ghost-cell layer makes owned
// rows complete, so no reverse scatter is needed).
template <int D, int DEG, int MODE>
__global__ void __launch_bounds__(128)
k_lowmem_vector(int64_t n_cells, const double* __restrict__ x, const int* __restrict__ cell_nodes,
                const int* __restrict__ vdofs, const int* __restrict__ qdofs, int nV_owned, int nQ_owned, int ld,
                const double* __restrict__ in, double scale, double* __restrict__ out) {
  using E = El<D, DEG>;
  constexpr int NV = E::NV, NQ = E::NQ;
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  Geo<D> g = cell_geometry<D>(x, cell_nodes + c * (D + 1));
  const double f = scale * g.detJ;
  if constexpr (MODE == 0 || MODE == 1) {
    double sq[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) sq[q] = __ldg(in + qdofs[c * NQ + q]);
    for (int j = 0; j < NV; ++j) {
      const int row = vdofs[c * NV + j];
      if (row >= nV_owned) continue;
      double gr[D];  // reference-direction sums  sum_q T[dl][j][q] s_q
#pragma unroll
      for (int dl = 0; dl < D; ++dl) {
        double a = 0;
#pragma unroll
        for (int q = 0; q < NQ; ++q) a = fma(MODE == 0 ? E::PX(dl, j, q) : E::GX(dl, j, q), sq[q], a);
        gr[dl] = a;
      }
#pragma unroll
      for (int k = 0; k < D; ++k) {
        double v = 0;
#pragma unroll
        for (int dl = 0; dl < D; ++dl) v = fma(g.Kinv[dl][k], gr[dl], v);
        atomicAdd(out + (size_t)k * ld + row, f * v);
      }
    }
  } else {
    double acc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = 0.0;
    for (int j = 0; j < NV; ++j) {
      const int dof = vdofs[c * NV + j];
      // w[dl] = sum_k Kinv[dl][k] u_k[dof]
      double w[D];
#pragma unroll
      for (int dl = 0; dl < D; ++dl) w[dl] = 0.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        const double uk = __ldg(in + (size_t)k * ld + dof);
#pragma unroll
        for (int dl = 0; dl < D; ++dl) w[dl] = fma(g.Kinv[dl][k], uk, w[dl]);
      }
#pragma unroll
      for (int q = 0; q < NQ; ++q)
#pragma unroll
        for (int dl = 0; dl < D; ++dl) acc[q] = fma(w[dl], E::PX(dl, j, q), acc[q]);
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int row = qdofs[c * NQ + q];
      if (row < nQ_owned) atomicAdd(out + row, f * acc[q]);
    }
  }
}
