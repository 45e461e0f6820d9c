/*
 * b200ipcs.h -- C ABI of libb200ipcs.so: the B200 (sm_100a) implementation of the oasisx IPCS
 * fractional-step time loop.
 *
 * oasisx itself has no FFI layer: every numerical call of the hot path goes from
 * src/oasisx/fracstep.py into DOLFINx (C++ assemblers + FFCx tabulate_tensor kernels) and PETSc
 * (Mat/Vec/KSP).  This header is the boundary a maintainer binds instead (ctypes stub in
 * INTEGRATION.md); each entry point names the reference lines it replaces.  All paths are relative
 * to /root/reference.
 *
 * Conventions
 *   - plain pointers and sizes only; host arrays are BORROWED for the duration of the call and
 *     copied to the device -- the library never keeps a host pointer;
 *   - every function returns 0 on success and a negative code on failure; b2_last_error() gives
 *     the message (CUDA error string included);
 *   - one host thread per context; calls are ordered on one CUDA stream owned by the context;
 *   - solver stages report PETSc KSPConvergedReason integers (>0 converged: 2 RTOL, 3 ATOL;
 *     <0 diverged: -3 ITS, -5 BREAKDOWN, -9 NANORINF), as the reference's callers assert on
 *     them (fracstep.py:681,684);
 *   - FP64 values, int32 indices (fracstep.py:63); velocity-space vectors are stored on the
 *     device component-major (component k at offset k * n_local: one contiguous array per
 *     component, as the reference's per-component Functions) and addressed through `comp`;
 *     comp = -1 moves the blocked [dof][gdim] view of `solver.u` (fracstep.py:698-705).
 */
#ifndef B200IPCS_H
#define B200IPCS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2_ctx b2_ctx;

#define B2_ABI_VERSION 1
#define B2_NCCL_UID_BYTES 128

/* function spaces: V = one velocity component (all components share it, fracstep.py:190),
 * Q = pressure (fracstep.py:212) */
enum { B2_SPACE_V = 0, B2_SPACE_Q = 1 };

/* CSR patterns of `create_matrix` (fracstep.py:293-352): rows x columns */
enum { B2_PAT_VV = 0, B2_PAT_VQ = 1, B2_PAT_QV = 2, B2_PAT_QQ = 3 };

/* matrices; comp selects i for the three per-direction families */
enum {
  B2_MAT_M = 0,  /* _M   u*v              fracstep.py:292,373 */
  B2_MAT_K = 1,  /* _K   grad u.grad v    fracstep.py:297-300,375 */
  B2_MAT_A = 2,  /* _A   convection / LHS fracstep.py:294,435-472 */
  B2_MAT_AP = 3, /* _Ap  grad p.grad q    fracstep.py:321-324,379 */
  B2_MAT_P = 4,  /* _p_vdxi_Mat[i]  p*dv/dx_i   fracstep.py:311-315,395 */
  B2_MAT_G = 5,  /* _grad_p_Mat[i]  dp/dx_i*v   fracstep.py:348-352,399 */
  B2_MAT_D = 6,  /* _divu_Mat[i]    du/dx_i*q   fracstep.py:332-336,403 */
  B2_MAT_MQ = 7  /* Projector mass matrix on Q, function.py:63-71 */
};

/* state vectors (fracstep.py:191-216) */
enum {
  B2_VEC_U = 0,      /* _u[i]      */
  B2_VEC_U1 = 1,     /* _u1[i]     */
  B2_VEC_U2 = 2,     /* _u2[i]     */
  B2_VEC_UAB = 3,    /* _uab[i]    */
  B2_VEC_RHS1 = 4,   /* _rhs1[i]   */
  B2_VEC_BFIRST = 5, /* _b_first[i]*/
  B2_VEC_B0 = 6,     /* _b0[i]     */
  B2_VEC_PSURF = 7,  /* assembled _p_surf[i] (PressureBC natural term, fracstep.py:461-465) */
  B2_VEC_B3 = 8,     /* _b3 for all components */
  B2_VEC_WRK = 9,    /* _wrk_comp for all components */
  B2_VEC_PS = 16,    /* _ps */
  B2_VEC_P = 17,     /* _p  */
  B2_VEC_DP = 18,    /* _dp */
  B2_VEC_B2 = 19,    /* _b2 */
  B2_VEC_MQ = 20     /* int psi_q dx (row sums of the Q mass matrix; used for the mean, :581-591) */
};

/* the three KSPSolver instances of fracstep.py:231-255 (+ the Projector's, function.py:84) */
enum { B2_SOLVER_TENTATIVE = 0, B2_SOLVER_PRESSURE = 1, B2_SOLVER_SCALAR = 2, B2_SOLVER_PROJECTOR = 3 };

typedef struct b2_stats {
  int32_t its_tentative[3]; /* Krylov iterations of the last tentative solve, per component */
  int32_t its_pressure;
  int32_t its_update[3];
  int32_t its_projector;
  int64_t kernel_launches; /* kernels launched by this context since creation */
  double ms_assemble_first, ms_tentative, ms_pressure, ms_update; /* CUDA-event times, last step */
  double ms_step;
  int64_t bytes_h2d, bytes_d2h; /* cumulative host<->device traffic through this ABI */
  int64_t halo_exchanges, allreduces; /* halo exchanges (either path) / ncclAllReduce calls enqueued since creation */
  double res0_tentative, res0_pressure, res0_update; /* |r0|/|b| of the last solves (max over components) */
  int64_t peer_kernels; /* kernels that carried a peer-memory collective (halo, scalar or vector all-reduce) */
} b2_stats;

/* ---- lifetime ------------------------------------------------------------------------ */
int b2_abi_version(void);
int b2_device_count(void);
/* Fills `uid` (B2_NCCL_UID_BYTES) on rank 0; the host layer distributes it to the other ranks. */
int b2_nccl_unique_id(void* uid);
/* One context per rank/GPU.  nranks == 1: `nccl_uid` may be NULL and NCCL is never loaded.
 * Replaces mesh.comm / PETSc communicator plumbing (fracstep.py:231-255). */
int b2_create(b2_ctx** ctx, int device, int nranks, int rank, const void* nccl_uid);
void b2_destroy(b2_ctx* ctx);
const char* b2_last_error(const b2_ctx* ctx);
/* pinned host staging buffers for callers that want async copies */
void* b2_host_alloc(int64_t bytes);
void b2_host_free(void* p);

/* ---- mesh, spaces, halos (what DOLFINx hands over: SURVEY.md Appendix D adapter list) -- */
/* mesh.geometry.x (n_nodes x 3, padded) and mesh.geometry.dofmap (n_cells x (gdim+1)); cells =
 * owned cells followed by the ghost cells that touch an owned dof. */
int b2_set_mesh(b2_ctx* ctx, int gdim, int64_t n_nodes, const double* x, int64_t n_cells,
                const int32_t* cell_nodes);
/* V.dofmap.list / Q.dofmap.list with local indices, owned dofs first then ghosts
 * (index_map.size_local / num_ghosts).  degree in {1,2}.  fracstep.py:187-190,212 */
int b2_set_space(b2_ctx* ctx, int space, int degree, int64_t n_owned, int64_t n_ghost,
                 const int32_t* cell_dofs);
/* Halo plan of one space (index_map.ghosts/owners turned into pack lists): for neighbour k,
 * send the owned entries send_idx[send_off[k]:send_off[k+1]] and receive into the ghost block
 * [n_owned + recv_off[k], n_owned + recv_off[k+1]).  Replaces Vector.scatter_forward and the
 * implicit MatMult gather (SURVEY.md 5.8). */
int b2_set_halo(b2_ctx* ctx, int space, int n_neighbors, const int32_t* neighbor_ranks,
                const int64_t* send_off, const int32_t* send_idx, const int64_t* recv_off);
/* Peer-memory collectives between the ranks of one NVSwitch box (replaces the MPI_Neighbor_alltoallv /
 * MPI_Allreduce traffic of DOLFINx Scatterer and PETSc KSP, SURVEY.md 5.8, WITHOUT a library call per
 * exchange): every rank exports an arena through CUDA IPC, the host layer all-gathers the
 * B2_PEER_BLOB_BYTES blobs over its own channel (mpi4py / oasisx_b200.comm) and hands them back.  After
 * segment 0 is imported, halo exchanges are one kernel (remote stores into the neighbours' staging +
 * release flag + wait + unpack) and the Krylov dot products are all-reduced inside the reducing kernel;
 * segment 1 (after the pressure multigrid is attached) carries the replicated coarse right-hand side.
 * Call order: b2_set_halo (both spaces) -> export(0) -> import(0) [-> mg levels -> export(1) -> import(1)].
 * If a rank cannot map a peer the call fails and the context keeps the NCCL path; the host layer must
 * then call b2_peer_disable on EVERY rank (the choice has to be the same everywhere). */
#define B2_PEER_BLOB_BYTES 256
int b2_peer_export(b2_ctx* ctx, int segment, void* blob);
int b2_peer_import(b2_ctx* ctx, int segment, const void* blobs /* [nranks][B2_PEER_BLOB_BYTES] */);
int b2_peer_disable(b2_ctx* ctx);
int b2_peer_enabled(b2_ctx* ctx); /* 1: peer-memory path active, 0: NCCL path */
/* Global (all-rank) sizes for the two means of fracstep.py:573-591. */
int b2_set_global_sizes(b2_ctx* ctx, int64_t n_global_v, int64_t n_global_q);

/* ---- sparsity (create_matrix, fracstep.py:293,294,300,315,324,336,352) ---------------- */
int b2_build_patterns(b2_ctx* ctx);
int64_t b2_pattern_nnz(b2_ctx* ctx, int pattern);
/* Layout statistics of a square pattern's sliced-ELL form: slots (padded entries) and the number of 32-entry slice
 * columns whose column indices form a run c0..c0+31 (their index loads are skipped by the SpMM).  -1 if unavailable. */
int64_t b2_pattern_sell_slots(b2_ctx* ctx, int pattern);
/* Optional schedule for the sliced-ELL kernels on a square pattern: a permutation of the 32-row slices
 * that lists them spatial tile by spatial tile, so that one thread block gathers from one
 * neighbourhood of the vector (host-side analogue of DOLFINx's graph reordering [ext]).  Results do
 * not depend on it. */
int b2_set_slice_order(b2_ctx* ctx, int pattern, int64_t n_slices, const int32_t* order);
/* copies indptr (n_rows+1) and indices (nnz) back: the bit-exact CSR check of north_star */
int b2_get_pattern(b2_ctx* ctx, int pattern, int32_t* indptr, int32_t* indices);

/* ---- boundary conditions (bcs.py:116-139, 245-253) ------------------------------------ */
/* merged dof list of all DirichletBCs of velocity component `comp` (local indices) */
int b2_set_velocity_bc_dofs(b2_ctx* ctx, int comp, int64_t n, const int32_t* dofs);
/* g_i at those dofs, same order: the result of update_bc() + what set_bc reads (bcs.py:128-139) */
int b2_set_velocity_bc_values(b2_ctx* ctx, int comp, int64_t n, const double* values);
/* Prefetch g_i for `n_steps` consecutive time steps ([n_steps][n], device resident) and pick the
 * one the next tentative solve applies: lets a driver evaluate time-dependent callables ahead of the
 * device and keeps the per-step H2D copy out of the step (update_bc, bcs.py:128-133). */
int b2_set_velocity_bc_series(b2_ctx* ctx, int comp, int n_steps, int64_t n, const double* values);
int b2_select_bc_step(b2_ctx* ctx, int step);
/* cudaProfilerStart / cudaProfilerStop after draining the stream: delimits the region `ncu --profile-from-start off`
 * (or nsys --capture-range=cudaProfilerApi) records, e.g. the timed steps of bench.py without the set-up kernels. */
int b2_profiler_range(b2_ctx* ctx, int on);
/* Forget the solution histories behind the extrapolated initial guesses (b200_guess) and the predicted iteration
 * counts: call when the state vectors are re-initialised to start another run on the same context. */
int b2_reset_time_history(b2_ctx* ctx);
/* homogeneous Dirichlet dofs of the pressure correction (bcs.py:245-253): LOCAL dofs, owned and ghost (the ghost ones
 * are needed to zero the matching columns of the owned rows, fracstep.py:379-380). */
int b2_set_pressure_bc_dofs(b2_ctx* ctx, int64_t n, const int32_t* dofs);
/* Multi-rank: whether ANY rank holds pressure Dirichlet dofs (len(bcs_p) > 0 in fracstep.py:381-384,562). A rank whose
 * slab touches none of them must still skip the null-space handling, collectively with the others. Call before
 * b2_set_pressure_bc_dofs / b2_preassemble; single-rank callers need not call it. */
int b2_declare_pressure_bcs(b2_ctx* ctx, int any);

/* ---- pressure multigrid hierarchy (optional; selected with pc_type=mg on B2_SOLVER_PRESSURE) --------
 * The reference forces a direct (MUMPS) solve of the singular pressure system (fracstep.py:562-578); at
 * 10^6 unknowns the device equivalent is PCG preconditioned by a geometric multigrid V-cycle (damped
 * Jacobi smoothing).  The host supplies, coarser level by coarser level, the level's P1 mesh (dofs = mesh
 * nodes) and the transfer operators as CSR: P (rows = OWNED dofs of the previous level, cols = this
 * level) and R = P^T (rows = this level, cols = local dofs of the previous level).  Coarse levels are
 * replicated on every rank; only the restriction to level 1 is all-reduced.  Call after b2_preassemble.
 * The first coarse level with at most 5000 dofs is solved exactly (dense inverse of the stiffness shifted by the
 * constant mode, built on the device by Gauss-Jordan); deeper levels, if supplied, are then never visited.
 * Defaults: V(1,1), damping 0.85, overridden by b2_pressure_mg_configure (coarse_sweeps: Jacobi sweeps on the last
 * level when no level qualifies for the exact solve). */
int b2_pressure_mg_add_level(b2_ctx* ctx, int64_t n_nodes, const double* x, int64_t n_cells, const int32_t* cell_nodes,
                             int64_t n_fine_rows, const int32_t* P_indptr, const int32_t* P_indices, const double* P_vals,
                             const int32_t* R_indptr, const int32_t* R_indices, const double* R_vals);
/* nu_pre, nu_post and coarse_sweeps apply to both kinds of hierarchy; omega is the damping of GEOMETRIC levels only
 * (an algebraic hierarchy damps every level, the fine one included, with its own 4 / (3 rho_l)). */
int b2_pressure_mg_configure(b2_ctx* ctx, int nu_pre, int nu_post, int coarse_sweeps, double omega);
/* Smoothed-aggregation algebraic multigrid built on the device from the assembled pressure matrix Ap, for meshes
 * without a nested hierarchy (pc_type gamg / hypre).  Strength graph: every nonzero off-diagonal entry.  Aggregates:
 * MIS(2) of that graph with hash keys (Bell, Dalton and Olson 2012).  P = (I - 4/(3 rho) D^-1 A) T with T the
 * aggregate indicator, R = P^T, A_c = R A P, repeated until a level has at most 5000 dofs (solved exactly), the
 * coarsening ratio drops below 2, or 15 coarse levels; rho = 20 power iterations on D^-1 A.  Deterministic: the same
 * Ap gives the same hierarchy bit for bit.  Call after b2_preassemble on a context without multigrid levels;
 * otherwise an error.  Pressure Dirichlet dofs (b2_set_pressure_bc_dofs) join no aggregate: their rows of P_1 are
 * zero, A_1 is the Galerkin operator of the interior block, and the exact coarse solve takes no null-space shift.  A
 * Dirichlet row of Ap with a nonzero off-diagonal entry fails the build.
 * Several ranks (collective; b2_set_pressure_global_ids first; one rank takes the same path once it has been given
 * global ids, numbering the hierarchy by them): the owned rows of Ap and their Dirichlet flags of all ranks are
 * gathered over NCCL into the global matrix and mask, and every rank builds the same hierarchy from them.  Levels 2 and below are global and
 * replicated; level 1 keeps this rank's part only: P_1 the rows of its owned dofs (local order), R_1 = P_1^T with
 * local columns (ghost columns empty), the aggregates of its owned dofs.  Set-up memory on every GPU: the global
 * matrix and its sort buffers (DESIGN.md section 2). */
int b2_pressure_amg_build(b2_ctx* ctx);
/* Global index of every local pressure dof, owned then ghost (n = n_owned + n_ghost), for the multi-rank algebraic
 * multigrid.  Collective on several ranks.  Every index lies in [0, n_global) (b2_set_global_sizes; n_global <= 2^31,
 * the pair keys of the set-up are row << 32 | col), no rank lists an index twice, and the owned indices of all ranks
 * cover 0 .. n_global-1 exactly once; otherwise an error on every rank. */
int b2_set_pressure_global_ids(b2_ctx* ctx, int64_t n, const int64_t* gids);
/* out[7] = {n, nnz(A_l), nnz(P_l), algebraic (0/1), solved densely (0/1), omega_l, rho_hat_l} of level `level`
 * (0 = the fine level: nnz(P) = 0; rho_hat = 0 on geometric levels).  On several ranks n and nnz of level 0 and
 * nnz(P_1) are this rank's. */
int b2_pressure_mg_level_info(b2_ctx* ctx, int level, double* out);
/* Test hook: level >= 1, what = 0: A_l as CSR with sorted columns, 1: P_l, 2: R_l (indptr, indices, vals; sizes from
 * b2_pressure_mg_level_info); 3 (algebraic levels): `indices` receives the aggregate of every dof of level - 1. */
int b2_pressure_mg_get_level(b2_ctx* ctx, int level, int what, int32_t* indptr, int32_t* indices, double* vals);

/* ---- _preassemble (fracstep.py:360-409) ----------------------------------------------- */
int b2_preassemble(b2_ctx* ctx, const double* body_force, int low_memory, int rotational);

/* ---- state access (Function.x.array, fracstep.py:432-434,673,689-693) ----------------- */
/* comp >= 0: one component (n = dofs of the space incl. ghosts); comp == -1 on a velocity vector:
 * the whole interleaved array (n = gdim * dofs) */
int b2_set_vector(b2_ctx* ctx, int vec, int comp, const double* host, int64_t n);
int b2_get_vector(b2_ctx* ctx, int vec, int comp, double* host, int64_t n);
/* Mat.getValuesCSR() values (test/test_tentative_velocity.py:28) in pattern order */
int b2_get_matrix_values(b2_ctx* ctx, int mat, int comp, double* host);
/* y = Mat * x on host arrays (Mat.mult; parity-test hook) */
int b2_mat_mult(b2_ctx* ctx, int mat, int comp, const double* x, double* y);

/* ---- solver options (ksp.py:38-53; SURVEY.md Appendix G) ------------------------------ */
/* GMRES keys (solver slots TENTATIVE, SCALAR and PROJECTOR; ksp_type gmres on the PRESSURE slot fails):
 *   ksp_type gmres                       restarted GMRES(m), left preconditioned with pc_type jacobi (or none);
 *   ksp_gmres_restart m                  restart length, 1 <= m <= 100 (default 30), anything else fails;
 *   ksp_gmres_cgs_refinement_type t      refine_never (default): one classical Gram-Schmidt pass per step;
 *                                        refine_always: two passes; refine_ifneeded runs two passes as well.
 * ksp_gmres_modifiedgramschmidt is not built and, like every unknown key, ignored.  Iterations count Arnoldi steps
 * over all restarts; the convergence test compares the Arnoldi residual estimate (and, at each restart, the true
 * preconditioned residual) with max(rtol |D^-1 b|, atol). */
int b2_set_solver_option(b2_ctx* ctx, int solver, const char* key, const char* value);

/* ---- the stages, one-to-one with the reference methods -------------------------------- */
int b2_assemble_first(b2_ctx* ctx, double dt, double nu);        /* fracstep.py:411-472 */
int b2_tentative_assemble(b2_ctx* ctx);                          /* fracstep.py:474-506 */
int b2_tentative_solve(b2_ctx* ctx, double* diff, int32_t* reasons); /* fracstep.py:508-525 */
int b2_pressure_assemble(b2_ctx* ctx, double dt);                /* fracstep.py:527-551 */
int b2_pressure_solve(b2_ctx* ctx, double nu, int32_t* reason);  /* fracstep.py:553-605 */
int b2_velocity_update(b2_ctx* ctx, double dt, int32_t* reasons);/* fracstep.py:607-658 */
/* Optional first half of a step: p* <- p and assemble_first (fracstep.py:673,676), enqueued without waiting,
 * so that the caller can evaluate this step's Dirichlet callables on the host meanwhile; b2_step then
 * continues from there.  (The velocity BC values are first read by the tentative solve, :517-518.) */
int b2_step_begin(b2_ctx* ctx, double dt, double nu);
/* whole step (fracstep.py:660-696) with the BC values already uploaded */
int b2_step(b2_ctx* ctx, double dt, double nu, double max_error, int max_iter, double* diff);

/* Natural pressure boundary term of PressureBC (bcs.py:233-242, assembled at fracstep.py:461-465):
 * B2_VEC_PSURF_i[j] (+)= int h n_i d(phi_j)/dx_i ds over the given exterior facets (local cell index,
 * local facet index = index of the opposite vertex), h nodal in Q.  Call before b2_assemble_first;
 * accumulate = 0 zeroes the vector first (one call per PressureBC). */
int b2_assemble_pressure_surface(b2_ctx* ctx, int64_t n_facets, const int32_t* facet_cells, const int32_t* facet_local,
                                 const double* h_nodal, int accumulate);

/* ---- Projector (function.py:48-133) ------------------------------------------------------
 * assemble_rhs (:108-119): b_k[i] = int f_k phi_i dx on the target space (B2_SPACE_V: the velocity component space,
 * B2_SPACE_Q), n_comp <= 3 components.  The source f is either nodal values of a Lagrange function of `src_space`
 * on the same mesh ([n_comp][n_local], component-major) -- its value (deriv < 0), its derivative along x_deriv, or,
 * with grad = 1, the gdim derivatives of ONE scalar function as the components (grad(u), test/test_projector.py:33)
 * -- or values sampled by the caller at the quadrature points (f_quad [cells][n_q][n_comp]; a Python callable).
 * solve (:121-133): M x_k = b_k with the options of B2_SOLVER_PROJECTOR; x is [n_comp][n_local], ghosts refreshed. */
int b2_project_assemble(b2_ctx* ctx, int target_space, int n_comp, int src_space, const double* src_nodal, int deriv,
                        int grad, int n_q, const double* ref_points, const double* weights, const double* f_quad);
int b2_project_get_rhs(b2_ctx* ctx, double* rhs);
/* solve(assemble_rhs=False) with a right-hand side the caller kept: [n_comp][n_local] */
int b2_project_set_rhs(b2_ctx* ctx, int target_space, int n_comp, const double* rhs);
int b2_project_solve(b2_ctx* ctx, double* x, int32_t* reasons);
/* Dirichlet conditions of the projection (function.py:70 assemble_matrix(lhs, bcs), :114-118 apply_lifting + set_bc):
 * x_k[dofs[i]] = values[k][i] (values: [n_comp][n]); applied by b2_project_solve; n = 0 removes them. */
int b2_project_set_bcs(b2_ctx* ctx, int target_space, int n_comp, int64_t n, const int32_t* dofs, const double* values);
/* KSPSolver.solve (ksp.py:71-78): Mat x = b with the options of solver slot `solver`, then scatter_forward;
 * b and x are host vectors of the operator's space (owned + ghosts), x is the initial guess when
 * ksp_initial_guess_nonzero is set.  Square operators only (B2_MAT_M, _K, _A, _AP, _MQ).  A solve on the pressure
 * slot reports its iterations in b2_stats.its_pressure. */
int b2_ksp_solve(b2_ctx* ctx, int solver, int mat, const double* b, double* x, int32_t* reason);

/* ---- functionals (assemble_scalar, demo/taylor_green.py:204-207) ----------------------- */
/* sum_k int (u_h,k - e_k)^2 dx where e is given nodally in a P2 (or P1 for Q) space of the same
 * mesh: `exact` has the layout of the vector it is compared with. */
int b2_l2_diff_sq(b2_ctx* ctx, int vec, const double* exact, int64_t n, double* out);
/* The reference's own error functional: sum_k int (u_h,k - e_k)^2 dx by quadrature on the first `n_cells`
 * local cells (the owned ones), e evaluated by the caller at the physical images of the n_q reference
 * points (`exact` is [n_cells][n_q][K]); summed over ranks. */
int b2_l2_error_quadrature(b2_ctx* ctx, int vec, int64_t n_cells, int n_q, const double* ref_points,
                           const double* weights, const double* exact, double* out);

/* ---- measurement ---------------------------------------------------------------------- */
/* The same functional with the exact field evaluated on the device from `n_terms` trigonometric product terms
 * (12 doubles each: c, a[3], a0, b[3], b0, f1, f2, component; value c F(f1, a.x + a0) F(f2, b.x + b0) with
 * F(0,.) = 1, F(1,.) = sin, F(2,.) = cos): the Taylor-Green fields of demo/taylor_green.py:41-53,176-191.  Moves a
 * few hundred bytes instead of cells x points x components doubles. */
int b2_l2_error_trig(b2_ctx* ctx, int vec, int64_t n_cells_owned, int n_q, const double* ref_points, const double* weights,
                     int n_terms, const double* terms, double* out);
/* demo/assembly_strategies.py:56-152 on the device: right-hand side (M/dt - nu/2 K - 1/2 C(UAB)) U1 by the
 * "matvec strategy" (one fused pass over the three assembled value arrays, result in RHS1; reference timed block
 * :128-133) and by the "action strategy" (matrix-free element kernel, result in BFIRST; :137-140), each averaged over
 * `reps` launches (CUDA events).  out[6] = ms of {convection assembly, matvec, action}, then their algorithmic bytes. */
int b2_bench_assembly_strategies(b2_ctx* ctx, double dt, double nu, int reps, double* out);
/* Cell schedule of assemble_first (k_first_cells): out[4] = schedule built (0/1), congruence classes found, slab
 * thickness in reference lengths (always 1), cells.  b2_set_tuning "first_order" 0 keeps the mesh order. */
int b2_first_plan_info(b2_ctx* ctx, int64_t* out);
int b2_get_stats(b2_ctx* ctx, b2_stats* out);
/* Times `reps` launches of one hot kernel on the context's stream with CUDA events (device
 * resident operands).  kernel: 0 = SpMM A*u (gdim RHS), 1 = assemble_first (k_first_cells and its row passes),
 * 2 = SpMV Ap*dp, 3 = SpMM M*u; multi-rank only (every rank must call): 10 = halo exchange of a Q vector, 11 = of a
 * V vector (gdim components), 12 = all-reduce of 3 doubles, 13 = sum of the replicated multigrid level.  Returns
 * average ms per launch and the algorithmic bytes moved. */
int b2_bench_kernel(b2_ctx* ctx, int kernel, int reps, double* ms_per_launch, double* bytes_per_launch);
int b2_synchronize(b2_ctx* ctx);
/* Alternative schedules kept as references for the tests: "first_order" (0: assemble_first in mesh order instead
 * of the congruence-class cell schedule), "mg_dense" (0: the pressure multigrid smooths down to its coarsest level
 * instead of solving the first small one exactly).  Any other key is an error. */
int b2_set_tuning(b2_ctx* ctx, const char* key, int value);
/* CUDA events on the context's stream (slots 0..7) for callers that time a region of stage calls. */
int b2_event_record(b2_ctx* ctx, int slot);
int b2_event_elapsed_ms(b2_ctx* ctx, int slot_start, int slot_stop, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* B200IPCS_H */
