// b200ipcs.cu -- context, sparsity builder, stage drivers and the C ABI of libb200ipcs.so.
// See include/b200ipcs.h for the contract and the reference lines each entry point replaces.
#include "../../include/b200ipcs.h"

#include <cub/cub.cuh>
#include <cuda_profiler_api.h>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library is dlopen'ed when a multi-rank context is created

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "elem.cuh"
#include "linalg.cuh"
#include "mg.cuh"
#include "amg.cuh"
#include "gmres.cuh"

namespace {

std::string g_last_error;

struct CSR {
  DBuf<int> rowptr, cols;
  int n_rows = 0, n_cols = 0;
  int64_t nnz = 0;
  // SELL-32 layout of the same pattern, where build_sell made one (every operator pattern but Q x V; see linalg.cuh)
  DBuf<int> slice_ptr, scols, diag_t, order;  // order: optional tile-major slice schedule
  int64_t slots = 0;
  bool has_sell() const { return slice_ptr.p != nullptr; }
};

struct Space {
  int degree = 0, nd = 0;           // dofs per cell
  int64_t n_owned = 0, n_ghost = 0; // local = owned + ghost
  int64_t n_global = 0;
  DBuf<int> cell_dofs;
  int64_t n_local() const { return n_owned + n_ghost; }
};

struct KSPOpts {
  int type = 0;  // 0 = cg, 1 = bcgs, 2 = chebyshev (mass solves: needs eig bounds, b2_set_solver_option ksp_chebyshev_eigenvalues), 3 = gmres
  int restart = 30;     // GMRES restart length m (ksp_gmres_restart)
  bool cgs2 = false;    // GMRES: a second classical Gram-Schmidt pass (ksp_gmres_cgs_refinement_type refine_always)
  double eig_lo = 0.0, eig_hi = 0.0;  // bounds of the spectrum of D^-1 A for type 2
  int pc = 0;    // 0 = jacobi, 1 = none, 2 = multigrid (pressure only, needs b2_pressure_mg_add_level)
  double rtol = 1e-5, atol = 1e-50;
  int maxit = 10000;
  bool nonzero_guess = false;
  bool block_rtol = false;  // "b200_block_rtol": rtol relative to max over the components' |b_k|
  bool extrapolate_guess = false;  // "b200_guess": "extrapolate" -- start from a time-extrapolated state (implies nonzero guess)
  int guess_order = 1;             // "extrapolate2": quadratic extrapolation of the solver's own solution history (u*, u - u*)
  bool scaled_operator = false;  // the matrix is stored row-scaled by its diagonal (tentative velocity)
  int expected_its = 0;  // iterations of the previous solve: first batch enqueued without a host sync
};

// NCCL entry points resolved at run time (no link-time dependency; single-rank runs never load it)
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  void load() {
    if (lib) return;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) throw B2Error(-30, std::string("cannot dlopen libnccl.so.2: ") + dlerror());
    auto sym = [&](const char* n) {
      void* p = dlsym(lib, n);
      if (!p) throw B2Error(-30, std::string("NCCL symbol missing: ") + n);
      return p;
    };
    GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
    GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
    Send = (decltype(Send))sym("ncclSend");
    Recv = (decltype(Recv))sym("ncclRecv");
    AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
    AllGather = (decltype(AllGather))sym("ncclAllGather");
    GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
  }
};
NcclApi g_nccl;

#define B2_NCCL(expr)                                                                               \
  do {                                                                                              \
    ncclResult_t _r = (expr);                                                                       \
    if (_r != ncclSuccess) throw B2Error(-31, std::string(#expr) + ": " + g_nccl.GetErrorString(_r)); \
  } while (0)

struct Halo {
  int n_neighbors = 0;
  std::vector<int> ranks;
  std::vector<int64_t> send_off, recv_off;  // host copies
  DBuf<int64_t> d_send_off, d_recv_off;
  DBuf<int> send_idx;
  DBuf<double> sendbuf, recvbuf;
};

// one replicated coarse level of the pressure multigrid (level 0 is the distributed fine space)
struct MgLevel {
  int n = 0;  // dofs (P1: = nodes of the level's mesh)
  CSR pat;
  DBuf<double> A, dinv, x, b, r, tmp;
  // transfer operators to/from the previous (finer) level, CSR with scalar values
  CSR P, R;  // P: rows = owned dofs of the finer level, cols = this level;  R = P^T
  DBuf<double> Pv, Rv;
  // algebraic levels (b2_pressure_amg_build): own damping 4 / (3 rho), rho = estimated spectral radius of D^-1 A, and
  // the aggregate of every dof of the finer level.  Geometric levels keep omega = 0: they smooth with ctx->mg_omega.
  bool algebraic = false;
  double omega = 0.0, rho = 0.0;
  DBuf<int> agg;
};

// one IPC-exported allocation of this rank and the peers' mappings of theirs
struct PeerSeg {
  void* base = nullptr;
  size_t bytes = 0;
  void* peer[B2_MAXR] = {};
  bool imported = false;
};

// byte offsets inside segment 0 (identical on every rank up to the staging block)
enum : size_t {
  PEER_OFF_SEQ = 128,        // u64 seq_red, seq_halo[2], seq_mg, err (local use only)
  PEER_OFF_SLOT_RED = 512,   // LLSlot [2][B2_MAXR][B2_RED_MAX]
  PEER_OFF_STAGE = 512 + 2 * B2_MAXR * B2_RED_MAX * sizeof(LLSlot)
};

// what travels with an IPC handle through the host channel (b2_peer_export / b2_peer_import)
struct PeerBlob {
  cudaIpcMemHandle_t handle;        // 64 bytes
  int64_t cap[2];                   // segment 0: staging capacity (doubles) per space; segment 1: [n, 0]
  int64_t recv_cnt[2][B2_MAXR];     // segment 0: ghosts received from each rank, per space; segment 1: [0][0..1] = lo, hi
  int64_t pad[6];
};
static_assert(sizeof(PeerBlob) == B2_PEER_BLOB_BYTES, "PeerBlob size");

struct FirstPlanHost {
  DBuf<int> cell_order;   // cells by congruence class, slab by slab (build_first_plan)
  int64_t n_classes = 0;
  bool ready = false;
};

struct DVec {
  DBuf<double> buf;
  int K = 1;
  int space = 0;
};

}  // namespace

struct b2_ctx {
  int device = 0, nranks = 1, rank = 0, sm = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  int gdim = 0;
  int64_t n_nodes = 0, n_cells = 0;
  DBuf<double> x;
  DBuf<int> cell_nodes;
  Space sp[2];
  CSR pat[4];
  Halo halo[2];
  std::vector<MgLevel> mg;  // coarse levels 1..L of the pressure hierarchy
  // V(1,1) with omega = 0.85: measured best at 96^3 (9 iterations of 0.33 ms against 7 of 0.46 ms for V(2,2), omega 0.8;
  // 6/7 is the optimal damping of the 7-point stencil the Kuhn P1 stiffness reduces to); b2_pressure_mg_configure overrides
  int mg_pre = 1, mg_post = 1, mg_coarse = 16;
  double mg_omega = 0.85;
  double mg_omega0 = 0.0, mg_rho0 = 0.0;  // fine-level damping and rho(D^-1 Ap) of an algebraic hierarchy (0: geometric)
  DBuf<double> mg_x0, mg_t0;  // fine-level work vectors (n_local of Q)
  DBuf<MgDev> mg_dev;         // device descriptors of the coarse levels (index = level - 1)
  int mg_dev_levels = 0;      // number of levels the descriptor array was built for
  int mg_small_from = 1 << 30; // first level (>= 1) handled by the single-block kernel
  int mg_dense_max = 5000;     // the first coarse level with at most this many dofs is solved exactly (dense inverse); 0 = off
  int mg_dense_level = -1;     // index into mg (level - 1) of that level, -1: none
  int mg_dense_on = 1;         // tuning "mg_dense": 0 falls back to smoothing all the way down (A/B comparisons)
  DBuf<double> mg_dense;       // (A_l + alpha e e^T)^-1, row-major
  double** d_mg_result = nullptr; double** h_mg_result = nullptr;
  ncclComm_t comm = nullptr;
  double* d_red = nullptr;  // raw reduction totals awaiting the all-reduce (multi rank, NCCL path)
  // peer-memory collectives (common.cuh): arenas mapped through CUDA IPC, no NCCL call on the data path
  int use_peer = 1;         // B200_PEER=0 keeps the NCCL path (A/B measurements, boxes without P2P)
  bool peer_on = false;     // segment 0 imported: halo + scalar all-reduce run through peer memory
  PeerSeg seg[2];           // 0: flags, scalar slots, halo staging; 1: staging of the replicated multigrid level
  PeerDev h_peer{};
  PeerDev* d_peer = nullptr;
  PeerHalo ph[2];
  PeerVecSum pvs{};
  bool pvs_ready = false;
  int mg_lo = 0, mg_hi = 0;  // range of level-1 dofs this rank's restriction touches
  unsigned* d_counter_peer = nullptr;
  unsigned long long* h_peer_err = nullptr;  // pinned copy of the arena's error word
  bool patterns_built = false, preassembled = false;
  bool low_memory = false, rotational = false;
  // matrices: values in the SELL slots of their pattern, P and G component-major; D in CSR order, [nnz][gdim]
  DBuf<double> M, Kst, A, Ap, MQ, P, G, D;
  DBuf<double> dinvA, dinvM, dinvAp, dinvMQ, onesV, onesQ;
  // boundary conditions
  DBuf<int> bc_dofs[B2_MAXK];
  DBuf<double> bc_vals[B2_MAXK];
  DBuf<double> bc_series[B2_MAXK];  // [n_steps][n] prefetched values
  int bc_series_steps[B2_MAXK] = {0, 0, 0};
  int bc_step = -1;                 // >= 0: apply bc_series[.][bc_step] instead of bc_vals
  DBuf<uint8_t> is_bc_row_v, is_bc_q;
  DBuf<uint8_t> pos8;  // per-cell scatter table of the convection assembly (elem.cuh)
  int maxlen_vv = 0;        // longest row of the P2xP2 pattern
  FirstPlanHost first;      // cell schedule of assemble_first (build_first_plan)
  int first_order = 1;      // tuning "first_order": 1 = congruence-class cell order (coalesced scatter), 0 = mesh order
  // CUDA graph of one multigrid-preconditioned CG iteration of the pressure solve (single rank): ~21 dependent
  // launches of a few microseconds each become one graph launch
  cudaGraphExec_t pcg_graph = nullptr;
  uint64_t pcg_graph_version = 0, cfg_version = 1;  // cfg_version: bumped by everything the captured body depends on
  const double* pcg_graph_x = nullptr;
  const double* pcg_graph_b = nullptr;
  int pcg_graph_launches = 0;
  DBuf<int> pbc_dofs;
  bool has_pbc = false;
  DBuf<int> q_gid;  // global id of every local pressure dof (b2_set_pressure_global_ids): the multi-rank algebraic set-up
  double vol = 0.0;  // sum of mQ over all ranks
  std::map<int, DVec> vecs;
  // Krylov work space
  DBuf<double> wv[5], wq[4];
  DBuf<double> wproj[5];    // Projector / KSPSolver.solve work vectors (any space, up to 3 components)
  DBuf<double> proj_rhs;    // right-hand side of the last b2_project_assemble
  int proj_space = 0, proj_comp = 1;
  // Dirichlet conditions of a Projector (function.py:70,114-118), per target space: dofs, values per component, the mass
  // matrix with their rows and columns replaced by the identity, its inverse diagonal
  struct ProjBC {
    DBuf<int> dofs;
    DBuf<double> vals;  // [n_comp][n]
    DBuf<uint8_t> mask;
    DBuf<double> Mbc, dinv;
    int n_comp = 0;
  } proj_bc[2];
  DBuf<double> stage;  // staging for strided host copies
  DBuf<double> dp_old;      // pressure correction of the step before the previous one (extrapolated guess)
  int dp_hist = 0;
  DBuf<double> delta_prev;  // previous velocity correction u - u* (initial guess of the next mass solve)
  // "extrapolate2": the last three tentative velocities u* and corrections u - u* (index 0 = newest)
  DBuf<double> ustar_hist[3], delta_hist[3];
  int n_ustar_hist = 0, n_delta_hist = 0;
  bool fresh_step = true;  // assemble_first ran since the last tentative solve: its solution opens a new history entry
  int steps_done = 0;
  bool step_begun = false;  // b2_step_begin was called for the step b2_step is about to finish
  KryState* d_st = nullptr;
  KryState* h_st = nullptr;  // pinned
  GmresState* d_gm = nullptr;  // GMRES Hessenberg / Givens state, allocated by the first GMRES solve
  DBuf<double> gm_V;           // GMRES basis: m+1 vectors of K components, vector i component k at (i K + k) ld
  double* d_sums = nullptr;  // small device scratch for reductions (16 doubles)
  double* h_sums = nullptr;  // pinned
  DBuf<double> partials;
  unsigned* d_counter = nullptr;
  KSPOpts ksp[4];
  b2_stats stats{};
  cudaEvent_t ev[6];
  cudaEvent_t user_ev[8];
  double last_dt = 0.0;

  double* vec(int id) {
    auto it = vecs.find(id);
    if (it == vecs.end()) throw B2Error(-2, "unknown vector id " + std::to_string(id));
    return it->second.buf.p;
  }
};

namespace {

// ---- launch helpers -------------------------------------------------------------------------
#define B2_LAUNCH(ctx, kernel, grid, block, ...)                         \
  do {                                                                   \
    kernel<<<(grid), (block), 0, (ctx)->stream>>>(__VA_ARGS__);          \
    (ctx)->stats.kernel_launches++;                                      \
    B2_CUDA(cudaGetLastError());                                         \
  } while (0)

inline int blocks_for(int64_t n, int block) { return (int)std::max<int64_t>(1, (n + block - 1) / block); }

// most blocks of a peer-memory halo / vector-sum kernel (two values per thread)
constexpr int PEER_GRID_MAX = 128;

// persistent grid for grid-stride kernels: enough blocks to fill the machine, never more than needed
inline int pgrid(const b2_ctx* c, int64_t n_items, int block = 256, int per_sm = 8) {
  int64_t need = (n_items + block - 1) / block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)c->sm * per_sm));
}

void alloc_vec(b2_ctx* c, int id, int space, int K) {
  DVec& v = c->vecs[id];
  v.K = K;
  v.space = space;
  v.buf.alloc(c->sp[space].n_local() * K);
  v.buf.zero(c->stream);
}

// ---- sparsity builder (create_matrix): keys = row<<32|col, radix sort, unique -----------------
__global__ void k_gen_keys(int64_t n_cells, const int* __restrict__ rdofs, int nr,
                           const int* __restrict__ cdofs, int nc, int n_rows_owned,
                           unsigned long long* __restrict__ keys) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = n_cells * nr * nc;
  if (t >= total) return;
  int64_t c = t / (nr * nc);
  int rem = (int)(t - c * nr * nc);
  int i = rem / nc, j = rem - i * nc;
  int row = rdofs[c * nr + i];
  int col = cdofs[c * nc + j];
  if (row >= n_rows_owned) { row = n_rows_owned; col = 0; }  // parked after the owned rows
  keys[t] = ((unsigned long long)(unsigned)row << 32) | (unsigned)col;
}

__global__ void k_keys_to_csr(int64_t n_keys, const unsigned long long* __restrict__ keys,
                              int n_rows, int* __restrict__ rowptr, int* __restrict__ cols) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n_keys) return;
  // row of this key (n_rows == "past the end" for i == n_keys or parked keys)
  int r = (i < n_keys) ? (int)min((unsigned long long)n_rows, keys[i] >> 32) : n_rows;
  int rprev = (i == 0) ? -1 : (int)min((unsigned long long)n_rows, keys[i - 1] >> 32);
  for (int rr = rprev + 1; rr <= r; ++rr) rowptr[rr] = (int)i;
  if (i < n_keys && r < n_rows) cols[i] = (int)(keys[i] & 0xffffffffull);
}

void build_pattern_raw(b2_ctx* c, int64_t n_cells, const int* rdofs, int nr, const int* cdofs, int nc, int n_rows,
                       int n_cols, CSR& out);

void build_pattern(b2_ctx* c, const Space& rs, const Space& cs, CSR& out) {
  build_pattern_raw(c, c->n_cells, rs.cell_dofs.p, rs.nd, cs.cell_dofs.p, cs.nd, (int)rs.n_owned, (int)cs.n_local(), out);
}

void build_pattern_raw(b2_ctx* c, int64_t n_cells, const int* rdofs, int nr, const int* cdofs, int nc, int n_rows,
                       int n_cols, CSR& out) {
  const int64_t n_pairs = n_cells * nr * nc;
  DBuf<unsigned long long> k0, k1;
  k0.alloc(n_pairs);
  k1.alloc(n_pairs);
  B2_LAUNCH(c, k_gen_keys, blocks_for(n_pairs, 256), 256, n_cells, rdofs, nr, cdofs, nc, n_rows, k0.p);
  int row_bits = 1;
  while ((1ll << row_bits) <= (int64_t)n_rows + 1) ++row_bits;
  size_t tmp_bytes = 0;
  B2_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, k0.p, k1.p, n_pairs, 0, 32 + row_bits, c->stream));
  DBuf<char> tmp;
  tmp.alloc((int64_t)tmp_bytes);
  B2_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, k0.p, k1.p, n_pairs, 0, 32 + row_bits, c->stream));
  DBuf<int64_t> d_n;
  d_n.alloc(1);
  size_t tmp2 = 0;
  B2_CUDA(cub::DeviceSelect::Unique(nullptr, tmp2, k1.p, k0.p, d_n.p, n_pairs, c->stream));
  if (tmp2 > tmp_bytes) tmp.alloc((int64_t)tmp2);
  B2_CUDA(cub::DeviceSelect::Unique(tmp.p, tmp2, k1.p, k0.p, d_n.p, n_pairs, c->stream));
  int64_t n_unique = 0;
  B2_CUDA(cudaMemcpyAsync(&n_unique, d_n.p, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_REQUIRE(n_unique < (1ll << 31), "pattern too large for int32 indptr");
  out.n_rows = n_rows;
  out.n_cols = n_cols;
  out.rowptr.alloc(n_rows + 1);
  DBuf<int> cols_tmp;
  cols_tmp.alloc(n_unique);
  B2_LAUNCH(c, k_keys_to_csr, blocks_for(n_unique + 1, 256), 256, n_unique, k0.p, n_rows, out.rowptr.p, cols_tmp.p);
  int nnz = 0;
  B2_CUDA(cudaMemcpyAsync(&nnz, out.rowptr.p + n_rows, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  out.nnz = nnz;
  out.cols.alloc(nnz);
  B2_CUDA(cudaMemcpyAsync(out.cols.p, cols_tmp.p, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// SELL-32 companion of a CSR pattern: slice offsets (in slots), padded column indices, position of the
// diagonal in each row (-1 where the row has none).
void build_sell(b2_ctx* c, CSR& pat) {
  const int n_rows = pat.n_rows;
  const int n_slices = (n_rows + 31) / 32;
  DBuf<int> entries;
  entries.alloc(n_slices + 1);
  entries.zero(c->stream);
  B2_LAUNCH(c, k_sell_slice_len, blocks_for(n_slices, 256), 256, n_rows, pat.rowptr.p, entries.p);
  pat.slice_ptr.alloc(n_slices + 1);
  size_t tmp_bytes = 0;
  B2_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, entries.p, pat.slice_ptr.p, n_slices + 1, c->stream));
  DBuf<char> tmp;
  tmp.alloc((int64_t)tmp_bytes);
  B2_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, entries.p, pat.slice_ptr.p, n_slices + 1, c->stream));
  int slots = 0;
  B2_CUDA(cudaMemcpyAsync(&slots, pat.slice_ptr.p + n_slices, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  pat.slots = slots;
  pat.scols.alloc(slots);
  pat.scols.zero(c->stream);
  pat.diag_t.alloc(n_rows);
  B2_LAUNCH(c, k_sell_fill_cols, blocks_for(n_rows, 256), 256, n_rows, pat.rowptr.p, pat.cols.p, pat.slice_ptr.p, pat.scols.p, pat.diag_t.p, pat.n_cols);
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// Assembly with a fixed summation order: k_assemble_square's (slot, value) pairs in cell order, stably sorted by slot,
// each slot summed sequentially.  The same mesh gives the same bits on every run (atomicAdd does not).
template <typename Launch>
void assemble_in_fixed_order(b2_ctx* c, int64_t n_pairs, int64_t slots, double* vals, Launch&& launch) {
  B2_REQUIRE(slots < 0xffffffffll, "operator too large for 32-bit slot keys");
  DBuf<unsigned> k0, k1;
  DBuf<double> v0, v1;
  k0.alloc(n_pairs); k1.alloc(n_pairs);
  v0.alloc(n_pairs); v1.alloc(n_pairs);
  B2_CUDA(cudaMemsetAsync(k0.p, 0xff, sizeof(unsigned) * (size_t)n_pairs, c->stream));
  launch(k0.p, v0.p);
  cub::DoubleBuffer<unsigned> kb(k0.p, k1.p);
  cub::DoubleBuffer<double> vb(v0.p, v1.p);
  size_t bytes = 0;
  B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kb, vb, n_pairs, 0, 32, c->stream));
  DBuf<char> tmp;
  tmp.alloc((int64_t)bytes);
  B2_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, kb, vb, n_pairs, 0, 32, c->stream));
  B2_LAUNCH(c, k_sum_slot_runs, blocks_for(n_pairs, 256), 256, n_pairs, kb.Current(), vb.Current(), vals);
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// ---- dispatch helpers -------------------------------------------------------------------------
template <typename F>
void dispatch_elem(const b2_ctx* c, F&& f) {
  const int d = c->gdim, deg = c->sp[B2_SPACE_V].degree;
  if (d == 2 && deg == 1) f(El<2, 1>{});
  else if (d == 2 && deg == 2) f(El<2, 2>{});
  else if (d == 3 && deg == 1) f(El<3, 1>{});
  else if (d == 3 && deg == 2) f(El<3, 2>{});
  else throw B2Error(-3, "unsupported (gdim, degree)");
}

// Owner -> ghost exchange of a component-major vector before it is gathered by columns
// (Vector.scatter_forward / the implicit MatMult gather, SURVEY.md 5.8): pack kernel, grouped
// ncclSend/ncclRecv with every neighbour, unpack kernel.  Single rank: nothing to do.
void halo_forward(b2_ctx* c, int space, double* v, int K) {
  if (c->nranks == 1) return;
  Halo& h = c->halo[space];
  if (h.n_neighbors == 0) return;
  const Space& S = c->sp[space];
  const int ld = (int)S.n_local();
  const int64_t ns = h.send_off.back(), nr = h.recv_off.back();
  if (c->peer_on) {  // one kernel: remote stores into the neighbours' staging, signal, wait, unpack
    // few, fat blocks: every block polls the neighbours' flags, and the exchange is latency-, not bandwidth-bound
    const int grid = std::min(PEER_GRID_MAX, blocks_for(std::max(ns, nr) * K, 512));
    B2_LAUNCH(c, k_halo_peer, grid, 256, c->ph[space], K, ld, v);
    c->stats.halo_exchanges++;
    c->stats.peer_kernels++;
    return;
  }
  if (ns > 0)
    B2_LAUNCH(c, k_halo_pack, pgrid(c, ns * K), 256, h.n_neighbors, h.d_send_off.p, h.send_idx.p, K, ld, v, h.sendbuf.p);
  B2_NCCL(g_nccl.GroupStart());
  for (int j = 0; j < h.n_neighbors; ++j) {
    const int64_t sc = h.send_off[j + 1] - h.send_off[j], rc = h.recv_off[j + 1] - h.recv_off[j];
    if (sc > 0) B2_NCCL(g_nccl.Send(h.sendbuf.p + K * h.send_off[j], (size_t)(K * sc), ncclDouble, h.ranks[j], c->comm, c->stream));
    if (rc > 0) B2_NCCL(g_nccl.Recv(h.recvbuf.p + K * h.recv_off[j], (size_t)(K * rc), ncclDouble, h.ranks[j], c->comm, c->stream));
  }
  B2_NCCL(g_nccl.GroupEnd());
  if (nr > 0)
    B2_LAUNCH(c, k_halo_unpack, pgrid(c, nr * K), 256, h.n_neighbors, h.d_recv_off.p, K, ld, (int)S.n_owned, h.recvbuf.p, v);
  c->stats.halo_exchanges++;
}

// sum over ranks of n doubles on the device (KSP reductions / comm.allreduce)
void allreduce_sum(b2_ctx* c, double* d, int n) {
  if (c->nranks == 1) return;
  if (c->peer_on) {
    for (int off = 0; off < n; off += B2_RED_MAX) {
      B2_LAUNCH(c, k_peer_allreduce, 1, 32, c->d_peer, d + off, std::min(B2_RED_MAX, n - off));
      c->stats.peer_kernels++;
    }
    return;
  }
  B2_NCCL(g_nccl.AllReduce(d, d, (size_t)n, ncclDouble, ncclSum, c->comm, c->stream));
  c->stats.allreduces++;
}

// k int64 values of every rank, in rank order (set-up only)
std::vector<int64_t> allgather_i64(b2_ctx* c, const int64_t* mine, int k) {
  std::vector<int64_t> out(mine, mine + k);
  if (c->nranks == 1) return out;
  DBuf<int64_t> d;
  d.alloc((int64_t)k * (c->nranks + 1));
  out.resize((size_t)k * c->nranks);
  B2_CUDA(cudaMemcpyAsync(d.p, mine, sizeof(int64_t) * k, cudaMemcpyHostToDevice, c->stream));
  B2_NCCL(g_nccl.AllGather(d.p, d.p + k, (size_t)k, ncclInt64, c->comm, c->stream));
  B2_CUDA(cudaMemcpyAsync(out.data(), d.p + k, sizeof(int64_t) * k * c->nranks, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return out;
}

// The blocks of every rank, counts[q] elements of `bytes` each, concatenated in rank order into `recv` on the device
// (set-up only): grouped ncclSend/ncclRecv with every other rank, this rank's own block copied in place.
void allgatherv(b2_ctx* c, const void* send, const std::vector<int64_t>& counts, void* recv, ncclDataType_t type, size_t bytes) {
  const int me = c->rank;
  int64_t off = 0;
  for (int q = 0; q < me; ++q) off += counts[q];
  if (counts[me] > 0)
    B2_CUDA(cudaMemcpyAsync((char*)recv + off * bytes, send, counts[me] * bytes, cudaMemcpyDeviceToDevice, c->stream));
  if (c->nranks > 1) {
    B2_NCCL(g_nccl.GroupStart());
    off = 0;
    for (int q = 0; q < c->nranks; ++q) {
      if (q != me && counts[me] > 0) B2_NCCL(g_nccl.Send(send, (size_t)counts[me], type, q, c->comm, c->stream));
      if (q != me && counts[q] > 0) B2_NCCL(g_nccl.Recv((char*)recv + off * bytes, (size_t)counts[q], type, q, c->comm, c->stream));
      off += counts[q];
    }
    B2_NCCL(g_nccl.GroupEnd());
  }
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// after a reducing Krylov kernel: (multi rank) all-reduce the raw totals and run the scalar update
void reduce_finish_host(b2_ctx* c, int fin, int n, bool is_init = false) {
  if (c->nranks == 1 || c->peer_on) return;  // peer path: all-reduced and finalized inside the reducing kernel
  allreduce_sum(c, c->d_red, n);
  B2_LAUNCH(c, k_kry_finalize, 1, 1, fin, c->d_st, c->d_red, (int)is_init);
}
inline RedCtl red_ptr(b2_ctx* c) {
  if (c->nranks == 1) return RedCtl{nullptr, nullptr};
  return c->peer_on ? RedCtl{nullptr, c->d_peer} : RedCtl{c->d_red, nullptr};
}

template <int K, int DOT>
void launch_spmm(b2_ctx* c, const CSR& pat, const double* vals, const double* x, int ld, double* y, const double* w,
                 KryState* st, int fin, const double* rscale) {
  constexpr int BLOCK = 256;
  const int n_slices = (pat.n_rows + 31) / 32;
  const int need = (n_slices + BLOCK / 32 - 1) / (BLOCK / 32);
  // Every warp takes the same whole number k of slices (k = 1 when the grid fits): a fixed persistent grid quantises
  // small operators -- the 1/4 or 1/8 slab of a multi-GPU run got 3.07 slices per warp, i.e. 3 or 4: 103 us against 86
  // on the 96 x 96 x 12 slab -- and is no faster on large ones.  The cap is what the grid-wide reduction has room for
  // (one set of partial sums per block).
  const int cap = (int)std::min<int64_t>(c->partials.n / 16, (int64_t)c->sm * 32);
  const int k_slices = std::max(1, (need + cap - 1) / cap);
  const int grid = std::max(1, (need + k_slices - 1) / k_slices);
  B2_REQUIRE(grid <= cap, "SpMM grid exceeds the reduction scratch");
#define B2_SPMM(RS_)                                                                                                   \
  B2_LAUNCH(c, (k_spmm<K, DOT, BLOCK, RS_>), grid, BLOCK, pat.n_rows, pat.slice_ptr.p, pat.scols.p, vals, pat.order.p, x, \
            ld, y, w, st, fin, c->partials.p, c->d_counter, red_ptr(c), rscale)
  if (rscale != nullptr) B2_SPMM(true);
  else B2_SPMM(false);
#undef B2_SPMM
  if (DOT > 0) reduce_finish_host(c, fin, DOT * K);
}

template <int K>
void launch_spmm_k(b2_ctx* c, const CSR& pat, const double* vals, const double* x, int ld, double* y, const double* w,
                   KryState* st, int fin, int dot, const double* rscale) {
  if (dot == 0) launch_spmm<K, 0>(c, pat, vals, x, ld, y, w, st, fin, rscale);
  else if (dot == 1) launch_spmm<K, 1>(c, pat, vals, x, ld, y, w, st, fin, rscale);
  else launch_spmm<K, 2>(c, pat, vals, x, ld, y, w, st, fin, rscale);
}

// rscale: optional row scaling of the result, y = diag(rscale) (A x)
void spmm(b2_ctx* c, const CSR& pat, const double* vals, int K, double* x, double* y, const double* w = nullptr,
          KryState* st = nullptr, int fin = FIN_NONE, int dot = 0, int xspace = -1, const double* rscale = nullptr) {
  B2_REQUIRE(pat.has_sell(), "SpMM needs the SELL layout of the pattern");
  if (xspace >= 0) halo_forward(c, xspace, x, K);
  const int ld = pat.n_cols;  // square operators: vectors of the space, owned + ghosts
  switch (K) {
    case 1: launch_spmm_k<1>(c, pat, vals, x, ld, y, w, st, fin, dot, rscale); break;
    case 2: launch_spmm_k<2>(c, pat, vals, x, ld, y, w, st, fin, dot, rscale); break;
    case 3: launch_spmm_k<3>(c, pat, vals, x, ld, y, w, st, fin, dot, rscale); break;
    default: throw B2Error(-3, "K must be 1..3");
  }
}

// ---- Krylov driver ------------------------------------------------------------------------------
template <int K>
void krylov_iterations(b2_ctx* c, const KSPOpts& o, const CSR& pat, const double* vals, const double* dinv, int space,
                       double* x, double* r, double* p, double* q, double* t, double* rhat, int n_iter) {
  const int64_t n = pat.n_rows;
  const int ld = pat.n_cols;
  const int g = pgrid(c, n, 256, 8);
  KryState* st = c->d_st;
  for (int it = 0; it < n_iter; ++it) {
    if (o.type == 0) {
      spmm(c, pat, vals, K, p, q, p, st, FIN_CG_PQ, 1, space);
      B2_LAUNCH(c, k_cg_update<K>, g, 256, n, ld, p, q, dinv, x, r, st, c->partials.p, c->d_counter, red_ptr(c));
      reduce_finish_host(c, FIN_CG_UPDATE, 2 * K);
      B2_LAUNCH(c, k_cg_p<K>, g, 256, n, ld, r, dinv, p, st);
    } else {
      spmm(c, pat, vals, K, p, q, rhat, st, FIN_BCGS_V, 1, space, dinv);          // v = D^-1 A p
      B2_LAUNCH(c, k_bcgs_s<K>, g, 256, n, ld, q, r, st);                            // s = r - alpha v
      spmm(c, pat, vals, K, r, t, r, st, FIN_BCGS_T, 2, space, dinv);             // t = D^-1 A s
      B2_LAUNCH(c, k_bcgs_update<K>, g, 256, n, ld, p, t, rhat, x, r, st, c->partials.p, c->d_counter, red_ptr(c));
      reduce_finish_host(c, FIN_BCGS_UPDATE, 2 * K);
      B2_LAUNCH(c, k_bcgs_p<K>, g, 256, n, ld, r, q, p, rhat, st);
    }
  }
}

template <int K>
void krylov_init(b2_ctx* c, const KSPOpts& o, const CSR& pat, const double* vals, const double* dinv, int space,
                 const double* b, double* x, double* r, double* p, double* q, double* rhat) {
  const int64_t n = pat.n_rows;
  const int ld = pat.n_cols;
  const int g = pgrid(c, n, 256, 8);
  const double* q0 = nullptr;
  if (o.nonzero_guess) {
    spmm(c, pat, vals, K, x, q, nullptr, nullptr, FIN_NONE, 0, space, o.type == 1 ? dinv : nullptr);
    q0 = q;
  }
  if (o.type == 0) {
    B2_LAUNCH(c, k_cg_init<K>, g, 256, n, ld, b, q0, dinv, x, r, p, c->d_st, c->partials.p, c->d_counter, red_ptr(c));
    reduce_finish_host(c, FIN_CG_INIT, 3 * K, true);
  } else {
    B2_LAUNCH(c, k_bcgs_init<K>, g, 256, n, ld, b, q0, dinv, x, r, rhat, p, c->d_st, c->partials.p, c->d_counter, red_ptr(c));
    reduce_finish_host(c, FIN_BCGS_INIT, 2 * K, true);
  }
}

// GMRES(m), left Jacobi (gmres.cuh).  Every active component is at the same Arnoldi index j, so the host knows where
// the cycles close and enqueues the solution update and the restart residual without reading the device; the state is
// read back once per batch of steps, as for the other methods.
template <int K>
void gmres_solve(b2_ctx* c, const KSPOpts& o, const CSR& pat, const double* vals, const double* dinv, int space,
                 const double* b, double* x, double* q) {
  const int64_t n = pat.n_rows;
  const int ld = pat.n_cols, m = o.restart;
  const size_t need = (size_t)(m + 1) * K * ld;
  if ((size_t)c->gm_V.n < need) c->gm_V.alloc((int64_t)need);  // 96^3, m = 30, K = 3: 5.3 GB
  if (c->d_gm == nullptr) B2_CUDA(cudaMalloc(&c->d_gm, sizeof(GmresState)));
  GmresState* gs = c->d_gm;
  KryState* st = c->d_st;
  double* V = c->gm_V.p;
  auto vec = [&](int i) { return V + (size_t)i * K * ld; };
  const int here = c->nranks == 1;  // one rank: the scalar updates run in the reducing kernels' last block
  const int g = pgrid(c, n, 256, 8);
  const int gd = (int)std::min<int64_t>(c->sm, (n + 511) / 512);  // k_gmres_dots: one set of (m+1) K partials per block
  constexpr int CH = 8;
  auto residual = [&](bool init) {  // v_0 = D^-1 (b - A x) / |.|
    const double* q0 = nullptr;
    if (!init || o.nonzero_guess) {
      spmm(c, pat, vals, K, x, q, nullptr, init ? nullptr : st, FIN_NONE, 0, space, dinv);
      q0 = q;
    }
    B2_LAUNCH(c, k_gmres_residual<K>, g, 256, n, ld, b, q0, dinv, x, vec(0), (int)init, here, gs, st, c->partials.p, c->d_counter);
    if (!here) {
      allreduce_sum(c, gs->tot, 2 * K);
      B2_LAUNCH(c, k_gmres_fin, 1, 1, init ? GM_FIN_INIT : GM_FIN_RESTART, gs, st, 0, 1, 1);
    }
    B2_LAUNCH(c, k_gmres_scale<K>, g, 256, n, ld, vec(0), gs, st);
  };
  auto step = [&](int j) {
    double* w = vec(j + 1);
    spmm(c, pat, vals, K, vec(j), w, nullptr, st, FIN_NONE, 0, space, dinv);  // w = D^-1 A v_j
    const int passes = o.cgs2 ? 2 : 1;
    for (int pass = 0; pass < passes; ++pass) {
      const int first = pass == 0, last = pass == passes - 1;
      B2_LAUNCH(c, (k_gmres_dots<K, CH>), gd, 512, n, ld, V, j, w, gs, st, c->partials.p, c->d_counter);
      if (!here) allreduce_sum(c, gs->hcol, (j + 1) * K);
      B2_LAUNCH(c, k_gmres_orth<K>, g, 256, n, ld, V, j, w, first, last, here, gs, st, c->partials.p, c->d_counter);
      if (!here) {
        allreduce_sum(c, gs->tot, K);
        B2_LAUNCH(c, k_gmres_fin, 1, 1, GM_FIN_ORTH, gs, st, j, first, last);
      }
    }
    B2_LAUNCH(c, k_gmres_scale<K>, g, 256, n, ld, w, gs, st);
  };
  auto close_cycle = [&]() {  // x += V y for every component that took steps in this cycle (not gated by `done`)
    B2_LAUNCH(c, k_gmres_backsolve, 1, 32, gs, K);
    B2_LAUNCH(c, k_gmres_update_x<K>, g, 256, n, ld, V, x, gs);
  };
  residual(true);
  int j = 0, launched = 0;
  int chunk = std::max(1, o.expected_its);
  for (;;) {
    for (int s = 0; s < chunk; ++s) {
      step(j);
      if (++j == m) {
        close_cycle();
        residual(false);
        j = 0;
      }
    }
    launched += chunk;
    B2_CUDA(cudaMemcpyAsync(c->h_st, c->d_st, sizeof(KryState), cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_d2h += sizeof(KryState);
    if (c->h_st->done || launched > o.maxit + 1) break;
    chunk = std::max(2, std::min(launched / 4, 16));
  }
  close_cycle();
}

// Solves K systems  A x_k = b_k  (interleaved storage) with the options of solver `which`.
void chebyshev_solve(b2_ctx* c, int which, const CSR& pat, const double* vals, const double* dinv, int space, int K,
                     const double* b, double* x, int32_t* reasons, int32_t* its);

void krylov_solve(b2_ctx* c, int which, const CSR& pat, const double* vals, const double* dinv_jacobi, int space,
                  int K, const double* b, double* x, int32_t* reasons, int32_t* its, DBuf<double>* work = nullptr) {
  KSPOpts& o = c->ksp[which];
  if (o.type == 2 && work == nullptr) {
    chebyshev_solve(c, which, pat, vals, dinv_jacobi, space, K, b, x, reasons, its);
    return;
  }
  DBuf<double>* w = work != nullptr ? work : (space == B2_SPACE_V ? c->wv : c->wq);
  // CG: Jacobi through dinv in the vector kernels.  BiCGStab and GMRES: left preconditioning D^-1 A x = D^-1 b -- dinv
  // scales the right-hand side in k_bcgs_init / k_gmres_residual and every operator application in the SpMM epilogue
  // (the matrix is stored as assembled).  pc_type none: dinv = 1.
  const double* dinv = (o.pc != 1) ? dinv_jacobi : (space == B2_SPACE_V ? c->onesV.p : c->onesQ.p);
  double *r = w[0].p, *p = w[1].p, *q = w[2].p, *t = nullptr, *rhat = nullptr;
  if (o.type == 1) {
    B2_REQUIRE(space == B2_SPACE_V || work != nullptr, "BiCGStab work vectors exist for the velocity space only");
    t = w[3].p;
    rhat = w[4].p;
  }
  std::memset(c->h_st, 0, sizeof(KryState));
  c->h_st->K = K;
  c->h_st->maxit = o.maxit;
  c->h_st->rtol = o.rtol;
  c->h_st->atol = o.atol;
  c->h_st->block_rtol = o.block_rtol ? 1 : 0;
  B2_CUDA(cudaMemcpyAsync(c->d_st, c->h_st, sizeof(KryState), cudaMemcpyHostToDevice, c->stream));
  auto run = [&](auto kc) {
    constexpr int KK = decltype(kc)::value;
    if (o.type == 3) {
      gmres_solve<KK>(c, o, pat, vals, dinv, space, b, x, q);
      return;
    }
    krylov_init<KK>(c, o, pat, vals, dinv, space, b, x, r, p, q, rhat);
    int chunk = std::max(1, o.expected_its);
    int launched = 0;
    for (;;) {
      krylov_iterations<KK>(c, o, pat, vals, dinv, space, x, r, p, q, t, rhat, chunk);
      launched += chunk;
      B2_CUDA(cudaMemcpyAsync(c->h_st, c->d_st, sizeof(KryState), cudaMemcpyDeviceToHost, c->stream));
      B2_CUDA(cudaStreamSynchronize(c->stream));
      c->stats.bytes_d2h += sizeof(KryState);
      if (c->h_st->done || launched > o.maxit + 1) break;
      chunk = std::max(2, std::min(launched / 4, 16));
    }
  };
  switch (K) {
    case 1: run(std::integral_constant<int, 1>{}); break;
    case 2: run(std::integral_constant<int, 2>{}); break;
    case 3: run(std::integral_constant<int, 3>{}); break;
    default: throw B2Error(-3, "K must be 1..3");
  }
  int mx = 0;
  double res0 = 0.0, bref = 0.0;
  for (int k = 0; k < K; ++k) bref = std::max(bref, c->h_st->bb[k]);
  for (int k = 0; k < K; ++k) {
    reasons[k] = c->h_st->reason[k];
    its[k] = c->h_st->its[k];
    mx = std::max(mx, c->h_st->its[k]);
    // initial residual relative to the norm the tolerance refers to (block_rtol: the largest component)
    const double ref = o.block_rtol ? bref : c->h_st->bb[k];
    if (ref > 0) res0 = std::max(res0, std::sqrt(c->h_st->rr0[k] / ref));
  }
  o.expected_its = mx;
  if (which == B2_SOLVER_TENTATIVE) c->stats.res0_tentative = res0;
  else if (which == B2_SOLVER_PRESSURE) c->stats.res0_pressure = res0;
  else if (which == B2_SOLVER_SCALAR) c->stats.res0_update = res0;
}

// ---- multigrid V-cycle on the pressure hierarchy ---------------------------------------------------
// level 0: distributed fine operator Ap (halo before every gather); levels >= 1 replicated.
struct MgView {
  int n, ld;
  const CSR* pat;
  const double *A, *dinv;
  double omega;
};

// Jacobi damping of level l: its own on an algebraic hierarchy, the configured one on a geometric one
double mg_level_omega(const b2_ctx* c, int l) {
  const double w = l == 0 ? c->mg_omega0 : c->mg[l - 1].omega;
  return w > 0.0 ? w : c->mg_omega;
}

void cgz_finish(b2_ctx* c, int fin, int n);

// first_done: x already holds the first sweep from zero (omega D^-1 b, written by the kernel that produced b);
// rz_fin >= 0: the LAST sweep also accumulates the PCG scalar product b.x_new (fine level, b = r)
void mg_sweeps(b2_ctx* c, const MgView& L, bool fine, const double* b, double*& x, double*& tmp, int n_sweeps, bool from_zero,
               bool first_done = false, int rz_fin = -1) {
  const int g = pgrid(c, L.n, 256, 8);
  int s = 0;
  if (from_zero && n_sweeps > 0) {
    if (!first_done) B2_LAUNCH(c, k_mg_first, pgrid(c, L.n), 256, (int64_t)L.n, L.dinv, b, L.omega, x);
    s = 1;
  }
  for (; s < n_sweeps; ++s) {
    if (fine) halo_forward(c, B2_SPACE_Q, x, 1);
    if (rz_fin >= 0 && s == n_sweeps - 1) {
      B2_LAUNCH(c, k_mg_sweep_rz, g, 256, L.n, L.pat->slice_ptr.p, L.pat->scols.p, L.A, L.dinv, b, x, L.omega, tmp, rz_fin, c->d_st,
                c->partials.p, c->d_counter, red_ptr(c));
      cgz_finish(c, rz_fin, 1);
    } else {
      B2_LAUNCH(c, k_mg_sweep<false>, g, 256, L.n, L.pat->slice_ptr.p, L.pat->scols.p, L.A, L.dinv, b, x, L.omega, tmp);
    }
    std::swap(x, tmp);
  }
}

void mg_build_descriptors(b2_ctx* c) {
  const int nl = (int)c->mg.size();
  std::vector<MgDev> h(nl);
  c->mg_small_from = 1 << 30;
  for (int i = 0; i < nl; ++i) {
    MgLevel& M = c->mg[i];
    h[i] = {M.n, M.P.n_rows, M.pat.slice_ptr.p, M.pat.scols.p, M.A.p, M.dinv.p, M.x.p, M.b.p, M.tmp.p,
            M.P.rowptr.p, M.P.cols.p, M.Pv.p, M.R.rowptr.p, M.R.cols.p, M.Rv.p, M.omega};
    // an algebraic hierarchy ends at its exactly solved level: the single-block sub-cycle must not smooth over it
    const bool past_dense = !M.algebraic || c->mg_dense_level < 0 || i > c->mg_dense_level;
    if (M.n <= 8192 && past_dense && c->mg_small_from == (1 << 30)) c->mg_small_from = i + 1;
  }
  if (nl - (c->mg_small_from - 1) > 15) c->mg_small_from = 1 << 30;  // shared pointer tables hold 16 levels
  c->mg_dev.alloc(nl);
  B2_CUDA(cudaMemcpyAsync(c->mg_dev.p, h.data(), sizeof(MgDev) * nl, cudaMemcpyHostToDevice, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  if (!c->d_mg_result) {
    B2_CUDA(cudaMalloc(&c->d_mg_result, sizeof(double*)));
    B2_CUDA(cudaMallocHost(&c->h_mg_result, sizeof(double*)));
  }
  c->mg_dev_levels = nl;
}

// dense inverse of (A_l + alpha e e^T) for coarse level index i (mg.cuh); alpha = A_00 / n keeps the shift at the
// scale of the operator
void mg_build_dense(b2_ctx* c, int i) {
  MgLevel& M = c->mg[i];
  const int n = M.n;
  c->mg_dense.alloc((int64_t)n * n);
  DBuf<double> rowk, colk;
  rowk.alloc(n);
  colk.alloc(n);
  double dinv0 = 0.0;
  B2_CUDA(cudaMemcpyAsync(&dinv0, M.dinv.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  const double alpha = 1.0 / (dinv0 * n);
  B2_LAUNCH(c, k_dense_from_sell, n, 128, n, M.pat.slice_ptr.p, M.pat.scols.p, M.A.p, alpha, c->mg_dense.p);
  const dim3 grid((unsigned)blocks_for(n, 256), (unsigned)n);
  for (int k = 0; k < n; ++k) {
    B2_LAUNCH(c, k_gj_pivot, blocks_for(n, 256), 256, n, k, c->mg_dense.p, rowk.p, colk.p);
    B2_LAUNCH(c, k_gj_update, grid, 256, n, k, c->mg_dense.p, rowk.p, colk.p);
  }
  B2_CUDA(cudaStreamSynchronize(c->stream));
  c->mg_dense_level = i;
}

// the end of every new coarse level, however its operator L.A (SELL) was made: inverse diagonal, work vectors, the
// exact solve if it is the first small level, and the fine-level work vectors with the first level
void mg_level_finish(b2_ctx* c, MgLevel& L) {
  L.dinv.alloc(L.n);
  B2_LAUNCH(c, k_inv_diag, blocks_for(L.n, 256), 256, L.n, L.pat.slice_ptr.p, L.pat.diag_t.p, L.A.p, L.dinv.p);
  for (auto* v : {&L.x, &L.b, &L.r, &L.tmp}) { v->alloc(L.n); v->zero(c->stream); }
  if (c->mg_dense_level < 0 && L.n <= c->mg_dense_max) mg_build_dense(c, (int)c->mg.size() - 1);
  if (c->mg.size() == 1) {
    c->mg_x0.alloc(c->sp[B2_SPACE_Q].n_local()); c->mg_x0.zero(c->stream);
    c->mg_t0.alloc(c->sp[B2_SPACE_Q].n_local()); c->mg_t0.zero(c->stream);
  }
}

// The range of level-1 dofs this rank's restriction writes nonzeros into (rows of R_1 that are not empty): what the
// peer-memory sum of the partial restrictions pushes to the other ranks.
void mg_set_restrict_range(b2_ctx* c, const int32_t* R_indptr, int n) {
  c->mg_lo = n;
  c->mg_hi = 0;
  for (int r = 0; r < n; ++r)
    if (R_indptr[r + 1] > R_indptr[r]) { c->mg_lo = std::min(c->mg_lo, r); c->mg_hi = std::max(c->mg_hi, r + 1); }
  if (c->mg_hi <= c->mg_lo) c->mg_lo = c->mg_hi = 0;
}

void csr_values(b2_ctx* c, int mat, int comp, DBuf<double>& out, const CSR** pat_out);
void amg_build(b2_ctx* c, const CSR& A0, DBuf<double> vals, const double* dinv0);
void amg_build_gathered(b2_ctx* c);

// x_l <- V-cycle(b_l), zero initial guess.  Returns the buffer that holds the result.
// first_done: x already holds omega D^-1 b; rz_fin >= 0 (level 0 only): fuse the PCG product r.z into the last post-sweep
// -- *rz_done tells the caller whether that happened.
double* mg_vcycle(b2_ctx* c, int l, const double* b, double* x, double* tmp, bool first_done = false, int rz_fin = -1,
                  bool* rz_done = nullptr) {
  if (c->mg_dev_levels != (int)c->mg.size()) mg_build_descriptors(c);
  if (l >= 1 && l - 1 == c->mg_dense_level && c->mg_dense_on) {
    // exact solve on this level: one dense mat-vec with the precomputed inverse; deeper levels are not visited
    MgLevel& M = c->mg[l - 1];
    B2_LAUNCH(c, k_dense_matvec, blocks_for((int64_t)M.n * 32, 256), 256, M.n, c->mg_dense.p, b, x);
    return x;
  }
  if (l >= c->mg_small_from) {
    // the rest of the hierarchy in one single-block kernel; b is c->mg[l-1].b by construction
    B2_LAUNCH(c, k_mg_small_cycle, 1, 1024, c->mg_dev.p, l - 1, (int)c->mg.size() - 1, c->mg_pre, c->mg_post, c->mg_coarse,
              c->mg_omega, c->d_mg_result);
    // the result lives in x or tmp of that level depending on the parity of the sweep counts
    const int last = (int)c->mg.size();
    const int sweeps = (l == last ? c->mg_coarse : c->mg_pre) - 1 + (l == last ? 0 : c->mg_post);
    return (sweeps % 2 == 0) ? c->mg[l - 1].x.p : c->mg[l - 1].tmp.p;
  }
  const bool fine = (l == 0);
  MgView L;
  if (fine) {
    const CSR& qq = c->pat[B2_PAT_QQ];
    L = {qq.n_rows, qq.n_cols, &qq, c->Ap.p, c->dinvAp.p, mg_level_omega(c, 0)};
  } else {
    MgLevel& M = c->mg[l - 1];
    L = {M.n, M.n, &M.pat, M.A.p, M.dinv.p, mg_level_omega(c, l)};
  }
  const bool coarsest = (l == (int)c->mg.size());
  if (coarsest) {
    mg_sweeps(c, L, fine, b, x, tmp, c->mg_coarse, true, first_done);
    return x;
  }
  MgLevel& C = c->mg[l];
  mg_sweeps(c, L, fine, b, x, tmp, c->mg_pre, true, first_done);
  // residual
  if (fine) halo_forward(c, B2_SPACE_Q, x, 1);
  B2_LAUNCH(c, k_mg_sweep<true>, pgrid(c, L.n, 256, 8), 256, L.n, L.pat->slice_ptr.p, L.pat->scols.p, L.A, L.dinv, b, x, 0.0, tmp);
  // restriction, with the coarse level's first sweep x_c = omega D_c^-1 b_c fused in when b_c is complete (one rank, or
  // a replicated level); partial sums of several slabs are added up first
  const bool partial = fine && c->nranks > 1;
  B2_LAUNCH(c, k_mg_restrict, blocks_for((int64_t)C.n * 8, 256), 256, C.n, C.R.rowptr.p, C.R.cols.p, C.Rv.p, tmp, C.dinv.p,
            mg_level_omega(c, l + 1), C.b.p, partial ? (double*)nullptr : C.x.p);
  if (partial) {  // coarse levels are replicated: sum the partial restrictions of the slabs
    if (c->peer_on && c->pvs_ready) {
      B2_LAUNCH(c, k_peer_vecsum, std::min(PEER_GRID_MAX, blocks_for(C.n, 1024)), 256, c->pvs, C.b.p);
      c->stats.peer_kernels++;
    } else {
      B2_REQUIRE(!c->peer_on, "peer path: import segment 1 (multigrid staging) before the first pressure solve");
      B2_NCCL(g_nccl.AllReduce(C.b.p, C.b.p, (size_t)C.n, ncclDouble, ncclSum, c->comm, c->stream));
      c->stats.allreduces++;
    }
  }
  double* xc = mg_vcycle(c, l + 1, C.b.p, C.x.p, C.tmp.p, !partial);
  // x += P xc   (rows: owned dofs of this level)
  B2_LAUNCH(c, k_mg_prolong, blocks_for(L.n, 256), 256, L.n, C.P.rowptr.p, C.P.cols.p, C.Pv.p, xc, x);
  const bool fuse_rz = rz_fin >= 0 && c->mg_post >= 1;
  mg_sweeps(c, L, fine, b, x, tmp, c->mg_post, false, false, fuse_rz ? rz_fin : -1);
  if (rz_done != nullptr) *rz_done = fuse_rz;
  return x;
}

void cgz_finish(b2_ctx* c, int fin, int n) {
  if (c->nranks == 1 || c->peer_on) return;
  allreduce_sum(c, c->d_red, n);
  B2_LAUNCH(c, k_cgz_finalize, 1, 1, fin, c->d_st, c->d_red);
}

// PCG on the pressure system with the V-cycle as preconditioner (K = 1)
void pcg_mg_solve(b2_ctx* c, const double* b, double* x, int32_t* reason, int32_t* its) {
  KSPOpts& o = c->ksp[B2_SOLVER_PRESSURE];
  const CSR& qq = c->pat[B2_PAT_QQ];
  const int64_t n = qq.n_rows;
  const int g = pgrid(c, n, 256, 8);
  double *r = c->wq[0].p, *p = c->wq[1].p, *q = c->wq[2].p;
  std::memset(c->h_st, 0, sizeof(KryState));
  c->h_st->K = 1;
  c->h_st->maxit = o.maxit;
  c->h_st->rtol = o.rtol;
  c->h_st->atol = o.atol;
  B2_CUDA(cudaMemcpyAsync(c->d_st, c->h_st, sizeof(KryState), cudaMemcpyHostToDevice, c->stream));
  const double* q0 = nullptr;
  if (o.nonzero_guess) {
    spmm(c, qq, c->Ap.p, 1, x, q, nullptr, nullptr, FIN_NONE, 0, B2_SPACE_Q);
    q0 = q;
  }
  // the first smoothing sweep of every V-cycle (x0 = omega D^-1 r) is written by the kernel that updates r
  const double omega0 = mg_level_omega(c, 0);
  B2_LAUNCH(c, k_cgz_init_x0, g, 256, n, b, q0, x, r, c->dinvAp.p, omega0, c->mg_x0.p, c->d_st, c->partials.p, c->d_counter, red_ptr(c));
  cgz_finish(c, FIN_CGZ_INIT, 2);
  // The device decides convergence; the host only has to stop enqueueing.  Iteration counts barely change
  // from one time step to the next, so nothing is polled (no pipeline drain) until one iteration short of
  // what the previous solve needed; kernels of a surplus iteration leave x untouched (st->done).
  const int first_poll = o.expected_its > 0 ? o.expected_its - 1 : 0;
  auto body = [&](int it) {
    const int rz_fin = it == 0 ? FIN_CGZ_RZ0 : FIN_CGZ_RZ;
    bool rz_done = false;
    double* z = mg_vcycle(c, 0, r, c->mg_x0.p, c->mg_t0.p, true, rz_fin, &rz_done);  // r.z fused into the last post-sweep
    if (!rz_done) {
      B2_LAUNCH(c, k_cgz_rz, g, 256, n, r, z, rz_fin, c->d_st, c->partials.p, c->d_counter, red_ptr(c));
      cgz_finish(c, rz_fin, 1);
    }
    B2_LAUNCH(c, k_cgz_p, g, 256, n, z, p, c->d_st);
    spmm(c, qq, c->Ap.p, 1, p, q, p, c->d_st, FIN_CG_PQ, 1, B2_SPACE_Q);
    B2_LAUNCH(c, k_cgz_update_x0, g, 256, n, p, q, x, r, c->dinvAp.p, omega0, c->mg_x0.p, c->d_st, c->partials.p, c->d_counter, red_ptr(c));
    cgz_finish(c, FIN_CGZ_UPDATE, 1);
  };
  // Iterations 1, 2, ... are identical streams of small dependent kernels (all scalars live in device memory):
  // captured once into a CUDA graph and replayed.  Multi-rank contexts keep plain launches (NCCL calls in between).
  const bool graphs = c->nranks == 1 || (c->peer_on && c->pvs_ready);  // no NCCL call inside the body
  for (int it = 0; it <= o.maxit; ++it) {
    if (it >= first_poll) {
      B2_CUDA(cudaMemcpyAsync(c->h_st, c->d_st, sizeof(KryState), cudaMemcpyDeviceToHost, c->stream));
      B2_CUDA(cudaStreamSynchronize(c->stream));
      c->stats.bytes_d2h += sizeof(KryState);
      if (c->h_st->done) break;
    }
    if (it == 0 || !graphs) {
      body(it);
      continue;
    }
    if (c->pcg_graph == nullptr || c->pcg_graph_version != c->cfg_version || c->pcg_graph_x != x || c->pcg_graph_b != b) {
      if (c->pcg_graph) { cudaGraphExecDestroy(c->pcg_graph); c->pcg_graph = nullptr; }
      const int64_t before = c->stats.kernel_launches;
      cudaGraph_t graph = nullptr;
      B2_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      try {
        body(it);
      } catch (...) {
        cudaStreamEndCapture(c->stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
      }
      B2_CUDA(cudaStreamEndCapture(c->stream, &graph));
      c->pcg_graph_launches = (int)(c->stats.kernel_launches - before);
      c->stats.kernel_launches = before;  // capturing launched nothing
      B2_CUDA(cudaGraphInstantiate(&c->pcg_graph, graph, 0));
      cudaGraphDestroy(graph);
      c->pcg_graph_version = c->cfg_version;
      c->pcg_graph_x = x;
      c->pcg_graph_b = b;
    }
    B2_CUDA(cudaGraphLaunch(c->pcg_graph, c->stream));
    c->stats.kernel_launches += c->pcg_graph_launches;
  }
  if (!c->h_st->done) {
    B2_CUDA(cudaMemcpyAsync(c->h_st, c->d_st, sizeof(KryState), cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  *reason = c->h_st->reason[0] != 0 ? c->h_st->reason[0] : -3;
  *its = c->h_st->its[0];
  o.expected_its = c->h_st->its[0];
  if (c->h_st->bb[0] > 0) c->stats.res0_pressure = std::sqrt(c->h_st->rr0[0] / c->h_st->bb[0]);
}

void read_sums(b2_ctx* c, int n);

// Chebyshev iteration for K SPD systems sharing `vals` (mass matrix), Jacobi-scaled, spectrum of D^-1 A in
// [eig_lo, eig_hi].  No reductions inside the iteration; the residual norm is checked after the predicted
// number of iterations and then every 4.
void chebyshev_solve(b2_ctx* c, int which, const CSR& pat, const double* vals, const double* dinv, int space, int K,
                     const double* b, double* x, int32_t* reasons, int32_t* its) {
  KSPOpts& o = c->ksp[which];
  B2_REQUIRE(o.eig_hi > o.eig_lo && o.eig_lo > 0.0, "ksp_type chebyshev needs ksp_chebyshev_eigenvalues lo,hi");
  DBuf<double>* w = space == B2_SPACE_V ? c->wv : c->wq;
  double *r = w[0].p, *d = w[1].p, *q = w[2].p;
  const int64_t n = pat.n_rows;
  const int ld = pat.n_cols;
  const int g = pgrid(c, n, 256, 8);
  const double theta = 0.5 * (o.eig_hi + o.eig_lo), delta = 0.5 * (o.eig_hi - o.eig_lo), sigma1 = theta / delta;
  const double* q0 = nullptr;
  if (o.nonzero_guess) {
    spmm(c, pat, vals, K, x, q, nullptr, nullptr, FIN_NONE, 0, space);
    q0 = q;
  }
  auto init = [&](auto kc) {
    constexpr int KK = decltype(kc)::value;
    B2_LAUNCH(c, k_cheb_init<KK>, g, 256, n, ld, b, q0, dinv, 1.0 / theta, x, r, d, c->d_sums, c->partials.p, c->d_counter);
  };
  auto update = [&](auto kc, bool norm, double c1, double c2) {
    constexpr int KK = decltype(kc)::value;
    if (norm)
      B2_LAUNCH(c, (k_cheb_update<KK, true>), g, 256, n, ld, q, dinv, c1, c2, x, r, d, c->d_sums, c->partials.p, c->d_counter);
    else
      B2_LAUNCH(c, (k_cheb_update<KK, false>), g, 256, n, ld, q, dinv, c1, c2, x, r, d, c->d_sums, c->partials.p, c->d_counter);
  };
  auto dispatch = [&](auto&& f) {
    if (K == 1) f(std::integral_constant<int, 1>{});
    else if (K == 2) f(std::integral_constant<int, 2>{});
    else f(std::integral_constant<int, 3>{});
  };
  dispatch([&](auto kc) { init(kc); });
  allreduce_sum(c, c->d_sums, 2 * K);
  read_sums(c, 2 * K);
  double tol2[B2_MAXK], need = 0.0, bbmax = 0.0;
  bool conv = true;
  for (int k = 0; k < K; ++k) bbmax = std::max(bbmax, c->h_sums[k]);
  for (int k = 0; k < K; ++k) {
    const double bb = o.block_rtol ? bbmax : c->h_sums[k], rr = c->h_sums[K + k];
    tol2[k] = std::max(o.rtol * o.rtol * bb, o.atol * o.atol);
    if (rr > tol2[k]) {
      conv = false;
      need = std::max(need, 0.5 * std::log(rr / tol2[k]));  // ln(|r0| / tol)
    }
  }
  int it = 0;
  if (!conv) {
    const double kappa = o.eig_hi / o.eig_lo;
    const double rate = (std::sqrt(kappa) - 1.0) / (std::sqrt(kappa) + 1.0);
    int next_check = std::max(1, (int)std::ceil((need + std::log(2.0)) / -std::log(rate)));
    double rho = 1.0 / sigma1;
    while (it < o.maxit) {
      spmm(c, pat, vals, K, d, q, nullptr, nullptr, FIN_NONE, 0, space);
      const double rho_new = 1.0 / (2.0 * sigma1 - rho);
      const bool check = (it + 1 >= next_check);
      dispatch([&](auto kc) { update(kc, check, rho_new * rho, 2.0 * rho_new / delta); });
      rho = rho_new;
      ++it;
      if (check) {
        allreduce_sum(c, c->d_sums, K);
        read_sums(c, K);
        conv = true;
        for (int k = 0; k < K; ++k) conv = conv && (c->h_sums[k] <= tol2[k]);
        if (conv) break;
        next_check = it + 4;
      }
    }
    // the last update already prepared the next direction; x holds the iterate of `it` steps
  }
  for (int k = 0; k < K; ++k) {
    reasons[k] = conv ? 2 : -3;
    its[k] = it;
  }
}

void require_ready(b2_ctx* c) { B2_REQUIRE(c->preassembled, "b2_preassemble has not been called"); }

// ---- cell schedule of the cell-parallel assemble_first (elem.cuh: k_first_cells) ------------------------------
// Cells are grouped by congruence class (equal edge vectors up to rounding: translates of each other) and listed,
// inside a class, along x then y then z, so that consecutive threads scatter to consecutive dofs; classes are
// interleaved slab by slab (a few cell layers in z) to keep the accumulated rows resident in L2.  No lattice is
// assumed: a mesh without congruent cells yields one class per cell and keeps its (z, y, x) order.
void build_first_plan(b2_ctx* c) {
  const int d = c->gdim;
  const int64_t nc = c->n_cells;
  FirstPlanHost& P = c->first;
  P = FirstPlanHost();
  if (nc == 0 || c->first_order == 0) return;
  std::vector<double> x((size_t)c->n_nodes * 3);
  std::vector<int> cn((size_t)nc * (d + 1));
  B2_CUDA(cudaMemcpyAsync(x.data(), c->x.p, sizeof(double) * x.size(), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaMemcpyAsync(cn.data(), c->cell_nodes.p, sizeof(int) * cn.size(), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  // reference length: mean edge of the first cells' first edges
  double h = 0.0;
  const int64_t ns = std::min<int64_t>(nc, 4096);
  for (int64_t e = 0; e < ns; ++e) {
    double l2 = 0;
    for (int k = 0; k < d; ++k) {
      const double v = x[3 * (size_t)cn[e * (d + 1) + 1] + k] - x[3 * (size_t)cn[e * (d + 1)] + k];
      l2 += v * v;
    }
    h += std::sqrt(l2);
  }
  h = std::max(h / (double)ns, 1e-300);
  struct Key { uint64_t cls; int64_t q[3]; int cell; };
  std::vector<Key> keys((size_t)nc);
  double lo[3] = {1e300, 1e300, 1e300};
  std::vector<double> cen((size_t)nc * 3, 0.0);
  for (int64_t e = 0; e < nc; ++e)
    for (int k = 0; k < d; ++k) {
      double sacc = 0;
      for (int v = 0; v <= d; ++v) sacc += x[3 * (size_t)cn[e * (d + 1) + v] + k];
      cen[3 * e + k] = sacc / (d + 1);
      lo[k] = std::min(lo[k], cen[3 * e + k]);
    }
  for (int64_t e = 0; e < nc; ++e) {
    uint64_t hsh = 1469598103934665603ull;  // FNV-1a over the rounded edge vectors (1/64 of the reference length)
    for (int v = 1; v <= d; ++v)
      for (int k = 0; k < d; ++k) {
        const double ev = x[3 * (size_t)cn[e * (d + 1) + v] + k] - x[3 * (size_t)cn[e * (d + 1)] + k];
        const int64_t r = (int64_t)std::llround(ev / h * 64.0);
        hsh = (hsh ^ (uint64_t)r) * 1099511628211ull;
      }
    Key& kk = keys[e];
    kk.cls = hsh;
    kk.cell = (int)e;
    for (int k = 0; k < 3; ++k) kk.q[k] = k < d ? (int64_t)std::floor((cen[3 * e + k] - lo[k]) / h * 8.0) : 0;  // h/8 bins
  }
  const int zk = d - 1;
  const int64_t slab = 8;  // bins per slab: one reference length
  std::sort(keys.begin(), keys.end(), [&](const Key& a, const Key& b) {
    const int64_t sa = a.q[zk] / slab, sb = b.q[zk] / slab;
    if (sa != sb) return sa < sb;
    if (a.cls != b.cls) return a.cls < b.cls;
    for (int k = d - 1; k >= 0; --k)
      if (a.q[k] != b.q[k]) return a.q[k] < b.q[k];
    return a.cell < b.cell;
  });
  std::vector<int> order((size_t)nc);
  for (int64_t e = 0; e < nc; ++e) order[e] = keys[e].cell;
  P.cell_order.alloc(nc);
  B2_CUDA(cudaMemcpyAsync(P.cell_order.p, order.data(), sizeof(int) * (size_t)nc, cudaMemcpyHostToDevice, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<uint64_t> cls((size_t)nc);
  for (int64_t e = 0; e < nc; ++e) cls[e] = keys[e].cls;
  std::sort(cls.begin(), cls.end());
  P.n_classes = (int64_t)(std::unique(cls.begin(), cls.end()) - cls.begin());
  P.ready = true;
}

// mode & 1: matrix A (as assembled, Dirichlet rows -> identity) + dinv;  mode & 2: b_first = R u1 + b0 (+ p_surf)
void first_cells(b2_ctx* c, int mode, double dt, double nu, const double* u1, const double* uab, const double* b0,
                 const double* psurf, double* A, double* bfirst, double* dinv) {
  const int K = c->gdim;
  const Space& V = c->sp[B2_SPACE_V];
  const CSR& vv = c->pat[B2_PAT_VV];
  const int ld = (int)V.n_local();
  B2_REQUIRE(c->pos8.p != nullptr, "assemble_first needs the scatter table (rows shorter than 256 entries)");
  const int scale = (int)(c->ksp[B2_SOLVER_TENTATIVE].pc == 0);
  if (mode & 1) B2_CUDA(cudaMemsetAsync(A, 0, sizeof(double) * (size_t)vv.slots, c->stream));  // :435
  if (mode & 2) B2_LAUNCH(c, k_first_init, pgrid(c, (int64_t)ld * K), 256, (int64_t)ld * K, b0, psurf, bfirst);
  const int* order = c->first.ready ? c->first.cell_order.p : nullptr;
  const int grid = blocks_for(c->n_cells, 128);
  dispatch_elem(c, [&](auto e) {
    using E = decltype(e);
    auto launch = [&](auto kern) {
      B2_LAUNCH(c, kern, grid, 128, c->n_cells, order, c->x.p, c->cell_nodes.p, V.cell_dofs.p, (int)V.n_owned, uab, u1, ld,
                vv.slice_ptr.p, c->pos8.p, c->is_bc_row_v.p, 1.0 / dt, 0.5 * nu, A, bfirst);
    };
    if (mode == 3) launch(k_first_cells<E::D, E::DEG, 3>);
    else if (mode == 1) launch(k_first_cells<E::D, E::DEG, 1>);
    else launch(k_first_cells<E::D, E::DEG, 2>);
  });
  if (mode & 1)
    B2_LAUNCH(c, k_first_finalize, blocks_for(vv.n_rows, 256), 256, vv.n_rows, vv.slice_ptr.p, vv.diag_t.p, c->is_bc_row_v.p, scale, A, dinv);
}

// ---- stages ---------------------------------------------------------------------------------
void stage_assemble_first(b2_ctx* c, double dt, double nu) {
  require_ready(c);
  const int K = c->gdim;
  const Space& V = c->sp[B2_SPACE_V];
  const CSR& vv = c->pat[B2_PAT_VV];
  const int ld = (int)V.n_local();
  double *u1 = c->vec(B2_VEC_U1), *u2 = c->vec(B2_VEC_U2), *uab = c->vec(B2_VEC_UAB);
  halo_forward(c, B2_SPACE_V, u1, K);
  halo_forward(c, B2_SPACE_V, u2, K);
  const int64_t nl = V.n_local() * K;
  B2_LAUNCH(c, k_lincomb2, pgrid(c, nl), 256, nl, 1.5, u1, -0.5, u2, uab);  // :432-434
  const double* psurf = c->vecs.count(B2_VEC_PSURF) ? c->vec(B2_VEC_PSURF) : nullptr;
  first_cells(c, 3, dt, nu, u1, uab, c->vec(B2_VEC_B0), psurf, c->A.p, c->vec(B2_VEC_BFIRST), c->dinvA.p);
  c->last_dt = dt;
  c->fresh_step = true;
}

// out_k = add_k + scale * Op_k xq for every direction k, Op = P or G (vals = c->P.p or c->G.p)
void rect_vq(b2_ctx* c, const double* vals, const double* xq, const double* add, double scale, double* out) {
  const CSR& vq = c->pat[B2_PAT_VQ];
  const int ld = (int)c->sp[B2_SPACE_V].n_local();
  const int grid = blocks_for(vq.n_rows, 256);
  if (c->gdim == 2)
    B2_LAUNCH(c, k_rect_vq_sell<2>, grid, 256, vq.n_rows, vq.slice_ptr.p, vq.scols.p, vals, (int64_t)vq.slots, xq, add, ld, scale, out);
  else
    B2_LAUNCH(c, k_rect_vq_sell<3>, grid, 256, vq.n_rows, vq.slice_ptr.p, vq.scols.p, vals, (int64_t)vq.slots, xq, add, ld, scale, out);
}

// out = scale * sum_k D_k xv_k, rows flagged in zero_row (if given) set to 0
void rect_qv(b2_ctx* c, const double* xv, double scale, const uint8_t* zero_row, double* out) {
  const CSR& qv = c->pat[B2_PAT_QV];
  const int ld = (int)c->sp[B2_SPACE_V].n_local();
  const int grid = blocks_for((int64_t)qv.n_rows * 16, 256);
  if (c->gdim == 2)
    B2_LAUNCH(c, (k_rect_qv<2, 16>), grid, 256, qv.n_rows, qv.rowptr.p, qv.cols.p, c->D.p, xv, ld, scale, zero_row, out);
  else
    B2_LAUNCH(c, (k_rect_qv<3, 16>), grid, 256, qv.n_rows, qv.rowptr.p, qv.cols.p, c->D.p, xv, ld, scale, zero_row, out);
}

// matrix-free element vectors of the low-memory strategy (elem.cuh: k_lowmem_vector)
void lowmem_vector(b2_ctx* c, int mode, const double* in, double scale, double* out) {
  const Space &V = c->sp[B2_SPACE_V], &Q = c->sp[B2_SPACE_Q];
  dispatch_elem(c, [&](auto e) {
    using E = decltype(e);
    const int grid = blocks_for(c->n_cells, 128);
    if (mode == 0)
      B2_LAUNCH(c, (k_lowmem_vector<E::D, E::DEG, 0>), grid, 128, c->n_cells, c->x.p, c->cell_nodes.p, V.cell_dofs.p, Q.cell_dofs.p,
                (int)V.n_owned, (int)Q.n_owned, (int)V.n_local(), in, scale, out);
    else if (mode == 1)
      B2_LAUNCH(c, (k_lowmem_vector<E::D, E::DEG, 1>), grid, 128, c->n_cells, c->x.p, c->cell_nodes.p, V.cell_dofs.p, Q.cell_dofs.p,
                (int)V.n_owned, (int)Q.n_owned, (int)V.n_local(), in, scale, out);
    else
      B2_LAUNCH(c, (k_lowmem_vector<E::D, E::DEG, 2>), grid, 128, c->n_cells, c->x.p, c->cell_nodes.p, V.cell_dofs.p, Q.cell_dofs.p,
                (int)V.n_owned, (int)Q.n_owned, (int)V.n_local(), in, scale, out);
  });
}

__global__ void k_zero_rows_q(int64_t n, const uint8_t* __restrict__ zero_row, double* __restrict__ v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && zero_row[i]) v[i] = 0.0;
}

void stage_tentative_assemble(b2_ctx* c) {
  require_ready(c);
  double* ps = c->vec(B2_VEC_PS);
  halo_forward(c, B2_SPACE_Q, ps, 1);
  if (c->low_memory) {  // :485-497: assemble int p* dv/dx_i directly; rhs1 = b_first + that (:505-506)
    const int64_t nl = c->sp[B2_SPACE_V].n_local() * c->gdim;
    B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_RHS1), c->vec(B2_VEC_BFIRST), sizeof(double) * nl, cudaMemcpyDeviceToDevice, c->stream));
    lowmem_vector(c, 0, ps, 1.0, c->vec(B2_VEC_RHS1));
    return;
  }
  rect_vq(c, c->P.p, ps, c->vec(B2_VEC_BFIRST), 1.0, c->vec(B2_VEC_RHS1));
}

void apply_velocity_bcs(b2_ctx* c, double* v) {
  for (int k = 0; k < c->gdim; ++k)
    if (c->bc_dofs[k].n) {
      B2_REQUIRE(c->bc_vals[k].n == c->bc_dofs[k].n, "velocity BC values not set");
      const double* vals = c->bc_vals[k].p;
      if (c->bc_step >= 0) {
        B2_REQUIRE(c->bc_step < c->bc_series_steps[k], "b2_select_bc_step beyond the prefetched series");
        vals = c->bc_series[k].p + (size_t)c->bc_step * c->bc_dofs[k].n;
      }
      B2_LAUNCH(c, k_set_bc, blocks_for(c->bc_dofs[k].n, 256), 256, c->bc_dofs[k].n, c->bc_dofs[k].p, vals,
                v + (size_t)k * c->sp[B2_SPACE_V].n_local());
    }
}

template <int K>
void sqdiff(b2_ctx* c, int64_t n, int ld, const double* a, const double* b, double* out_dev) {
  B2_LAUNCH(c, k_sqdiff<K>, pgrid(c, n), 256, n, ld, a, b, out_dev, c->partials.p, c->d_counter);
  allreduce_sum(c, out_dev, K);
}

void read_sums(b2_ctx* c, int n) {
  B2_CUDA(cudaMemcpyAsync(c->h_sums, c->d_sums, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  c->stats.bytes_d2h += sizeof(double) * n;
}

// out = (add) + time extrapolation of a solution history (h[0] newest): h0 | 2 h0 - h1 | 3 h0 - 3 h1 + h2
void hist_extrapolate(b2_ctx* c, DBuf<double>* h, int n_avail, int64_t n, const double* add, double* out) {
  const int g = pgrid(c, n);
  if (n_avail >= 3) B2_LAUNCH(c, k_lincomb4, g, 256, n, 3.0, h[0].p, -3.0, h[1].p, 1.0, h[2].p, add, out);
  else if (n_avail == 2) B2_LAUNCH(c, k_lincomb4, g, 256, n, 2.0, h[0].p, -1.0, h[1].p, 0.0, h[0].p, add, out);
  else B2_LAUNCH(c, k_lincomb4, g, 256, n, 1.0, h[0].p, 0.0, h[0].p, 0.0, h[0].p, add, out);
}

// newest <- v: rotate the three buffers, copy into slot 0
void hist_push(b2_ctx* c, DBuf<double>* h, int& n_avail, int64_t n, const double* v, bool replace_newest) {
  if (!replace_newest || n_avail == 0) {
    std::swap(h[2], h[1]);
    std::swap(h[1], h[0]);  // (h0, h1, h2) <- (old h2 = free slot, old h0, old h1)
    n_avail = std::min(n_avail + 1, 3);
  }
  if (h[0].p == nullptr) h[0].alloc(n);
  B2_CUDA(cudaMemcpyAsync(h[0].p, v, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
}

// defer_diff: leave the squared differences in pinned memory (h_sums[8..8+K), valid after the next stream
// synchronisation) instead of draining the pipeline for a number only the caller of the whole step needs
void stage_tentative_solve(b2_ctx* c, double* diff, int32_t* reasons, bool defer_diff = false) {
  require_ready(c);
  const int K = c->gdim;
  const Space& V = c->sp[B2_SPACE_V];
  double *rhs1 = c->vec(B2_VEC_RHS1), *u = c->vec(B2_VEC_U), *wrk = c->vec(B2_VEC_WRK);
  apply_velocity_bcs(c, rhs1);                                                                  // :517-518
  B2_CUDA(cudaMemcpyAsync(wrk, u, sizeof(double) * V.n_local() * K, cudaMemcpyDeviceToDevice, c->stream));  // :520
  int32_t its[B2_MAXK] = {0, 0, 0};
  const KSPOpts& ot = c->ksp[B2_SOLVER_TENTATIVE];
  const bool hist2 = ot.extrapolate_guess && ot.guess_order == 2;
  const bool new_entry = c->fresh_step;
  c->fresh_step = false;
  if (hist2) {
    // quadratic extrapolation of the tentative velocities of the last three steps (the sequence u* is smooth in
    // time even where u^n - u* is not); a repeated pass of the same step starts from the pass before (u)
    if (new_entry && c->n_ustar_hist >= 1) hist_extrapolate(c, c->ustar_hist, c->n_ustar_hist, V.n_local() * K, nullptr, u);
  } else if (ot.extrapolate_guess && c->steps_done >= 1) {
    // initial guess 2 u^n - u^{n-1} - (u - u*)^n, i.e. the extrapolated velocity minus the last pressure
    // correction (the tentative velocity lacks it): the converged solution does not depend on the guess, the
    // iteration count does
    const int64_t nl = V.n_local() * K;
    B2_LAUNCH(c, k_lincomb2, pgrid(c, nl), 256, nl, 2.0, c->vec(B2_VEC_U1), -1.0, c->vec(B2_VEC_U2), u);
    if (c->delta_prev.p != nullptr) B2_LAUNCH(c, k_lincomb2, pgrid(c, nl), 256, nl, 1.0, u, -1.0, c->delta_prev.p, u);
  }
  krylov_solve(c, B2_SOLVER_TENTATIVE, c->pat[B2_PAT_VV], c->A.p, c->dinvA.p, B2_SPACE_V, K, rhs1, u, reasons, its);  // :521
  for (int k = 0; k < K; ++k) c->stats.its_tentative[k] = its[k];
  if (hist2) hist_push(c, c->ustar_hist, c->n_ustar_hist, V.n_local() * K, u, !new_entry);
  double* dsq = c->d_sums + (defer_diff ? 8 : 0);
  if (K == 2) sqdiff<2>(c, V.n_owned, (int)V.n_local(), wrk, u, dsq);
  else sqdiff<3>(c, V.n_owned, (int)V.n_local(), wrk, u, dsq);
  if (defer_diff) {
    B2_CUDA(cudaMemcpyAsync(c->h_sums + 8, dsq, sizeof(double) * K, cudaMemcpyDeviceToHost, c->stream));
    c->stats.bytes_d2h += sizeof(double) * K;
    return;
  }
  read_sums(c, K);
  double d = 0.0;
  for (int k = 0; k < K; ++k) d += std::sqrt(c->h_sums[k]);  // :523-524 (sum of per-component 2-norms)
  *diff = d;
}

void stage_pressure_assemble(b2_ctx* c, double dt) {
  require_ready(c);
  double* u = c->vec(B2_VEC_U);
  halo_forward(c, B2_SPACE_V, u, c->gdim);
  const uint8_t* zr = c->has_pbc ? c->is_bc_q.p : nullptr;
  if (c->low_memory) {  // :537-538: b2 = -(1/dt) int div(u) q, Dirichlet rows zeroed (:549-550)
    const Space& Q = c->sp[B2_SPACE_Q];
    B2_CUDA(cudaMemsetAsync(c->vec(B2_VEC_B2), 0, sizeof(double) * Q.n_local(), c->stream));
    lowmem_vector(c, 2, u, -1.0 / dt, c->vec(B2_VEC_B2));
    if (zr) B2_LAUNCH(c, k_zero_rows_q, blocks_for(Q.n_owned, 256), 256, Q.n_owned, zr, c->vec(B2_VEC_B2));
    return;
  }
  rect_qv(c, u, -1.0 / dt, zr, c->vec(B2_VEC_B2));
}

void stage_pressure_solve(b2_ctx* c, double nu, int32_t* reason) {
  require_ready(c);
  const Space& Q = c->sp[B2_SPACE_Q];
  double *b2 = c->vec(B2_VEC_B2), *dp = c->vec(B2_VEC_DP), *p = c->vec(B2_VEC_P), *ps = c->vec(B2_VEC_PS);
  const int64_t n = Q.n_owned;
  if (!c->has_pbc) {  // MatNullSpaceRemove: subtract the arithmetic mean of the entries (:573-574)
    B2_LAUNCH(c, k_sums, pgrid(c, n), 256, n, b2, (const double*)nullptr, c->d_sums, c->partials.p, c->d_counter);
    allreduce_sum(c, c->d_sums, 2);
    B2_LAUNCH(c, k_shift, pgrid(c, n), 256, n, b2, c->d_sums, 0, 1.0 / (double)Q.n_global, (const double*)nullptr, (double*)nullptr);
  }
  int32_t its = 0;
  if (c->ksp[B2_SOLVER_PRESSURE].extrapolate_guess) {  // start from 2 dp^{n-1} - dp^{n-2}
    const int64_t nq = Q.n_local();
    if (c->dp_old.p == nullptr) { c->dp_old.alloc(nq); c->dp_old.zero(c->stream); }
    double* t3 = c->wq[3].p;
    if (c->dp_hist >= 2) B2_LAUNCH(c, k_lincomb2, pgrid(c, nq), 256, nq, 2.0, dp, -1.0, c->dp_old.p, t3);
    B2_CUDA(cudaMemcpyAsync(c->dp_old.p, dp, sizeof(double) * nq, cudaMemcpyDeviceToDevice, c->stream));
    if (c->dp_hist >= 2) B2_CUDA(cudaMemcpyAsync(dp, t3, sizeof(double) * nq, cudaMemcpyDeviceToDevice, c->stream));
    c->dp_hist++;
  }
  if (c->ksp[B2_SOLVER_PRESSURE].pc == 2 && !c->mg.empty() && !c->has_pbc)
    pcg_mg_solve(c, b2, dp, reason, &its);
  else
    krylov_solve(c, B2_SOLVER_PRESSURE, c->pat[B2_PAT_QQ], c->Ap.p, c->dinvAp.p, B2_SPACE_Q, 1, b2, dp, reason, &its);  // :578
  c->stats.its_pressure = its;
  if (!c->has_pbc) {  // dp -= int dp / int 1  (:579-591), then ps = p + dp (:604)
    B2_LAUNCH(c, k_sums, pgrid(c, n), 256, n, dp, c->vec(B2_VEC_MQ), c->d_sums, c->partials.p, c->d_counter);
    allreduce_sum(c, c->d_sums, 2);
    B2_LAUNCH(c, k_shift, pgrid(c, n), 256, n, dp, c->d_sums, 1, 1.0 / c->vol, c->rotational ? nullptr : p,
              c->rotational ? nullptr : ps);
  } else if (!c->rotational) {
    B2_LAUNCH(c, k_lincomb2, pgrid(c, n), 256, n, 1.0, p, 1.0, dp, ps);
  }
  if (c->rotational) {
    // ps = Proj_Q(p + dp - xi nu div u): MQ ps = MQ (p + dp) - 0.5 nu sum_i D_i u_i   (:238-247,593-602)
    const CSR& qq = c->pat[B2_PAT_QQ];
    double *t0 = c->wq[3].p, *rhs = c->vec(B2_VEC_B2);
    B2_LAUNCH(c, k_lincomb2, pgrid(c, n), 256, n, 1.0, p, 1.0, dp, t0);
    halo_forward(c, B2_SPACE_Q, t0, 1);
    double* u = c->vec(B2_VEC_U);
    // rhs <- -0.5 nu sum_i D_i u_i (reusing b2 as scratch: it is rebuilt by the next pressure_assemble)
    if (c->low_memory) {
      B2_CUDA(cudaMemsetAsync(rhs, 0, sizeof(double) * Q.n_local(), c->stream));
      lowmem_vector(c, 2, u, -0.5 * nu, rhs);
    } else {
      rect_qv(c, u, -0.5 * nu, nullptr, rhs);
    }
    double* mq = c->wq[2].p;  // q work vector is free between solves
    spmm(c, qq, c->MQ.p, 1, t0, mq);
    B2_LAUNCH(c, k_lincomb2, pgrid(c, n), 256, n, 1.0, mq, 1.0, rhs, rhs);
    int32_t r2 = 0, its2 = 0;
    // wq[3] (t0) doubles as the solution buffer start; solve into ps directly
    krylov_solve(c, B2_SOLVER_PROJECTOR, qq, c->MQ.p, c->dinvMQ.p, B2_SPACE_Q, 1, rhs, ps, &r2, &its2);
    c->stats.its_projector = its2;
    B2_REQUIRE(r2 > 0, "rotational pressure projection did not converge");  // :601
  }
}

void stage_velocity_update(b2_ctx* c, double dt, int32_t* reasons) {
  require_ready(c);
  const int K = c->gdim;
  double *u = c->vec(B2_VEC_U), *b3 = c->vec(B2_VEC_B3), *dp = c->vec(B2_VEC_DP);
  spmm(c, c->pat[B2_PAT_VV], c->M.p, K, u, b3, nullptr, nullptr, FIN_NONE, 0, B2_SPACE_V);  // :638
  halo_forward(c, B2_SPACE_Q, dp, 1);
  if (c->low_memory) lowmem_vector(c, 1, dp, -dt, b3);  // :617-622: b3 -= dt int d(dp)/dx_i v
  else rect_vq(c, c->G.p, dp, b3, -dt, b3);  // :642-645
  int32_t its[B2_MAXK] = {0, 0, 0};
  const bool extrap = c->ksp[B2_SOLVER_SCALAR].extrapolate_guess;
  const int64_t nl = c->sp[B2_SPACE_V].n_local() * K;
  double* ustar = c->vec(B2_VEC_WRK);  // free after the tentative solve's diff
  const bool hist2m = extrap && c->ksp[B2_SOLVER_SCALAR].guess_order == 2;
  if (extrap) {
    if (c->delta_prev.p == nullptr) { c->delta_prev.alloc(nl); c->delta_prev.zero(c->stream); }
    B2_CUDA(cudaMemcpyAsync(ustar, u, sizeof(double) * nl, cudaMemcpyDeviceToDevice, c->stream));
    if (hist2m && c->n_delta_hist >= 1) hist_extrapolate(c, c->delta_hist, c->n_delta_hist, nl, ustar, u);  // u* + extrapolated correction
    else B2_LAUNCH(c, k_lincomb2, pgrid(c, nl), 256, nl, 1.0, u, 1.0, c->delta_prev.p, u);  // guess u* + (u - u*)_previous step
  }
  krylov_solve(c, B2_SOLVER_SCALAR, c->pat[B2_PAT_VV], c->M.p, c->dinvM.p, B2_SPACE_V, K, b3, u, reasons, its);  // :656
  if (extrap) B2_LAUNCH(c, k_lincomb2, pgrid(c, nl), 256, nl, 1.0, u, -1.0, ustar, c->delta_prev.p);
  if (hist2m) hist_push(c, c->delta_hist, c->n_delta_hist, nl, c->delta_prev.p, false);
  for (int k = 0; k < K; ++k) c->stats.its_update[k] = its[k];
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  return ms;
}

// first half of a step: everything that does not need this step's Dirichlet values.  Only enqueues work,
// so the host can evaluate time-dependent boundary callables while the GPU assembles.
void stage_step_begin(b2_ctx* c, double dt, double nu) {
  require_ready(c);
  const Space& Q = c->sp[B2_SPACE_Q];
  B2_CUDA(cudaEventRecord(c->ev[0], c->stream));
  B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_PS), c->vec(B2_VEC_P), sizeof(double) * Q.n_local(), cudaMemcpyDeviceToDevice, c->stream));  // :673
  stage_assemble_first(c, dt, nu);
  B2_CUDA(cudaEventRecord(c->ev[1], c->stream));
  c->step_begun = true;
}

void stage_step(b2_ctx* c, double dt, double nu, double max_error, int max_iter, double* diff_out) {
  require_ready(c);
  const int K = c->gdim;
  const Space &V = c->sp[B2_SPACE_V], &Q = c->sp[B2_SPACE_Q];
  if (!c->step_begun) stage_step_begin(c, dt, nu);
  c->step_begun = false;
  int inner = 0;
  double diff = 1e8;
  float ms_t = 0, ms_p = 0;
  bool pending = false;  // the last pass leaves its diff and stage times to be collected after the step's final sync
  while (inner < max_iter && diff > max_error) {  // :677-684
    ++inner;
    const bool last_pass = inner >= max_iter;  // diff cannot start another pass: no need to wait for it here
    int32_t reasons[B2_MAXK] = {0, 0, 0}, rp = 0;
    B2_CUDA(cudaEventRecord(c->ev[2], c->stream));
    stage_tentative_assemble(c);
    stage_tentative_solve(c, &diff, reasons, last_pass);
    for (int k = 0; k < K; ++k)
      if (reasons[k] <= 0) throw B2Error(-20, "tentative velocity solve diverged, component " + std::to_string(k) + " reason " + std::to_string(reasons[k]));
    B2_CUDA(cudaEventRecord(c->ev[3], c->stream));
    stage_pressure_assemble(c, dt);
    stage_pressure_solve(c, nu, &rp);
    if (rp <= 0) throw B2Error(-21, "pressure solve diverged, reason " + std::to_string(rp));
    B2_CUDA(cudaEventRecord(c->ev[4], c->stream));
    if (last_pass) { pending = true; break; }
    B2_CUDA(cudaEventSynchronize(c->ev[4]));
    ms_t += ev_ms(c->ev[2], c->ev[3]);
    ms_p += ev_ms(c->ev[3], c->ev[4]);
  }
  int32_t ru[B2_MAXK] = {0, 0, 0};
  stage_velocity_update(c, dt, ru);
  // u2 <- u1 ; u1 <- u ; p <- ps   (:689-693): swap the two history buffers, one copy each
  std::swap(c->vecs[B2_VEC_U1].buf, c->vecs[B2_VEC_U2].buf);
  B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_U1), c->vec(B2_VEC_U), sizeof(double) * V.n_local() * K, cudaMemcpyDeviceToDevice, c->stream));
  B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_P), c->vec(B2_VEC_PS), sizeof(double) * Q.n_local(), cudaMemcpyDeviceToDevice, c->stream));
  if (c->peer_on)
    B2_CUDA(cudaMemcpyAsync(c->h_peer_err, c->h_peer.err, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaEventRecord(c->ev[5], c->stream));
  B2_CUDA(cudaEventSynchronize(c->ev[5]));
  if (c->peer_on && *c->h_peer_err != 0)
    throw B2Error(-32, "peer-memory collective timed out: a rank of the job stopped taking part");
  if (pending) {
    ms_t += ev_ms(c->ev[2], c->ev[3]);
    ms_p += ev_ms(c->ev[3], c->ev[4]);
    diff = 0.0;
    for (int k = 0; k < K; ++k) diff += std::sqrt(c->h_sums[8 + k]);  // :523-524
  }
  c->stats.ms_assemble_first = ev_ms(c->ev[0], c->ev[1]);
  c->stats.ms_tentative = ms_t;
  c->stats.ms_pressure = ms_p;
  c->stats.ms_update = ev_ms(c->ev[4], c->ev[5]);
  c->stats.ms_step = ev_ms(c->ev[0], c->ev[5]);
  c->steps_done++;
  *diff_out = diff;
}

// ---- preassembly ----------------------------------------------------------------------------------
void do_preassemble(b2_ctx* c, const double* body_force, int low_memory, int rotational) {
  B2_REQUIRE(c->patterns_built, "b2_build_patterns has not been called");
  c->cfg_version++;  // every buffer a captured graph refers to is (re)allocated below
  c->low_memory = low_memory != 0;
  c->rotational = rotational != 0;
  const int K = c->gdim;
  const Space &V = c->sp[B2_SPACE_V], &Q = c->sp[B2_SPACE_Q];
  const CSR &vv = c->pat[B2_PAT_VV], &vq = c->pat[B2_PAT_VQ], &qv = c->pat[B2_PAT_QV], &qq = c->pat[B2_PAT_QQ];
  // vectors
  for (int id : {B2_VEC_U, B2_VEC_U1, B2_VEC_U2, B2_VEC_UAB, B2_VEC_RHS1, B2_VEC_BFIRST, B2_VEC_B0, B2_VEC_B3, B2_VEC_WRK})
    alloc_vec(c, id, B2_SPACE_V, K);
  for (int id : {B2_VEC_PS, B2_VEC_P, B2_VEC_DP, B2_VEC_B2, B2_VEC_MQ}) alloc_vec(c, id, B2_SPACE_Q, 1);
  for (auto& w : c->wv) { w.alloc(V.n_local() * K); w.zero(c->stream); }
  for (auto& w : c->wq) { w.alloc(Q.n_local()); w.zero(c->stream); }
  c->stage.alloc(std::max<int64_t>(std::max<int64_t>(V.n_local() * K, vv.nnz), 1));
  // matrices
  c->M.alloc(vv.slots); c->M.zero(c->stream);
  c->Kst.alloc(vv.slots); c->Kst.zero(c->stream);
  c->A.alloc(vv.slots); c->A.zero(c->stream);
  c->Ap.alloc(qq.slots); c->Ap.zero(c->stream);
  if (!c->low_memory) {  // the 3d rectangular operator families exist only in the matrix-vector strategy (:392-404)
    c->P.alloc(vq.slots * K); c->P.zero(c->stream);
    c->G.alloc(vq.slots * K); c->G.zero(c->stream);
    c->D.alloc(qv.nnz * K); c->D.zero(c->stream);
  }
  if (c->rotational) { c->MQ.alloc(qq.slots); c->MQ.zero(c->stream); }
  c->dinvA.alloc(V.n_local()); c->dinvM.alloc(V.n_local()); c->dinvAp.alloc(Q.n_local());
  c->onesV.alloc(V.n_local()); c->onesQ.alloc(Q.n_local());
  B2_LAUNCH(c, k_fill, pgrid(c, V.n_local()), 256, V.n_local(), 1.0, c->onesV.p);
  B2_LAUNCH(c, k_fill, pgrid(c, Q.n_local()), 256, Q.n_local(), 1.0, c->onesQ.p);
  B2_LAUNCH(c, k_fill, pgrid(c, V.n_local()), 256, V.n_local(), 1.0, c->dinvA.p);
  double f[3] = {0, 0, 0};
  if (body_force)
    for (int k = 0; k < K; ++k) f[k] = body_force[k];
  dispatch_elem(c, [&](auto e) {
    using E = decltype(e);
    constexpr int D = E::D, DEG = E::DEG;
    const int64_t nc = c->n_cells;
    B2_LAUNCH(c, (k_assemble_square<D, DEG, B2_FORM_MASS_V>), blocks_for(nc * E::NV, 128), 128, nc, c->x.p, c->cell_nodes.p,
              V.cell_dofs.p, vv.n_rows, vv.rowptr.p, vv.cols.p, vv.slice_ptr.p, c->M.p);                       // :373
    B2_LAUNCH(c, (k_assemble_square<D, DEG, B2_FORM_STIFF_V>), blocks_for(nc * E::NV, 128), 128, nc, c->x.p, c->cell_nodes.p,
              V.cell_dofs.p, vv.n_rows, vv.rowptr.p, vv.cols.p, vv.slice_ptr.p, c->Kst.p);                     // :375
    // :379 -- in a fixed order: the algebraic multigrid (b2_pressure_amg_build) is built from Ap, and the same mesh must give
    // the same hierarchy on every run
    assemble_in_fixed_order(c, nc * E::NQ * E::NQ, qq.slots, c->Ap.p, [&](unsigned* slot, double* val) {
      B2_LAUNCH(c, (k_assemble_square<D, DEG, B2_FORM_STIFF_Q>), blocks_for(nc * E::NQ, 128), 128, nc, c->x.p, c->cell_nodes.p,
                Q.cell_dofs.p, qq.n_rows, qq.rowptr.p, qq.cols.p, qq.slice_ptr.p, c->Ap.p, slot, val);
    });
    if (c->rotational)
      B2_LAUNCH(c, (k_assemble_square<D, DEG, B2_FORM_MASS_Q>), blocks_for(nc * E::NQ, 128), 128, nc, c->x.p, c->cell_nodes.p,
                Q.cell_dofs.p, qq.n_rows, qq.rowptr.p, qq.cols.p, qq.slice_ptr.p, c->MQ.p);                    // function.py:63-71
    if (!c->low_memory) {
      B2_LAUNCH(c, (k_assemble_PG<D, DEG>), blocks_for(nc * E::NV, 128), 128, nc, c->x.p, c->cell_nodes.p, V.cell_dofs.p,
                Q.cell_dofs.p, vq.n_rows, vq.rowptr.p, vq.cols.p, vq.slice_ptr.p, (int64_t)vq.slots, c->P.p, c->G.p);  // :395,399
      B2_LAUNCH(c, (k_assemble_D<D, DEG>), blocks_for(nc * E::NQ, 128), 128, nc, c->x.p, c->cell_nodes.p, V.cell_dofs.p,
                Q.cell_dofs.p, qv.n_rows, qv.rowptr.p, qv.cols.p, c->D.p);                      // :403
    }
    B2_LAUNCH(c, (k_assemble_loads<D, DEG>), blocks_for(nc, 128), 128, nc, c->x.p, c->cell_nodes.p, V.cell_dofs.p, Q.cell_dofs.p,
              (int)V.n_owned, (int)Q.n_owned, (int)V.n_local(), f[0], f[1], f[2], c->vec(B2_VEC_B0), c->vec(B2_VEC_MQ));  // :387-390
  });
  // scatter table for the per-step convection assembly (needs rows shorter than 256 entries)
  {
    std::vector<int> sp((size_t)(vv.n_rows + 31) / 32 + 1);
    B2_CUDA(cudaMemcpyAsync(sp.data(), vv.slice_ptr.p, sizeof(int) * sp.size(), cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    int maxlen = 0;
    for (size_t i = 0; i + 1 < sp.size(); ++i) maxlen = std::max(maxlen, (sp[i + 1] - sp[i]) / 32);
    c->maxlen_vv = maxlen;
    if (maxlen < 256) {
      dispatch_elem(c, [&](auto e) {
        using E = decltype(e);
        constexpr int NVP = (E::NV + 3) / 4 * 4;
        c->pos8.alloc(c->n_cells * E::NV * NVP);
        B2_LAUNCH(c, (k_build_pos8<E::NV>), blocks_for(c->n_cells * E::NV, 128), 128, c->n_cells, V.cell_dofs.p, (int)V.n_owned,
                  vv.rowptr.p, vv.cols.p, c->pos8.p);
      });
    }
  }
  build_first_plan(c);
  // Dirichlet masks
  c->is_bc_row_v.alloc(V.n_local()); c->is_bc_row_v.zero(c->stream);
  c->is_bc_q.alloc(Q.n_local()); c->is_bc_q.zero(c->stream);
  if (c->bc_dofs[0].n)  // the shared matrix takes component 0's dof set (:470-472)
    B2_LAUNCH(c, k_mark, blocks_for(c->bc_dofs[0].n, 256), 256, c->bc_dofs[0].n, c->bc_dofs[0].p, c->is_bc_row_v.p);
  if (c->has_pbc) {
    B2_LAUNCH(c, k_mark, blocks_for(c->pbc_dofs.n, 256), 256, c->pbc_dofs.n, c->pbc_dofs.p, c->is_bc_q.p);
    B2_LAUNCH(c, k_apply_bc_rows_cols, blocks_for(qq.n_rows, 256), 256, qq.n_rows, qq.slice_ptr.p, qq.scols.p, qq.diag_t.p, c->is_bc_q.p, c->Ap.p);
  }
  B2_LAUNCH(c, k_inv_diag, blocks_for(vv.n_rows, 256), 256, vv.n_rows, vv.slice_ptr.p, vv.diag_t.p, c->M.p, c->dinvM.p);
  B2_LAUNCH(c, k_inv_diag, blocks_for(qq.n_rows, 256), 256, qq.n_rows, qq.slice_ptr.p, qq.diag_t.p, c->Ap.p, c->dinvAp.p);
  if (c->rotational) {
    c->dinvMQ.alloc(Q.n_local());
    B2_LAUNCH(c, k_inv_diag, blocks_for(qq.n_rows, 256), 256, qq.n_rows, qq.slice_ptr.p, qq.diag_t.p, c->MQ.p, c->dinvMQ.p);
  }
  // measure of the domain = sum mQ  (:581-584)
  B2_LAUNCH(c, k_sums, pgrid(c, Q.n_owned), 256, Q.n_owned, c->vec(B2_VEC_MQ), (const double*)nullptr, c->d_sums, c->partials.p, c->d_counter);
  allreduce_sum(c, c->d_sums, 2);
  read_sums(c, 1);
  c->vol = c->h_sums[0];
  if (Q.n_global == 0) c->sp[B2_SPACE_Q].n_global = Q.n_owned;
  if (V.n_global == 0) c->sp[B2_SPACE_V].n_global = V.n_owned;
  c->preassembled = true;
}

// how a matrix' values are stored (linalg.cuh, "storage")
enum class Layout {
  Sell,           // square operators: one value per SELL slot of the pattern
  SellByComp,     // P, G: SELL slots, direction k at vals + k * slots
  CsrInterleaved  // D: CSR positions, the gdim directions of a nonzero side by side ([nnz][gdim])
};

const DBuf<double>* matrix_values(b2_ctx* c, int mat, const CSR** pat, Layout* layout) {
  *layout = Layout::Sell;
  switch (mat) {
    case B2_MAT_M: *pat = &c->pat[B2_PAT_VV]; return &c->M;
    case B2_MAT_K: *pat = &c->pat[B2_PAT_VV]; return &c->Kst;
    case B2_MAT_A: *pat = &c->pat[B2_PAT_VV]; return &c->A;
    case B2_MAT_AP: *pat = &c->pat[B2_PAT_QQ]; return &c->Ap;
    case B2_MAT_MQ: *pat = &c->pat[B2_PAT_QQ]; return &c->MQ;
    case B2_MAT_P: *pat = &c->pat[B2_PAT_VQ]; *layout = Layout::SellByComp; return &c->P;
    case B2_MAT_G: *pat = &c->pat[B2_PAT_VQ]; *layout = Layout::SellByComp; return &c->G;
    case B2_MAT_D: *pat = &c->pat[B2_PAT_QV]; *layout = Layout::CsrInterleaved; return &c->D;
    default: throw B2Error(-2, "unknown matrix id");
  }
}

template <typename F>
int guarded(b2_ctx* c, F&& f) {
  try {
    if (c) B2_CUDA(cudaSetDevice(c->device));
    f();
    return 0;
  } catch (const B2Error& e) {
    (c ? c->err : g_last_error) = e.what();
    g_last_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    (c ? c->err : g_last_error) = e.what();
    g_last_error = e.what();
    return -99;
  }
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int b2_abi_version(void) { return B2_ABI_VERSION; }

int b2_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int b2_nccl_unique_id(void* uid) {
  return guarded(nullptr, [&] {
    g_nccl.load();
    static_assert(sizeof(ncclUniqueId) == B2_NCCL_UID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    B2_NCCL(g_nccl.GetUniqueId(&id));
    std::memcpy(uid, &id, sizeof(id));
  });
}

int b2_create(b2_ctx** out, int device, int nranks, int rank, const void* nccl_uid) {
  *out = nullptr;
  b2_ctx* c = nullptr;
  int rc = guarded(nullptr, [&] {
    int ndev = 0;
    B2_CUDA(cudaGetDeviceCount(&ndev));
    B2_REQUIRE(ndev > 0, "no CUDA device visible: libb200ipcs has no CPU fallback");
    B2_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    B2_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank / nranks");
    B2_REQUIRE(nranks == 1 || nccl_uid != nullptr, "multi-rank contexts need the NCCL unique id of rank 0");
    B2_CUDA(cudaSetDevice(device));
    c = new b2_ctx();
    c->device = device;
    c->nranks = nranks;
    c->rank = rank;
    cudaDeviceProp prop;
    B2_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sm = prop.multiProcessorCount;
    B2_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    B2_CUDA(cudaMalloc(&c->d_st, sizeof(KryState)));
    B2_CUDA(cudaMallocHost(&c->h_st, sizeof(KryState)));
    B2_CUDA(cudaMalloc(&c->d_sums, sizeof(double) * 16));
    B2_CUDA(cudaMallocHost(&c->h_sums, sizeof(double) * 16));
    c->partials.alloc((int64_t)c->sm * 32 * 16);
    B2_CUDA(cudaMalloc(&c->d_counter, sizeof(unsigned)));
    B2_CUDA(cudaMemsetAsync(c->d_counter, 0, sizeof(unsigned), c->stream));
    for (auto& e : c->ev) B2_CUDA(cudaEventCreate(&e));
    for (auto& e : c->user_ev) B2_CUDA(cudaEventCreate(&e));
    c->ksp[B2_SOLVER_TENTATIVE].type = 1;
    if (const char* e = std::getenv("B200_PEER")) c->use_peer = std::atoi(e);  // 0: keep every collective on NCCL
    B2_CUDA(cudaMalloc(&c->d_red, sizeof(double) * 16));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    if (nranks > 1) {
      g_nccl.load();
      ncclUniqueId id;
      std::memcpy(&id, nccl_uid, sizeof(id));
      B2_NCCL(g_nccl.CommInitRank(&c->comm, nranks, id, rank));
    }
  });
  if (rc != 0) { delete c; return rc; }
  *out = c;
  return 0;
}

void b2_destroy(b2_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  cudaFree(c->d_st);
  cudaFreeHost(c->h_st);
  cudaFree(c->d_sums);
  cudaFreeHost(c->h_sums);
  cudaFree(c->d_counter);
  cudaFree(c->d_red);
  cudaFree(c->d_gm);
  if (c->pcg_graph) cudaGraphExecDestroy(c->pcg_graph);
  for (auto& sg : c->seg) {
    for (int q = 0; q < B2_MAXR; ++q)
      if (sg.peer[q] && sg.peer[q] != sg.base) cudaIpcCloseMemHandle(sg.peer[q]);
    if (sg.base) cudaFree(sg.base);
  }
  cudaFree(c->d_peer);
  cudaFree(c->d_counter_peer);
  if (c->h_peer_err) cudaFreeHost(c->h_peer_err);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  for (auto& e : c->ev) cudaEventDestroy(e);
  for (auto& e : c->user_ev) cudaEventDestroy(e);
  cudaStreamDestroy(c->stream);
  delete c;
}

const char* b2_last_error(const b2_ctx* c) { return c ? c->err.c_str() : g_last_error.c_str(); }

void* b2_host_alloc(int64_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) return nullptr;
  return p;
}
void b2_host_free(void* p) { if (p) cudaFreeHost(p); }

int b2_set_mesh(b2_ctx* c, int gdim, int64_t n_nodes, const double* x, int64_t n_cells, const int32_t* cell_nodes) {
  return guarded(c, [&] {
    B2_REQUIRE(gdim == 2 || gdim == 3, "gdim must be 2 or 3");
    c->gdim = gdim;
    c->n_nodes = n_nodes;
    c->n_cells = n_cells;
    c->x.alloc(n_nodes * 3);
    c->cell_nodes.alloc(n_cells * (gdim + 1));
    B2_CUDA(cudaMemcpyAsync(c->x.p, x, sizeof(double) * n_nodes * 3, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(c->cell_nodes.p, cell_nodes, sizeof(int) * n_cells * (gdim + 1), cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(double) * n_nodes * 3 + sizeof(int) * n_cells * (gdim + 1);
  });
}

int b2_set_space(b2_ctx* c, int space, int degree, int64_t n_owned, int64_t n_ghost, const int32_t* cell_dofs) {
  return guarded(c, [&] {
    B2_REQUIRE(c->gdim != 0, "b2_set_mesh must come first");
    B2_REQUIRE(space == B2_SPACE_V || space == B2_SPACE_Q, "bad space id");
    B2_REQUIRE(degree == 1 || degree == 2, "Lagrange degree must be 1 or 2");
    B2_REQUIRE(space == B2_SPACE_V || degree == 1, "pressure space must be P1");
    Space& s = c->sp[space];
    s.degree = degree;
    const int d = c->gdim;
    s.nd = degree == 1 ? d + 1 : (d == 2 ? 6 : 10);
    s.n_owned = n_owned;
    s.n_ghost = n_ghost;
    s.cell_dofs.alloc(c->n_cells * s.nd);
    B2_CUDA(cudaMemcpyAsync(s.cell_dofs.p, cell_dofs, sizeof(int) * c->n_cells * s.nd, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(int) * c->n_cells * s.nd;
  });
}

int b2_set_halo(b2_ctx* c, int space, int n_neighbors, const int32_t* neighbor_ranks, const int64_t* send_off,
                const int32_t* send_idx, const int64_t* recv_off) {
  return guarded(c, [&] {
    B2_REQUIRE(space == B2_SPACE_V || space == B2_SPACE_Q, "bad space id");
    B2_REQUIRE(n_neighbors == 0 || c->nranks > 1, "halo plan on a single-rank context");
    Halo& h = c->halo[space];
    h.n_neighbors = n_neighbors;
    h.ranks.assign(neighbor_ranks, neighbor_ranks + n_neighbors);
    h.send_off.assign(send_off, send_off + n_neighbors + 1);
    h.recv_off.assign(recv_off, recv_off + n_neighbors + 1);
    B2_REQUIRE(h.recv_off.back() == c->sp[space].n_ghost, "halo plan does not cover the ghost block");
    h.d_send_off.alloc(n_neighbors + 1);
    h.d_recv_off.alloc(n_neighbors + 1);
    B2_CUDA(cudaMemcpyAsync(h.d_send_off.p, send_off, sizeof(int64_t) * (n_neighbors + 1), cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(h.d_recv_off.p, recv_off, sizeof(int64_t) * (n_neighbors + 1), cudaMemcpyHostToDevice, c->stream));
    const int64_t ns = h.send_off.back(), nr = h.recv_off.back();
    h.send_idx.alloc(ns);
    if (ns) B2_CUDA(cudaMemcpyAsync(h.send_idx.p, send_idx, sizeof(int) * ns, cudaMemcpyHostToDevice, c->stream));
    h.sendbuf.alloc(ns * B2_MAXK);
    h.recvbuf.alloc(nr * B2_MAXK);
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// ---- peer-memory collectives: arena export / import (include/b200ipcs.h) ---------------------------------
int b2_peer_export(b2_ctx* c, int segment, void* blob_out) {
  return guarded(c, [&] {
    B2_REQUIRE(c->nranks > 1 && c->nranks <= B2_MAXR, "peer path: 2..8 ranks of one box");
    B2_REQUIRE(c->use_peer, "peer path disabled (B200_PEER=0)");
    B2_REQUIRE(segment == 0 || segment == 1, "bad segment");
    PeerSeg& sg = c->seg[segment];
    B2_REQUIRE(sg.base == nullptr, "segment already exported");
    PeerBlob blob;
    std::memset(&blob, 0, sizeof(blob));
    if (segment == 0) {
      const int K = std::max(c->gdim, 1);
      blob.cap[0] = std::max<int64_t>(1, c->sp[B2_SPACE_V].n_ghost * K);
      blob.cap[1] = std::max<int64_t>(1, c->sp[B2_SPACE_Q].n_ghost);
      for (int sp = 0; sp < 2; ++sp) {
        const Halo& h = c->halo[sp];
        for (int j = 0; j < h.n_neighbors; ++j) {
          B2_REQUIRE(j == 0 || h.ranks[j] > h.ranks[j - 1], "peer path: neighbour ranks must be strictly increasing");
          blob.recv_cnt[sp][h.ranks[j]] = h.recv_off[j + 1] - h.recv_off[j];
        }
      }
      sg.bytes = PEER_OFF_STAGE + sizeof(LLSlot) * 2 * (size_t)(blob.cap[0] + blob.cap[1]);
    } else {
      B2_REQUIRE(c->peer_on, "segment 0 must be imported first");
      B2_REQUIRE(!c->mg.empty(), "segment 1 carries the first replicated multigrid level: add the levels first");
      blob.cap[0] = c->mg[0].n;
      blob.recv_cnt[0][0] = c->mg_lo;
      blob.recv_cnt[0][1] = c->mg_hi;
      sg.bytes = sizeof(LLSlot) * 2 * (size_t)c->nranks * (size_t)c->mg[0].n;
    }
    B2_CUDA(cudaMalloc(&sg.base, sg.bytes));
    B2_CUDA(cudaMemsetAsync(sg.base, 0, sg.bytes, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    B2_CUDA(cudaIpcGetMemHandle(&blob.handle, sg.base));
    std::memcpy(blob_out, &blob, sizeof(blob));
  });
}

int b2_peer_import(b2_ctx* c, int segment, const void* blobs_in) {
  return guarded(c, [&] {
    B2_REQUIRE(segment == 0 || segment == 1, "bad segment");
    PeerSeg& sg = c->seg[segment];
    B2_REQUIRE(sg.base != nullptr && !sg.imported, "export the segment first (once)");
    const int R = c->nranks, me = c->rank;
    std::vector<PeerBlob> blobs(R);
    std::memcpy(blobs.data(), blobs_in, sizeof(PeerBlob) * R);
    for (int q = 0; q < R; ++q) {
      if (q == me) { sg.peer[q] = sg.base; continue; }
      B2_CUDA(cudaIpcOpenMemHandle(&sg.peer[q], blobs[q].handle, cudaIpcMemLazyEnablePeerAccess));
    }
    sg.imported = true;
    auto at = [](void* base, size_t off) { return (void*)((char*)base + off); };
    if (!c->d_counter_peer) {
      B2_CUDA(cudaMalloc(&c->d_counter_peer, sizeof(unsigned)));
      B2_CUDA(cudaMemsetAsync(c->d_counter_peer, 0, sizeof(unsigned), c->stream));
      B2_CUDA(cudaMallocHost(&c->h_peer_err, sizeof(unsigned long long)));
      *c->h_peer_err = 0;
    }
    unsigned long long* seqs = (unsigned long long*)at(sg.base, PEER_OFF_SEQ);
    if (segment == 0) {
      PeerDev& P = c->h_peer;
      P.nranks = R;
      P.rank = me;
      P.seq_red = seqs + 0;
      P.err = seqs + 4;
      P.slot_red = (LLSlot*)at(sg.base, PEER_OFF_SLOT_RED);
      for (int q = 0; q < R; ++q) P.peer_slot_red[q] = (LLSlot*)at(sg.peer[q], PEER_OFF_SLOT_RED);
      B2_CUDA(cudaMalloc(&c->d_peer, sizeof(PeerDev)));
      B2_CUDA(cudaMemcpyAsync(c->d_peer, &P, sizeof(PeerDev), cudaMemcpyHostToDevice, c->stream));
      for (int sp = 0; sp < 2; ++sp) {
        const Halo& h = c->halo[sp];
        PeerHalo& H = c->ph[sp];
        std::memset(&H, 0, sizeof(H));
        B2_REQUIRE(h.n_neighbors <= B2_MAXR, "too many neighbours");
        H.n_neighbors = h.n_neighbors;
        H.rank = me;
        H.n_owned = (int)c->sp[sp].n_owned;
        H.send_idx = h.send_idx.p;
        H.seq = seqs + 1 + sp;
        H.cap = blobs[me].cap[sp];
        H.recv = (LLSlot*)at(sg.base, PEER_OFF_STAGE) + (sp == 0 ? 0 : 2 * blobs[me].cap[0]);
        H.counter = c->d_counter_peer;
        H.err = P.err;
        for (int j = 0; j <= h.n_neighbors; ++j) { H.send_off[j] = h.send_off[j]; H.recv_off[j] = h.recv_off[j]; }
        for (int j = 0; j < h.n_neighbors; ++j) {
          const int q = h.ranks[j];
          H.nbr[j] = q;
          H.peer_cap[j] = blobs[q].cap[sp];
          H.peer_recv[j] = (LLSlot*)at(sg.peer[q], PEER_OFF_STAGE) + (sp == 0 ? 0 : 2 * blobs[q].cap[0]);
          int64_t off = 0;  // my block in q's staging: after what q receives from lower ranks (its neighbours are sorted)
          for (int r = 0; r < me; ++r) off += blobs[q].recv_cnt[sp][r];
          H.dst_off[j] = off;
          const int64_t mine = h.send_off[j + 1] - h.send_off[j];
          B2_REQUIRE(blobs[q].recv_cnt[sp][me] == mine, "peer path: send count does not match the neighbour's receive count");
        }
      }
      B2_CUDA(cudaStreamSynchronize(c->stream));
      c->peer_on = true;
      c->cfg_version++;
    } else {
      PeerVecSum& V = c->pvs;
      std::memset(&V, 0, sizeof(V));
      V.nranks = R;
      V.rank = me;
      V.n = c->mg[0].n;
      for (int q = 0; q < R; ++q) {
        B2_REQUIRE(blobs[q].cap[0] == V.n, "peer path: ranks disagree on the size of the replicated level");
        V.lo[q] = (int)blobs[q].recv_cnt[0][0];
        V.hi[q] = (int)blobs[q].recv_cnt[0][1];
        V.peer_stage[q] = (LLSlot*)sg.peer[q];
      }
      PeerSeg& s0 = c->seg[0];
      V.seq = (unsigned long long*)at(s0.base, PEER_OFF_SEQ) + 3;
      V.stage = (LLSlot*)sg.base;
      V.counter = c->d_counter_peer;
      V.err = c->h_peer.err;
      c->pvs_ready = true;
      c->cfg_version++;
    }
  });
}

int b2_peer_disable(b2_ctx* c) {
  return guarded(c, [&] {
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->peer_on = false;
    c->pvs_ready = false;
    c->cfg_version++;
  });
}

int b2_peer_enabled(b2_ctx* c) { return c && c->peer_on ? 1 : 0; }

int b2_set_global_sizes(b2_ctx* c, int64_t nv, int64_t nq) {
  return guarded(c, [&] {
    c->sp[B2_SPACE_V].n_global = nv;
    c->sp[B2_SPACE_Q].n_global = nq;
  });
}

int b2_pressure_mg_add_level(b2_ctx* c, int64_t n_nodes, const double* x, int64_t n_cells, const int32_t* cell_nodes,
                             int64_t n_fine_rows, const int32_t* P_indptr, const int32_t* P_indices, const double* P_vals,
                             const int32_t* R_indptr, const int32_t* R_indices, const double* R_vals) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "add multigrid levels after b2_preassemble");
    c->cfg_version++;
    const int d = c->gdim;
    const int64_t fine_n = c->mg.empty() ? c->sp[B2_SPACE_Q].n_owned : c->mg.back().n;
    const int64_t fine_cols = c->mg.empty() ? c->sp[B2_SPACE_Q].n_local() : c->mg.back().n;
    B2_REQUIRE(n_fine_rows == fine_n, "prolongation rows must equal the owned dofs of the previous level");
    c->mg.emplace_back();
    MgLevel& L = c->mg.back();
    L.n = (int)n_nodes;
    // mesh of the level: P1 dofs are the mesh nodes
    DBuf<double> dx;
    DBuf<int> dcells;
    dx.alloc(n_nodes * 3);
    dcells.alloc(n_cells * (d + 1));
    B2_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(double) * n_nodes * 3, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dcells.p, cell_nodes, sizeof(int) * n_cells * (d + 1), cudaMemcpyHostToDevice, c->stream));
    build_pattern_raw(c, n_cells, dcells.p, d + 1, dcells.p, d + 1, L.n, L.n, L.pat);
    build_sell(c, L.pat);
    L.A.alloc(L.pat.slots);
    L.A.zero(c->stream);
    if (d == 2)
      B2_LAUNCH(c, (k_assemble_square<2, 1, B2_FORM_STIFF_Q>), blocks_for(n_cells * 3, 128), 128, n_cells, dx.p, dcells.p, dcells.p,
                L.n, L.pat.rowptr.p, L.pat.cols.p, L.pat.slice_ptr.p, L.A.p);
    else
      B2_LAUNCH(c, (k_assemble_square<3, 1, B2_FORM_STIFF_Q>), blocks_for(n_cells * 4, 128), 128, n_cells, dx.p, dcells.p, dcells.p,
                L.n, L.pat.rowptr.p, L.pat.cols.p, L.pat.slice_ptr.p, L.A.p);
    auto upload_csr = [&](CSR& m, DBuf<double>& vals, int rows, int cols, const int32_t* ip, const int32_t* ix, const double* vv) {
      int nnz = ip[rows];
      m.n_rows = rows; m.n_cols = cols; m.nnz = nnz;
      m.rowptr.alloc(rows + 1); m.cols.alloc(nnz); vals.alloc(nnz);
      B2_CUDA(cudaMemcpyAsync(m.rowptr.p, ip, sizeof(int) * (rows + 1), cudaMemcpyHostToDevice, c->stream));
      if (nnz) {
        B2_CUDA(cudaMemcpyAsync(m.cols.p, ix, sizeof(int) * nnz, cudaMemcpyHostToDevice, c->stream));
        B2_CUDA(cudaMemcpyAsync(vals.p, vv, sizeof(double) * nnz, cudaMemcpyHostToDevice, c->stream));
      }
    };
    upload_csr(L.P, L.Pv, (int)fine_n, L.n, P_indptr, P_indices, P_vals);
    upload_csr(L.R, L.Rv, L.n, (int)fine_cols, R_indptr, R_indices, R_vals);
    if (c->mg.size() == 1) mg_set_restrict_range(c, R_indptr, L.n);
    mg_level_finish(c, L);
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_pressure_amg_build(b2_ctx* c) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "b2_pressure_amg_build: call it after b2_preassemble");
    B2_REQUIRE(c->mg.empty(), "b2_pressure_amg_build: the context already has a multigrid hierarchy");
    B2_REQUIRE(!c->has_pbc, "b2_pressure_amg_build: the pressure has Dirichlet dofs (the coarse solve assumes the constant null space)");
    B2_REQUIRE(c->nranks == 1 || c->q_gid.p != nullptr,
               "b2_pressure_amg_build: several ranks need the global pressure dof ids first (b2_set_pressure_global_ids)");
    if (c->q_gid.p != nullptr) {
      amg_build_gathered(c);
      return;
    }
    DBuf<double> vals;
    const CSR* pat = nullptr;
    csr_values(c, B2_MAT_AP, 0, vals, &pat);
    amg_build(c, c->pat[B2_PAT_QQ], std::move(vals), c->dinvAp.p);
  });
}

int b2_set_pressure_global_ids(b2_ctx* c, int64_t n, const int64_t* gids) {
  return guarded(c, [&] {
    const Space& Q = c->sp[B2_SPACE_Q];
    const int64_t ng = Q.n_global, n_owned = Q.n_owned;
    B2_REQUIRE(n == Q.n_local(), "b2_set_pressure_global_ids: one global index per local pressure dof, owned then ghost");
    B2_REQUIRE(ng > 0 && ng <= (1ll << 31), "b2_set_pressure_global_ids: set the global sizes first (b2_set_global_sizes), below 2^31");
    // local checks first, but every rank takes part in the exchange below before any of them fails
    int64_t bad = 0;  // 1: an index outside [0, n_global), 2: an index listed twice
    for (int64_t i = 0; i < n; ++i)
      if (gids[i] < 0 || gids[i] >= ng) bad = 1;
    if (!bad) {
      std::vector<int64_t> s(gids, gids + n);
      std::sort(s.begin(), s.end());
      if (std::adjacent_find(s.begin(), s.end()) != s.end()) bad = 2;
    }
    const int64_t mine[2] = {n_owned, bad};
    const std::vector<int64_t> all = allgather_i64(c, mine, 2);
    std::vector<int64_t> counts(c->nranks);
    int64_t total = 0;
    for (int q = 0; q < c->nranks; ++q) {
      B2_REQUIRE(all[2 * q + 1] == 0, "b2_set_pressure_global_ids: rank " + std::to_string(q) +
                                          (all[2 * q + 1] == 1 ? " has a global index outside [0, n_global)"
                                                               : " lists the same global index twice"));
      counts[q] = all[2 * q];
      total += counts[q];
    }
    B2_REQUIRE(total == ng, "b2_set_pressure_global_ids: the ranks own " + std::to_string(total) + " dofs, not n_global = " +
                                std::to_string(ng));
    std::vector<int32_t> ids(gids, gids + n);
    c->q_gid.alloc(n);
    B2_CUDA(cudaMemcpyAsync(c->q_gid.p, ids.data(), sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    // the owned indices of all ranks cover 0 .. n_global-1 exactly once
    DBuf<int> owned;
    owned.alloc(ng);
    allgatherv(c, c->q_gid.p, counts, owned.p, ncclInt32, sizeof(int));
    std::vector<int32_t> h(ng);
    B2_CUDA(cudaMemcpyAsync(h.data(), owned.p, sizeof(int) * ng, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    std::vector<char> seen(ng, 0);
    for (int32_t g : h) {
      if (seen[g]) {
        c->q_gid.release();
        throw B2Error(-1, "b2_set_pressure_global_ids: global index " + std::to_string(g) + " is owned twice");
      }
      seen[g] = 1;
    }
  });
}

int b2_pressure_mg_level_info(b2_ctx* c, int level, double* out) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "multigrid levels exist after b2_preassemble");
    B2_REQUIRE(level >= 0 && level <= (int)c->mg.size(), "no such multigrid level");
    if (level == 0) {
      const CSR& qq = c->pat[B2_PAT_QQ];
      const double v[7] = {(double)qq.n_rows, (double)qq.nnz, 0.0, c->mg_omega0 > 0.0 ? 1.0 : 0.0, 0.0, mg_level_omega(c, 0), c->mg_rho0};
      std::memcpy(out, v, sizeof(v));
      return;
    }
    const MgLevel& M = c->mg[level - 1];
    const bool dense = level - 1 == c->mg_dense_level && c->mg_dense_on;
    const double v[7] = {(double)M.n, (double)M.pat.nnz, (double)M.P.nnz, M.algebraic ? 1.0 : 0.0, dense ? 1.0 : 0.0,
                         mg_level_omega(c, level), M.rho};
    std::memcpy(out, v, sizeof(v));
  });
}

int b2_pressure_mg_get_level(b2_ctx* c, int level, int what, int32_t* indptr, int32_t* indices, double* vals) {
  return guarded(c, [&] {
    B2_REQUIRE(level >= 1 && level <= (int)c->mg.size(), "no such coarse multigrid level");
    B2_REQUIRE(what >= 0 && what <= 3, "what: 0 = A, 1 = P, 2 = R, 3 = aggregates");
    MgLevel& M = c->mg[level - 1];
    auto d2h = [&](void* dst, const void* src, size_t bytes) {
      if (bytes) B2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    };
    if (what == 3) {
      B2_REQUIRE(M.algebraic, "aggregates exist on algebraic levels only");
      d2h(indices, M.agg.p, sizeof(int) * M.P.n_rows);
    } else {
      const CSR& m = what == 0 ? M.pat : (what == 1 ? M.P : M.R);
      d2h(indptr, m.rowptr.p, sizeof(int) * (m.n_rows + 1));
      d2h(indices, m.cols.p, sizeof(int) * m.nnz);
      if (what == 0) {
        DBuf<double> v;
        v.alloc(m.nnz);
        B2_LAUNCH(c, k_sell_convert, blocks_for(m.n_rows, 256), 256, m.n_rows, m.rowptr.p, m.slice_ptr.p, 0, M.A.p, v.p,
                  (const double*)nullptr);
        d2h(vals, v.p, sizeof(double) * m.nnz);
        B2_CUDA(cudaStreamSynchronize(c->stream));
      } else {
        d2h(vals, (what == 1 ? M.Pv : M.Rv).p, sizeof(double) * m.nnz);
      }
    }
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_pressure_mg_configure(b2_ctx* c, int nu_pre, int nu_post, int coarse_sweeps, double omega) {
  return guarded(c, [&] {
    B2_REQUIRE(nu_pre >= 1 && nu_post >= 0 && coarse_sweeps >= 1 && omega > 0 && omega < 2, "bad multigrid parameters");
    c->cfg_version++;
    c->mg_pre = nu_pre;
    c->mg_post = nu_post;
    c->mg_coarse = coarse_sweeps;
    c->mg_omega = omega;
  });
}

int b2_set_slice_order(b2_ctx* c, int pattern, int64_t n_slices, const int32_t* order) {
  return guarded(c, [&] {
    B2_REQUIRE(c->patterns_built && (pattern == B2_PAT_VV || pattern == B2_PAT_QQ), "slice order: square patterns, after b2_build_patterns");
    CSR& pat = c->pat[pattern];
    B2_REQUIRE(n_slices == (pat.n_rows + 31) / 32, "slice order length must equal the number of 32-row slices");
    c->cfg_version++;
    pat.order.alloc(n_slices);
    B2_CUDA(cudaMemcpyAsync(pat.order.p, order, sizeof(int) * n_slices, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_build_patterns(b2_ctx* c) {
  return guarded(c, [&] {
    Space &V = c->sp[B2_SPACE_V], &Q = c->sp[B2_SPACE_Q];
    B2_REQUIRE(V.nd && Q.nd, "both spaces must be set before building patterns");
    build_pattern(c, V, V, c->pat[B2_PAT_VV]);
    build_pattern(c, V, Q, c->pat[B2_PAT_VQ]);
    build_pattern(c, Q, V, c->pat[B2_PAT_QV]);
    build_pattern(c, Q, Q, c->pat[B2_PAT_QQ]);
    build_sell(c, c->pat[B2_PAT_VV]);
    build_sell(c, c->pat[B2_PAT_QQ]);
    build_sell(c, c->pat[B2_PAT_VQ]);  // P_i / G_i live in the sliced-ELL form too (component-major values)
    c->patterns_built = true;
  });
}

int64_t b2_pattern_nnz(b2_ctx* c, int pattern) {
  if (!c || pattern < 0 || pattern > 3 || !c->patterns_built) return -1;
  return c->pat[pattern].nnz;
}

int64_t b2_pattern_sell_slots(b2_ctx* c, int pattern) {
  if (!c || pattern < 0 || pattern > 3 || !c->patterns_built || !c->pat[pattern].has_sell()) return -1;
  return c->pat[pattern].slots;
}

int b2_get_pattern(b2_ctx* c, int pattern, int32_t* indptr, int32_t* indices) {
  return guarded(c, [&] {
    B2_REQUIRE(c->patterns_built && pattern >= 0 && pattern <= 3, "pattern not available");
    const CSR& p = c->pat[pattern];
    B2_CUDA(cudaMemcpyAsync(indptr, p.rowptr.p, sizeof(int) * (p.n_rows + 1), cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaMemcpyAsync(indices, p.cols.p, sizeof(int) * p.nnz, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_d2h += sizeof(int) * (p.n_rows + 1 + p.nnz);
  });
}

int b2_set_velocity_bc_dofs(b2_ctx* c, int comp, int64_t n, const int32_t* dofs) {
  return guarded(c, [&] {
    B2_REQUIRE(comp >= 0 && comp < c->gdim, "bad component");
    c->bc_dofs[comp].alloc(n);
    c->bc_vals[comp].alloc(n);
    c->bc_vals[comp].zero(c->stream);
    if (n) B2_CUDA(cudaMemcpyAsync(c->bc_dofs[comp].p, dofs, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    if (c->preassembled && comp == 0) {
      // component 0's dof set drives the unit rows of the shared matrix (fracstep.py:470-472): rebuild the row mask
      c->is_bc_row_v.zero(c->stream);
      if (n) B2_LAUNCH(c, k_mark, blocks_for(n, 256), 256, n, c->bc_dofs[0].p, c->is_bc_row_v.p);
    }
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(int) * n;
  });
}

int b2_set_velocity_bc_values(b2_ctx* c, int comp, int64_t n, const double* values) {
  return guarded(c, [&] {
    B2_REQUIRE(comp >= 0 && comp < c->gdim, "bad component");
    B2_REQUIRE(n == c->bc_dofs[comp].n, "BC value count does not match the dof list");
    if (n) B2_CUDA(cudaMemcpyAsync(c->bc_vals[comp].p, values, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->bc_step = -1;  // fresh values override a prefetched series
    c->stats.bytes_h2d += sizeof(double) * n;
  });
}

int b2_set_velocity_bc_series(b2_ctx* c, int comp, int n_steps, int64_t n, const double* values) {
  return guarded(c, [&] {
    B2_REQUIRE(comp >= 0 && comp < c->gdim, "bad component");
    B2_REQUIRE(n == c->bc_dofs[comp].n && n_steps >= 0, "BC series does not match the dof list");
    c->bc_series[comp].alloc((int64_t)n_steps * n);
    c->bc_series_steps[comp] = n_steps;
    if (n_steps * n)
      B2_CUDA(cudaMemcpyAsync(c->bc_series[comp].p, values, sizeof(double) * n_steps * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(double) * n_steps * n;
  });
}

int b2_select_bc_step(b2_ctx* c, int step) {
  return guarded(c, [&] { c->bc_step = step; });
}

int b2_profiler_range(b2_ctx* c, int on) {
  return guarded(c, [&] {
    B2_CUDA(cudaStreamSynchronize(c->stream));
    if (on) B2_CUDA(cudaProfilerStart());
    else B2_CUDA(cudaProfilerStop());
  });
}

int b2_reset_time_history(b2_ctx* c) {
  return guarded(c, [&] {
    c->steps_done = 0;
    c->dp_hist = 0;
    c->n_ustar_hist = 0;
    c->n_delta_hist = 0;
    c->fresh_step = true;
    if (c->delta_prev.p) c->delta_prev.zero(c->stream);
    if (c->dp_old.p) c->dp_old.zero(c->stream);
    for (auto& o : c->ksp) o.expected_its = 0;
  });
}

int b2_declare_pressure_bcs(b2_ctx* c, int any) {
  return guarded(c, [&] {
    B2_REQUIRE(!c->preassembled, "pressure BCs must be declared before b2_preassemble");
    c->has_pbc = any != 0;
  });
}

int b2_set_pressure_bc_dofs(b2_ctx* c, int64_t n, const int32_t* dofs) {
  return guarded(c, [&] {
    B2_REQUIRE(!c->preassembled, "pressure BC dofs must be set before b2_preassemble");
    c->pbc_dofs.alloc(n);
    c->has_pbc = c->has_pbc || n > 0;
    if (n) B2_CUDA(cudaMemcpyAsync(c->pbc_dofs.p, dofs, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_preassemble(b2_ctx* c, const double* body_force, int low_memory, int rotational) {
  return guarded(c, [&] { do_preassemble(c, body_force, low_memory, rotational); });
}

int b2_set_vector(b2_ctx* c, int vec, int comp, const double* host, int64_t n) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "vectors exist after b2_preassemble");
    auto it = c->vecs.find(vec);
    B2_REQUIRE(it != c->vecs.end(), "unknown vector id");
    DVec& v = it->second;
    const int64_t nl = c->sp[v.space].n_local();
    if (v.K > 1 && comp < 0) {  // whole blocked array [n][K] -> component-major
      B2_REQUIRE(n == nl * v.K, "size mismatch in b2_set_vector");
      B2_CUDA(cudaMemcpyAsync(c->stage.p, host, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
      B2_LAUNCH(c, k_from_blocked, pgrid(c, n), 256, nl, v.K, (int)nl, c->stage.p, v.buf.p);
    } else {
      B2_REQUIRE(comp >= 0 && comp < v.K && n == nl, "size/component mismatch in b2_set_vector");
      B2_CUDA(cudaMemcpyAsync(v.buf.p + (size_t)comp * nl, host, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    }
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(double) * n;
  });
}

int b2_get_vector(b2_ctx* c, int vec, int comp, double* host, int64_t n) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "vectors exist after b2_preassemble");
    auto it = c->vecs.find(vec);
    B2_REQUIRE(it != c->vecs.end(), "unknown vector id");
    DVec& v = it->second;
    const int64_t nl = c->sp[v.space].n_local();
    halo_forward(c, v.space, v.buf.p, v.K);  // ghost copies are refreshed lazily: do it before handing them out
    if (v.K > 1 && comp < 0) {
      B2_REQUIRE(n == nl * v.K, "size mismatch in b2_get_vector");
      B2_LAUNCH(c, k_to_blocked, pgrid(c, n), 256, nl, v.K, (int)nl, v.buf.p, c->stage.p);
      B2_CUDA(cudaMemcpyAsync(host, c->stage.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    } else {
      B2_REQUIRE(comp >= 0 && comp < v.K && n == nl, "size/component mismatch in b2_get_vector");
      B2_CUDA(cudaMemcpyAsync(host, v.buf.p + (size_t)comp * nl, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    }
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_d2h += sizeof(double) * n;
  });
}

}  // extern "C"

namespace {

// CSR-ordered copy of a matrix' values (direction comp of P, G, D)
void csr_values(b2_ctx* c, int mat, int comp, DBuf<double>& out, const CSR** pat_out) {
  const CSR* pat = nullptr;
  Layout layout;
  const DBuf<double>* v = matrix_values(c, mat, &pat, &layout);
  B2_REQUIRE(v->p != nullptr, "matrix not assembled (rotational/low-memory option?)");
  B2_REQUIRE(layout == Layout::Sell || (comp >= 0 && comp < c->gdim), "bad component");
  out.alloc(pat->nnz);
  if (layout == Layout::CsrInterleaved) {
    B2_LAUNCH(c, k_extract, pgrid(c, pat->nnz), 256, pat->nnz, c->gdim, comp, v->p, out.p);
  } else {
    const double* vals = layout == Layout::SellByComp ? v->p + (size_t)comp * pat->slots : v->p;
    B2_LAUNCH(c, k_sell_convert, blocks_for(pat->n_rows, 256), 256, pat->n_rows, pat->rowptr.p, pat->slice_ptr.p, 0, vals,
              out.p, (const double*)nullptr);
  }
  *pat_out = pat;
}

// ---- smoothed-aggregation AMG set-up (amg.cuh) ----------------------------------------------------
template <typename T>
T read_scalar(b2_ctx* c, const T* d) {
  T h{};
  B2_CUDA(cudaMemcpyAsync(&h, d, sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return h;
}

template <typename T>
void exclusive_sum(b2_ctx* c, const T* in, T* out, int64_t n) {
  size_t bytes = 0;
  B2_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, c->stream));
  DBuf<char> tmp;
  tmp.alloc((int64_t)bytes);
  B2_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, bytes, in, out, n, c->stream));
}

// n pairs (row << 32 | col, value) in a deterministic generation order -> CSR with sorted columns; the values of equal
// keys are summed sequentially in that order (stable radix sort, one thread per run), so the result is the same bit
// for bit on every run.  The pair buffers are consumed.
void amg_pairs_to_csr(b2_ctx* c, DBuf<unsigned long long>& keys, DBuf<double>& vals, int64_t n, int n_rows, int n_cols,
                      CSR& out, DBuf<double>& out_vals) {
  B2_REQUIRE(n < (1ll << 31), "algebraic multigrid: sparse product too large for int32 indices");
  DBuf<unsigned long long> k2;
  DBuf<double> v2;
  k2.alloc(n);
  v2.alloc(n);
  int row_bits = 1;
  while ((1ll << row_bits) <= (int64_t)n_rows) ++row_bits;
  cub::DoubleBuffer<unsigned long long> kb(keys.p, k2.p);
  cub::DoubleBuffer<double> vb(vals.p, v2.p);
  size_t bytes = 0;
  B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kb, vb, n, 0, 32 + row_bits, c->stream));
  DBuf<char> tmp;
  tmp.alloc((int64_t)bytes);
  B2_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, kb, vb, n, 0, 32 + row_bits, c->stream));
  DBuf<int> head, run;
  head.alloc(n + 1);
  run.alloc(n + 1);
  B2_LAUNCH(c, k_amg_heads, blocks_for(n + 1, 256), 256, n, kb.Current(), head.p);
  exclusive_sum(c, head.p, run.p, n + 1);
  const int n_unique = read_scalar(c, run.p + n);
  DBuf<unsigned long long> uk;
  uk.alloc(n_unique);
  out_vals.alloc(n_unique);
  B2_LAUNCH(c, k_amg_reduce_runs, blocks_for(n, 256), 256, n, kb.Current(), vb.Current(), head.p, run.p, uk.p, out_vals.p);
  out.n_rows = n_rows;
  out.n_cols = n_cols;
  out.nnz = n_unique;
  out.rowptr.alloc(n_rows + 1);
  out.cols.alloc(n_unique);
  B2_LAUNCH(c, k_keys_to_csr, blocks_for((int64_t)n_unique + 1, 256), 256, (int64_t)n_unique, uk.p, n_rows, out.rowptr.p, out.cols.p);
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// C = A B (CSR, sorted columns) by expansion into one pair per product, sort and reduce
void amg_spgemm(b2_ctx* c, const CSR& A, const double* va, const CSR& B, const double* vb, CSR& C, DBuf<double>& vc) {
  const int64_t nnz = A.nnz;
  DBuf<int> rows;
  DBuf<int64_t> cnt, off;
  rows.alloc(nnz);
  cnt.alloc(nnz + 1);
  off.alloc(nnz + 1);
  cnt.zero(c->stream);
  B2_LAUNCH(c, k_amg_entry_rows, blocks_for(A.n_rows, 256), 256, A.n_rows, A.rowptr.p, rows.p);
  B2_LAUNCH(c, k_amg_product_counts, blocks_for(nnz, 256), 256, nnz, A.cols.p, B.rowptr.p, cnt.p);
  exclusive_sum(c, cnt.p, off.p, nnz + 1);
  const int64_t total = read_scalar(c, off.p + nnz);
  DBuf<unsigned long long> keys;
  DBuf<double> vals;
  keys.alloc(total);
  vals.alloc(total);
  B2_LAUNCH(c, k_amg_expand, blocks_for(nnz, 256), 256, nnz, rows.p, A.cols.p, va, B.rowptr.p, B.cols.p, vb, off.p, keys.p, vals.p);
  amg_pairs_to_csr(c, keys, vals, total, A.n_rows, B.n_cols, C, vc);
}

void amg_transpose(b2_ctx* c, const CSR& A, const double* va, CSR& T, DBuf<double>& vt) {
  DBuf<int> rows;
  rows.alloc(A.nnz);
  DBuf<unsigned long long> keys;
  DBuf<double> vals;
  keys.alloc(A.nnz);
  vals.alloc(A.nnz);
  B2_LAUNCH(c, k_amg_entry_rows, blocks_for(A.n_rows, 256), 256, A.n_rows, A.rowptr.p, rows.p);
  B2_LAUNCH(c, k_amg_transpose_keys, blocks_for(A.nnz, 256), 256, A.nnz, rows.p, A.cols.p, va, keys.p, vals.p);
  amg_pairs_to_csr(c, keys, vals, A.nnz, A.n_cols, A.n_rows, T, vt);
}

// rho(D^-1 A) from 20 power iterations (normalised on the device, no host round trip; sums in a fixed order), reported as the Rayleigh
// quotient x^T A x / x^T D x of the last iterate: D^-1 A is self-adjoint in the D inner product, so the estimate is
// a lower bound whose error is quadratic in the iterate's
double amg_spectral_radius(b2_ctx* c, const CSR& A, const double* va, const double* dinv) {
  const int n = A.n_rows;
  DBuf<double> x, y, y2, sums;
  x.alloc(n);
  y.alloc(n);
  y2.alloc(n);
  sums.alloc(3);
  B2_LAUNCH(c, k_amg_seed, blocks_for(n, 256), 256, n, x.p);
  for (int k = 0; k < 20; ++k) {
    B2_LAUNCH(c, k_amg_power, blocks_for(n, 256), 256, n, A.rowptr.p, A.cols.p, va, dinv, x.p, k == 0 ? nullptr : sums.p,
              y.p, y2.p);
    B2_LAUNCH(c, k_amg_sum, 1, 1024, n, y2.p, sums.p);
    std::swap(x.p, y.p);
  }
  B2_LAUNCH(c, k_amg_rayleigh, blocks_for(n, 256), 256, n, A.rowptr.p, A.cols.p, va, dinv, x.p, y.p, y2.p);
  B2_LAUNCH(c, k_amg_sum, 1, 1024, n, y.p, sums.p + 1);
  B2_LAUNCH(c, k_amg_sum, 1, 1024, n, y2.p, sums.p + 2);
  double h[3];
  B2_CUDA(cudaMemcpyAsync(h, sums.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_REQUIRE(h[2] > 0.0 && h[1] > 0.0, "algebraic multigrid: spectral radius estimate failed");
  return h[1] / h[2];
}

// MIS(2) aggregation of the strength graph of A; returns the number of aggregates
int amg_aggregate(b2_ctx* c, const CSR& A, const double* va, DBuf<int>& agg) {
  const int n = A.n_rows;
  B2_REQUIRE(n < (1 << 30), "algebraic multigrid: at most 2^30 dofs");
  const int g = blocks_for(n, 256);
  DBuf<int> state, cnt, flag, id, agg1;
  DBuf<unsigned long long> t0, m1, m2;
  state.alloc(n);
  cnt.alloc(1);
  t0.alloc(n);
  m1.alloc(n);
  m2.alloc(n);
  B2_LAUNCH(c, k_amg_init, g, 256, n, state.p);
  for (int round = 0;; ++round) {
    B2_REQUIRE(round <= n, "algebraic multigrid: MIS(2) did not terminate");
    cnt.zero(c->stream);
    B2_LAUNCH(c, k_amg_tuples, g, 256, n, state.p, t0.p);
    B2_LAUNCH(c, k_amg_max_hop, g, 256, n, A.rowptr.p, A.cols.p, va, t0.p, m1.p);
    B2_LAUNCH(c, k_amg_max_hop, g, 256, n, A.rowptr.p, A.cols.p, va, m1.p, m2.p);
    B2_LAUNCH(c, k_amg_mis_update, g, 256, n, state.p, t0.p, m2.p, cnt.p);
    if (read_scalar(c, cnt.p) == 0) break;
  }
  flag.alloc(n + 1);
  id.alloc(n + 1);
  flag.zero(c->stream);
  B2_LAUNCH(c, k_amg_root_flags, g, 256, n, state.p, flag.p);
  exclusive_sum(c, flag.p, id.p, (int64_t)n + 1);
  const int nc = read_scalar(c, id.p + n);
  agg1.alloc(n);
  agg.alloc(n);
  cnt.zero(c->stream);
  B2_LAUNCH(c, k_amg_pass1, g, 256, n, A.rowptr.p, A.cols.p, va, state.p, id.p, agg1.p);
  B2_LAUNCH(c, k_amg_pass2, g, 256, n, A.rowptr.p, A.cols.p, va, agg1.p, agg.p, cnt.p);
  B2_REQUIRE(read_scalar(c, cnt.p) == 0, "algebraic multigrid: a node was left without an aggregate");
  return nc;
}

// Smoothed-aggregation hierarchy of the fine operator A0 (CSR with sorted columns, its values in CSR order, its inverse
// diagonal), coarsened until a level is small enough for the exact dense solve, the coarsening ratio drops below 2, or
// 15 coarse levels (the single-block sub-cycle's tables hold 16).  One rank passes Ap itself; several ranks pass the
// gathered global Ap (amg_build_gathered), so that every rank builds the same hierarchy.
void amg_build(b2_ctx* c, const CSR& A0, DBuf<double> vals, const double* dinv0) {
  c->cfg_version++;
  const CSR* A = &A0;
  const double* dinv = dinv0;
  c->mg_rho0 = amg_spectral_radius(c, *A, vals.p, dinv);
  c->mg_omega0 = 4.0 / (3.0 * c->mg_rho0);
  double omega_p = c->mg_omega0;
  c->mg.reserve(16);  // A points into c->mg below
  while (c->mg.size() < 15) {
    const int n = A->n_rows;
    DBuf<int> agg;
    const int nc = amg_aggregate(c, *A, vals.p, agg);
    if (nc >= n) break;  // no coarsening at all
    // P = (I - omega_P D^-1 A) T
    CSR T;
    DBuf<double> tv, sv;
    T.n_rows = n;
    T.n_cols = nc;
    T.nnz = n;
    T.rowptr.alloc(n + 1);
    T.cols.alloc(n);
    tv.alloc(n);
    B2_LAUNCH(c, k_amg_tentative, blocks_for(n + 1, 256), 256, n, agg.p, T.rowptr.p, T.cols.p, tv.p);
    sv.alloc(A->nnz);
    B2_LAUNCH(c, k_amg_smoother, blocks_for(n, 256), 256, n, A->rowptr.p, A->cols.p, vals.p, dinv, omega_p, sv.p);
    c->mg.emplace_back();
    MgLevel& L = c->mg.back();
    L.algebraic = true;
    L.n = nc;
    L.agg = std::move(agg);
    amg_spgemm(c, *A, sv.p, T, tv.p, L.P, L.Pv);
    amg_transpose(c, L.P, L.Pv.p, L.R, L.Rv);
    // A_c = R (A P)
    CSR AP;
    DBuf<double> apv, acv;
    amg_spgemm(c, *A, vals.p, L.P, L.Pv.p, AP, apv);
    amg_spgemm(c, L.R, L.Rv.p, AP, apv.p, L.pat, acv);
    build_sell(c, L.pat);
    L.A.alloc(L.pat.slots);
    L.A.zero(c->stream);
    B2_LAUNCH(c, k_sell_convert, blocks_for(nc, 256), 256, nc, L.pat.rowptr.p, L.pat.slice_ptr.p, 1, acv.p, L.A.p,
              (const double*)nullptr);
    mg_level_finish(c, L);
    L.rho = amg_spectral_radius(c, L.pat, acv.p, L.dinv.p);
    L.omega = 4.0 / (3.0 * L.rho);
    omega_p = L.omega;
    vals = std::move(acv);
    A = &L.pat;
    dinv = L.dinv.p;
    if (nc <= c->mg_dense_max || 2 * (int64_t)nc > n) break;
  }
  B2_CUDA(cudaStreamSynchronize(c->stream));
}

// Several ranks: every rank expands its owned rows of Ap into (global row << 32 | global col, value) pairs, the pairs
// of all ranks are gathered in rank order, and every rank builds the global Ap from them and the hierarchy from that.
// Each entry comes from exactly one rank (b2_set_pressure_global_ids checked that the owned rows cover the global
// range once), so nothing is summed and every rank holds the same matrix bit for bit.  Levels 2 and below stay global
// and replicated; level 1 is then cut back to this rank's owned rows: P_1 keeps the rows of the owned dofs in local
// order, R_1 = P_1^T has local columns (ghost columns empty), the aggregates are those of the owned dofs.
void amg_build_gathered(b2_ctx* c) {
  const CSR& qq = c->pat[B2_PAT_QQ];
  const Space& Q = c->sp[B2_SPACE_Q];
  const int n_owned = qq.n_rows, ng = (int)Q.n_global;
  CSR A;
  DBuf<double> av;
  {
    DBuf<double> vals;
    const CSR* pat = nullptr;
    csr_values(c, B2_MAT_AP, 0, vals, &pat);
    DBuf<unsigned long long> mk, keys;
    DBuf<double> mv, kv;
    mk.alloc(qq.nnz);
    mv.alloc(qq.nnz);
    B2_LAUNCH(c, k_amg_global_pairs, blocks_for(n_owned, 256), 256, n_owned, qq.rowptr.p, qq.cols.p, vals.p, c->q_gid.p, mk.p, mv.p);
    const std::vector<int64_t> counts = allgather_i64(c, &qq.nnz, 1);
    int64_t total = 0;
    for (int64_t k : counts) total += k;
    keys.alloc(total);
    kv.alloc(total);
    allgatherv(c, mk.p, counts, keys.p, ncclUint64, sizeof(unsigned long long));
    allgatherv(c, mv.p, counts, kv.p, ncclDouble, sizeof(double));
    mk.release();
    mv.release();
    vals.release();
    amg_pairs_to_csr(c, keys, kv, total, ng, ng, A, av);
    B2_REQUIRE(A.nnz == total, "algebraic multigrid: two ranks contributed the same entry of Ap");
  }
  DBuf<double> dinv;
  dinv.alloc(ng);
  B2_LAUNCH(c, k_amg_inv_diag, blocks_for(ng, 256), 256, ng, A.rowptr.p, A.cols.p, av.p, dinv.p);
  amg_build(c, A, std::move(av), dinv.p);
  A = CSR();
  dinv.release();

  MgLevel& L = c->mg[0];
  CSR P;
  DBuf<double> pv;
  DBuf<int> len, agg;
  P.n_rows = n_owned;
  P.n_cols = L.n;
  P.rowptr.alloc(n_owned + 1);
  len.alloc(n_owned + 1);
  len.zero(c->stream);
  B2_LAUNCH(c, k_amg_row_lengths, blocks_for(n_owned, 256), 256, n_owned, L.P.rowptr.p, c->q_gid.p, len.p);
  exclusive_sum(c, len.p, P.rowptr.p, (int64_t)n_owned + 1);
  P.nnz = read_scalar(c, P.rowptr.p + n_owned);
  P.cols.alloc(P.nnz);
  pv.alloc(P.nnz);
  agg.alloc(n_owned);
  B2_LAUNCH(c, k_amg_gather_rows, blocks_for(n_owned, 256), 256, n_owned, L.P.rowptr.p, L.P.cols.p, L.Pv.p, L.agg.p, c->q_gid.p,
            P.rowptr.p, P.cols.p, pv.p, agg.p);
  L.P = std::move(P);
  L.Pv = std::move(pv);
  L.agg = std::move(agg);
  amg_transpose(c, L.P, L.Pv.p, L.R, L.Rv);
  L.R.n_cols = (int)Q.n_local();
  std::vector<int32_t> rp(L.n + 1);
  B2_CUDA(cudaMemcpyAsync(rp.data(), L.R.rowptr.p, sizeof(int) * (L.n + 1), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  mg_set_restrict_range(c, rp.data(), L.n);
}

}  // namespace

extern "C" {

int b2_get_matrix_values(b2_ctx* c, int mat, int comp, double* host) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "matrices exist after b2_preassemble");
    DBuf<double> tmp;
    const CSR* pat = nullptr;
    csr_values(c, mat, comp, tmp, &pat);
    B2_CUDA(cudaMemcpyAsync(host, tmp.p, sizeof(double) * pat->nnz, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_d2h += sizeof(double) * pat->nnz;
  });
}

// y = Mat * x through the products of the time step: the SELL SpMM for square operators; rect_vq for P_i and G_i (every
// direction computed, direction comp returned); rect_qv for D_i (the other directions of its input set to zero)
int b2_mat_mult(b2_ctx* c, int mat, int comp, const double* x, double* y) {
  return guarded(c, [&] {
    B2_REQUIRE(c->preassembled, "matrices exist after b2_preassemble");
    const CSR* pat = nullptr;
    Layout layout;
    const DBuf<double>* v = matrix_values(c, mat, &pat, &layout);
    B2_REQUIRE(v->p != nullptr, "matrix not assembled");
    B2_REQUIRE(layout == Layout::Sell || (comp >= 0 && comp < c->gdim), "bad component");
    const int64_t nv = c->sp[B2_SPACE_V].n_local();  // ld of velocity-space vectors
    DBuf<double> dx, dy;
    const double* yk = nullptr;
    if (layout == Layout::Sell) {
      dx.alloc(pat->n_cols);
      dy.alloc(pat->n_rows);
      B2_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(double) * pat->n_cols, cudaMemcpyHostToDevice, c->stream));
      spmm(c, *pat, v->p, 1, dx.p, dy.p);
      yk = dy.p;
    } else if (layout == Layout::SellByComp) {
      dx.alloc(pat->n_cols);
      dy.alloc(c->gdim * nv);
      B2_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(double) * pat->n_cols, cudaMemcpyHostToDevice, c->stream));
      rect_vq(c, v->p, dx.p, nullptr, 1.0, dy.p);
      yk = dy.p + comp * nv;
    } else {
      dx.alloc(c->gdim * nv);
      dx.zero(c->stream);
      dy.alloc(pat->n_rows);
      B2_CUDA(cudaMemcpyAsync(dx.p + comp * nv, x, sizeof(double) * pat->n_cols, cudaMemcpyHostToDevice, c->stream));
      rect_qv(c, dx.p, 1.0, nullptr, dy.p);
      yk = dy.p;
    }
    B2_CUDA(cudaMemcpyAsync(y, yk, sizeof(double) * pat->n_rows, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_set_solver_option(b2_ctx* c, int solver, const char* key, const char* value) {
  return guarded(c, [&] {
    B2_REQUIRE(solver >= 0 && solver < 4, "bad solver id");
    KSPOpts& o = c->ksp[solver];
    std::string k(key), v(value);
    if (k == "ksp_type") {
      if (v == "cg") o.type = 0;
      else if (v == "bcgs" || v == "bicgstab") o.type = 1;
      else if (v == "preonly") { /* direct solve requested: keep the Krylov default, tighten below */ }
      else if (v == "gmres") {
        // the pressure solve is CG (with multigrid or Jacobi); PETSc would accept GMRES there
        B2_REQUIRE(solver != B2_SOLVER_PRESSURE, "ksp_type gmres is not available for the pressure solve (cg only)");
        o.type = 3;
      }
      else if (v == "chebyshev") {
        B2_REQUIRE(solver == B2_SOLVER_SCALAR || solver == B2_SOLVER_PROJECTOR, "chebyshev is for the SPD mass solves");
        o.type = 2;
      }
      else throw B2Error(-5, "unsupported ksp_type " + v);
      if (o.type == 1) B2_REQUIRE(solver == B2_SOLVER_TENTATIVE || solver == B2_SOLVER_SCALAR, "bcgs only on the velocity space");
    } else if (k == "pc_type") {
      if (v == "jacobi") o.pc = 0;
      else if (v == "none") o.pc = 1;
      else if (v == "mg" || v == "gamg" || v == "hypre") o.pc = (solver == B2_SOLVER_PRESSURE) ? 2 : 0;
      else if (v == "lu" || v == "cholesky") { o.pc = 0; o.rtol = 1e-12; o.atol = 1e-50; }  // "exact" solve (Appendix G)
      else throw B2Error(-5, "unsupported pc_type " + v + " (jacobi | none | mg | gamg | hypre | lu | cholesky)");  // PETSc errors on an unknown PC type too
    } else if (k == "ksp_gmres_restart") {
      const int m = std::stoi(v);
      B2_REQUIRE(m >= 1 && m <= B2_GMRES_MAXM, "ksp_gmres_restart must be in 1.." + std::to_string(B2_GMRES_MAXM));
      o.restart = m;
    } else if (k == "ksp_gmres_cgs_refinement_type") {
      std::string u = v;
      for (auto& ch : u) ch = (char)std::tolower((unsigned char)ch);
      if (u.rfind("ksp_gmres_cgs_", 0) == 0) u = u.substr(14);  // PETSc also accepts the enum's C name
      // refine_ifneeded runs the second pass always (no estimate of the cancellation is made)
      if (u == "refine_never") o.cgs2 = false;
      else if (u == "refine_ifneeded" || u == "refine_always") o.cgs2 = true;
      else throw B2Error(-5, "unsupported ksp_gmres_cgs_refinement_type " + v + " (refine_never | refine_ifneeded | refine_always)");
    } else if (k == "ksp_rtol") o.rtol = std::stod(v);
    else if (k == "ksp_atol") o.atol = std::stod(v);
    else if (k == "ksp_max_it") o.maxit = std::stoi(v);
    else if (k == "ksp_chebyshev_eigenvalues") {  // "lo,hi" of D^-1 A (PETSc: -ksp_chebyshev_eigenvalues)
      const size_t comma = v.find(',');
      B2_REQUIRE(comma != std::string::npos, "ksp_chebyshev_eigenvalues expects lo,hi");
      o.eig_lo = std::stod(v.substr(0, comma));
      o.eig_hi = std::stod(v.substr(comma + 1));
    } else if (k == "ksp_initial_guess_nonzero") o.nonzero_guess = (v == "1" || v == "true" || v == "True");
    else if (k == "b200_block_rtol") o.block_rtol = (v == "1" || v == "true" || v == "True");
    else if (k == "b200_guess") {
      B2_REQUIRE(v == "extrapolate" || v == "extrapolate2" || v == "none" || v == "", "b200_guess: none | extrapolate | extrapolate2");
      o.extrapolate_guess = (v == "extrapolate" || v == "extrapolate2");
      o.guess_order = v == "extrapolate2" ? 2 : 1;
      if (o.extrapolate_guess) o.nonzero_guess = true;
    }
    // anything else: ignored (PETSc leaves unused options in the database without error)
  });
}

int b2_assemble_first(b2_ctx* c, double dt, double nu) {
  return guarded(c, [&] { stage_assemble_first(c, dt, nu); });
}
int b2_tentative_assemble(b2_ctx* c) {
  return guarded(c, [&] { stage_tentative_assemble(c); });
}
int b2_tentative_solve(b2_ctx* c, double* diff, int32_t* reasons) {
  return guarded(c, [&] { stage_tentative_solve(c, diff, reasons); });
}
int b2_pressure_assemble(b2_ctx* c, double dt) {
  return guarded(c, [&] { stage_pressure_assemble(c, dt); });
}
int b2_pressure_solve(b2_ctx* c, double nu, int32_t* reason) {
  return guarded(c, [&] { stage_pressure_solve(c, nu, reason); });
}
int b2_velocity_update(b2_ctx* c, double dt, int32_t* reasons) {
  return guarded(c, [&] { stage_velocity_update(c, dt, reasons); });
}
int b2_step_begin(b2_ctx* c, double dt, double nu) {
  return guarded(c, [&] { stage_step_begin(c, dt, nu); });
}
int b2_step(b2_ctx* c, double dt, double nu, double max_error, int max_iter, double* diff) {
  return guarded(c, [&] { stage_step(c, dt, nu, max_error, max_iter, diff); });
}

int b2_assemble_pressure_surface(b2_ctx* c, int64_t n_facets, const int32_t* facet_cells, const int32_t* facet_local,
                                 const double* h_nodal, int accumulate) {
  return guarded(c, [&] {
    require_ready(c);
    const Space &V = c->sp[B2_SPACE_V], &Q = c->sp[B2_SPACE_Q];
    if (!c->vecs.count(B2_VEC_PSURF)) alloc_vec(c, B2_VEC_PSURF, B2_SPACE_V, c->gdim);
    double* ps = c->vec(B2_VEC_PSURF);
    if (!accumulate) B2_CUDA(cudaMemsetAsync(ps, 0, sizeof(double) * V.n_local() * c->gdim, c->stream));
    if (n_facets > 0) {
      DBuf<int> fc, fl;
      DBuf<double> h;
      fc.alloc(n_facets);
      fl.alloc(n_facets);
      h.alloc(Q.n_local());
      B2_CUDA(cudaMemcpyAsync(fc.p, facet_cells, sizeof(int) * n_facets, cudaMemcpyHostToDevice, c->stream));
      B2_CUDA(cudaMemcpyAsync(fl.p, facet_local, sizeof(int) * n_facets, cudaMemcpyHostToDevice, c->stream));
      B2_CUDA(cudaMemcpyAsync(h.p, h_nodal, sizeof(double) * Q.n_local(), cudaMemcpyHostToDevice, c->stream));
      dispatch_elem(c, [&](auto e) {
        using E = decltype(e);
        B2_LAUNCH(c, (k_pressure_surface<E::D, E::DEG>), blocks_for(n_facets, 128), 128, n_facets, fc.p, fl.p, c->x.p,
                  c->cell_nodes.p, V.cell_dofs.p, Q.cell_dofs.p, (int)V.n_owned, (int)V.n_local(), h.p, ps);
      });
      B2_CUDA(cudaStreamSynchronize(c->stream));
      c->stats.bytes_h2d += sizeof(int) * 2 * n_facets + sizeof(double) * Q.n_local();
    }
  });
}

}  // extern "C"

namespace {

// the Q mass matrix is assembled with rotational=1; a Projector or KSPSolver may ask for it later
void ensure_mq(b2_ctx* c) {
  if (c->MQ.p != nullptr) return;
  const Space& Q = c->sp[B2_SPACE_Q];
  const CSR& qq = c->pat[B2_PAT_QQ];
  c->MQ.alloc(qq.slots);
  c->MQ.zero(c->stream);
  dispatch_elem(c, [&](auto e) {
    using E = decltype(e);
    B2_LAUNCH(c, (k_assemble_square<E::D, E::DEG, B2_FORM_MASS_Q>), blocks_for(c->n_cells * E::NQ, 128), 128, c->n_cells, c->x.p,
              c->cell_nodes.p, Q.cell_dofs.p, qq.n_rows, qq.rowptr.p, qq.cols.p, qq.slice_ptr.p, c->MQ.p);
  });
  c->dinvMQ.alloc(Q.n_local());
  B2_LAUNCH(c, k_inv_diag, blocks_for(qq.n_rows, 256), 256, qq.n_rows, qq.slice_ptr.p, qq.diag_t.p, c->MQ.p, c->dinvMQ.p);
}

// work vectors of a K-component Krylov solve outside the step (Projector, KSPSolver.solve): five of K * n_local
void ensure_proj_work(b2_ctx* c, int64_t n) {
  for (auto& w : c->wproj)
    if (w.n < n) { w.alloc(n); w.zero(c->stream); }
}

}  // namespace

extern "C" {

int b2_project_assemble(b2_ctx* c, int target_space, int n_comp, int src_space, const double* src_nodal, int deriv, int grad,
                        int n_q, const double* ref_points, const double* weights, const double* f_quad) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE(target_space == B2_SPACE_V || target_space == B2_SPACE_Q, "bad target space");
    B2_REQUIRE(n_comp >= 1 && n_comp <= 3 && n_q > 0, "1..3 components, at least one quadrature point");
    B2_REQUIRE((src_nodal != nullptr) != (f_quad != nullptr), "give either nodal source values or values at the quadrature points");
    B2_REQUIRE(!grad || (n_comp == c->gdim && src_nodal != nullptr), "grad: gdim components from one scalar nodal source");
    B2_REQUIRE(deriv < c->gdim, "bad derivative direction");
    const int d = c->gdim;
    const Space& T = c->sp[target_space];
    const int64_t ldt = T.n_local();
    c->proj_rhs.alloc(ldt * n_comp);
    c->proj_rhs.zero(c->stream);
    c->proj_space = target_space;
    c->proj_comp = n_comp;
    DBuf<double> dsrc, dfq, dp, dw;
    dp.alloc((int64_t)n_q * d);
    dw.alloc(n_q);
    B2_CUDA(cudaMemcpyAsync(dp.p, ref_points, sizeof(double) * n_q * d, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dw.p, weights, sizeof(double) * n_q, cudaMemcpyHostToDevice, c->stream));
    int64_t lds = 0;
    const Space* S = &T;
    if (src_nodal != nullptr) {
      B2_REQUIRE(src_space == B2_SPACE_V || src_space == B2_SPACE_Q, "bad source space");
      S = &c->sp[src_space];
      lds = S->n_local();
      const int ncs = grad ? 1 : n_comp;
      dsrc.alloc(lds * ncs);
      B2_CUDA(cudaMemcpyAsync(dsrc.p, src_nodal, sizeof(double) * lds * ncs, cudaMemcpyHostToDevice, c->stream));
      c->stats.bytes_h2d += sizeof(double) * lds * ncs;
    } else {
      dfq.alloc(c->n_cells * n_q * n_comp);
      B2_CUDA(cudaMemcpyAsync(dfq.p, f_quad, sizeof(double) * c->n_cells * n_q * n_comp, cudaMemcpyHostToDevice, c->stream));
      c->stats.bytes_h2d += sizeof(double) * c->n_cells * n_q * n_comp;
    }
    const int grid = blocks_for(c->n_cells, 128);
    auto launch = [&](auto kern) {
      B2_LAUNCH(c, kern, grid, 128, c->n_cells, c->x.p, c->cell_nodes.p, T.cell_dofs.p, (int)T.n_owned, (int)ldt, S->cell_dofs.p,
                (int)lds, (const double*)dsrc.p, (const double*)dfq.p, n_comp, deriv, grad, n_q, (const double*)dp.p,
                (const double*)dw.p, c->proj_rhs.p);
    };
    const int td = T.degree, sd = S->degree;
    if (d == 2 && td == 1 && sd == 1) launch(k_project_rhs<2, 1, 1>);
    else if (d == 2 && td == 1 && sd == 2) launch(k_project_rhs<2, 1, 2>);
    else if (d == 2 && td == 2 && sd == 1) launch(k_project_rhs<2, 2, 1>);
    else if (d == 2 && td == 2 && sd == 2) launch(k_project_rhs<2, 2, 2>);
    else if (d == 3 && td == 1 && sd == 1) launch(k_project_rhs<3, 1, 1>);
    else if (d == 3 && td == 1 && sd == 2) launch(k_project_rhs<3, 1, 2>);
    else if (d == 3 && td == 2 && sd == 1) launch(k_project_rhs<3, 2, 1>);
    else launch(k_project_rhs<3, 2, 2>);
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_project_set_rhs(b2_ctx* c, int target_space, int n_comp, const double* rhs) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE((target_space == B2_SPACE_V || target_space == B2_SPACE_Q) && n_comp >= 1 && n_comp <= 3, "bad space / components");
    const int64_t n = c->sp[target_space].n_local() * n_comp;
    c->proj_rhs.alloc(n);
    c->proj_space = target_space;
    c->proj_comp = n_comp;
    B2_CUDA(cudaMemcpyAsync(c->proj_rhs.p, rhs, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(double) * n;
  });
}

/* Dirichlet conditions of the projection (function.py:70 assemble_matrix(bcs=), :114-118 apply_lifting + set_bc):
 * x_k[dofs[i]] = values[k][i]; n = 0 removes them.  Applied by b2_project_solve to whatever right-hand side is loaded. */
int b2_project_set_bcs(b2_ctx* c, int target_space, int n_comp, int64_t n, const int32_t* dofs, const double* values) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE((target_space == B2_SPACE_V || target_space == B2_SPACE_Q) && n_comp >= 1 && n_comp <= 3 && n >= 0, "bad space / components");
    auto& B = c->proj_bc[target_space];
    B.n_comp = n > 0 ? n_comp : 0;
    B.dofs.alloc(n);
    B.vals.alloc(n * n_comp);
    if (n == 0) return;
    const bool onV = target_space == B2_SPACE_V;
    if (!onV) ensure_mq(c);
    const CSR& pat = c->pat[onV ? B2_PAT_VV : B2_PAT_QQ];
    const int64_t nl = c->sp[target_space].n_local();
    B2_CUDA(cudaMemcpyAsync(B.dofs.p, dofs, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(B.vals.p, values, sizeof(double) * n * n_comp, cudaMemcpyHostToDevice, c->stream));
    B.mask.alloc(nl);
    B.mask.zero(c->stream);
    B2_LAUNCH(c, k_mark, blocks_for(n, 256), 256, n, B.dofs.p, B.mask.p);
    B.Mbc.alloc(pat.slots);
    B2_CUDA(cudaMemcpyAsync(B.Mbc.p, onV ? c->M.p : c->MQ.p, sizeof(double) * (size_t)pat.slots, cudaMemcpyDeviceToDevice, c->stream));
    B2_LAUNCH(c, k_apply_bc_rows_cols, blocks_for(pat.n_rows, 256), 256, pat.n_rows, pat.slice_ptr.p, pat.scols.p, pat.diag_t.p, B.mask.p, B.Mbc.p);
    B.dinv.alloc(nl);
    B2_LAUNCH(c, k_fill, pgrid(c, nl), 256, nl, 1.0, B.dinv.p);
    B2_LAUNCH(c, k_inv_diag, blocks_for(pat.n_rows, 256), 256, pat.n_rows, pat.slice_ptr.p, pat.diag_t.p, B.Mbc.p, B.dinv.p);
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_project_get_rhs(b2_ctx* c, double* rhs) {
  return guarded(c, [&] {
    B2_REQUIRE(c->proj_rhs.p != nullptr, "b2_project_assemble first");
    B2_CUDA(cudaMemcpyAsync(rhs, c->proj_rhs.p, sizeof(double) * c->proj_rhs.n, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int b2_project_solve(b2_ctx* c, double* x, int32_t* reasons) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE(c->proj_rhs.p != nullptr, "b2_project_assemble first");
    const int sp = c->proj_space, K = c->proj_comp;
    const Space& T = c->sp[sp];
    const int64_t n = T.n_local() * K;
    const bool onV = sp == B2_SPACE_V;
    if (!onV) ensure_mq(c);
    ensure_proj_work(c, n);
    DBuf<double> sol;
    sol.alloc(n);
    sol.zero(c->stream);
    int32_t its[B2_MAXK] = {0, 0, 0};
    KSPOpts& o = c->ksp[B2_SOLVER_PROJECTOR];
    const bool guess = o.nonzero_guess;
    o.nonzero_guess = false;
    const CSR& ppat = c->pat[onV ? B2_PAT_VV : B2_PAT_QQ];
    const double* Mv = onV ? c->M.p : c->MQ.p;
    const double* dinv = onV ? c->dinvM.p : c->dinvMQ.p;
    auto& B = c->proj_bc[sp];
    DBuf<double> rhs_bc, gext;
    const double* rhs = c->proj_rhs.p;
    if (B.n_comp > 0) {
      // lifting: b -= M g (g extended by zero), then b[dofs] = g; solve with the identity on the Dirichlet rows/columns
      B2_REQUIRE(B.n_comp == K, "Projector BCs were set for a different number of components");
      const int64_t nl = T.n_local(), nb = B.dofs.n;
      gext.alloc(n);
      gext.zero(c->stream);
      rhs_bc.alloc(n);
      for (int k = 0; k < K; ++k)
        B2_LAUNCH(c, k_set_bc, blocks_for(nb, 256), 256, nb, B.dofs.p, B.vals.p + (size_t)k * nb, gext.p + (size_t)k * nl);
      spmm(c, ppat, Mv, K, gext.p, rhs_bc.p, nullptr, nullptr, FIN_NONE, 0, sp);
      B2_LAUNCH(c, k_lincomb2, pgrid(c, n), 256, n, 1.0, c->proj_rhs.p, -1.0, rhs_bc.p, rhs_bc.p);
      for (int k = 0; k < K; ++k)
        B2_LAUNCH(c, k_set_bc, blocks_for(nb, 256), 256, nb, B.dofs.p, B.vals.p + (size_t)k * nb, rhs_bc.p + (size_t)k * nl);
      rhs = rhs_bc.p;
      Mv = B.Mbc.p;
      dinv = B.dinv.p;
    }
    krylov_solve(c, B2_SOLVER_PROJECTOR, ppat, Mv, dinv, sp, K, rhs, sol.p, reasons, its, c->wproj);
    o.nonzero_guess = guess;
    c->stats.its_projector = *std::max_element(its, its + K);
    halo_forward(c, sp, sol.p, K);  // x.scatter_forward(), function.py:132
    B2_CUDA(cudaMemcpyAsync(x, sol.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_d2h += sizeof(double) * n;
  });
}

/* KSPSolver.solve (ksp.py:71-78): solve  Mat x = b  with the options of solver slot `solver`; x holds the initial
 * guess on entry when ksp_initial_guess_nonzero is set. */
int b2_ksp_solve(b2_ctx* c, int solver, int mat, const double* b, double* x, int32_t* reason) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE(solver >= 0 && solver < 4, "bad solver id");
    B2_REQUIRE(mat == B2_MAT_M || mat == B2_MAT_K || mat == B2_MAT_A || mat == B2_MAT_AP || mat == B2_MAT_MQ, "square operators only");
    if (mat == B2_MAT_MQ) ensure_mq(c);
    const CSR* pat = nullptr;
    Layout layout;
    const DBuf<double>* v = matrix_values(c, mat, &pat, &layout);
    const int sp =(mat == B2_MAT_AP || mat == B2_MAT_MQ) ? B2_SPACE_Q : B2_SPACE_V;
    const int64_t n = c->sp[sp].n_local();
    ensure_proj_work(c, n);
    DBuf<double> db, dx, dinv;
    db.alloc(n);
    dx.alloc(n);
    dinv.alloc(n);
    B2_CUDA(cudaMemcpyAsync(db.p, b, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    B2_LAUNCH(c, k_fill, pgrid(c, n), 256, n, 1.0, dinv.p);
    B2_LAUNCH(c, k_inv_diag, blocks_for(pat->n_rows, 256), 256, pat->n_rows, pat->slice_ptr.p, pat->diag_t.p, v->p, dinv.p);
    int32_t its = 0;
    if (mat == B2_MAT_AP && c->ksp[solver].pc == 2 && !c->mg.empty() && !c->has_pbc && solver == B2_SOLVER_PRESSURE) {
      B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_B2), db.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
      B2_CUDA(cudaMemcpyAsync(c->vec(B2_VEC_DP), dx.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
      pcg_mg_solve(c, c->vec(B2_VEC_B2), c->vec(B2_VEC_DP), reason, &its);
      B2_CUDA(cudaMemcpyAsync(dx.p, c->vec(B2_VEC_DP), sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
    } else {
      krylov_solve(c, solver, *pat, v->p, dinv.p, sp, 1, db.p, dx.p, reason, &its, c->wproj);
    }
    if (solver == B2_SOLVER_PRESSURE) c->stats.its_pressure = its;
    halo_forward(c, sp, dx.p, 1);  // x.x.scatter_forward(), ksp.py:77
    B2_CUDA(cudaMemcpyAsync(x, dx.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    c->stats.bytes_h2d += sizeof(double) * 2 * n;
    c->stats.bytes_d2h += sizeof(double) * n;
  });
}

int b2_l2_diff_sq(b2_ctx* c, int vec, const double* exact, int64_t n, double* out) {
  return guarded(c, [&] {
    require_ready(c);
    auto it = c->vecs.find(vec);
    B2_REQUIRE(it != c->vecs.end(), "unknown vector id");
    DVec& v = it->second;
    const Space& S = c->sp[v.space];
    const int64_t nl = S.n_local();
    B2_REQUIRE(n == nl * v.K, "size mismatch in b2_l2_diff_sq");
    // e = u_h - exact (nodal, blocked [n][K] on the host); ||e||^2 = sum_k e_k^T M e_k
    B2_REQUIRE(v.space == B2_SPACE_V, "b2_l2_diff_sq: only velocity-space vectors in this version");
    double* e = c->wv[0].p;
    double* me = c->wv[1].p;
    B2_CUDA(cudaMemcpyAsync(c->stage.p, exact, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    B2_LAUNCH(c, k_from_blocked, pgrid(c, n), 256, nl, v.K, (int)nl, c->stage.p, e);
    B2_LAUNCH(c, k_lincomb2, pgrid(c, n), 256, n, 1.0, v.buf.p, -1.0, e, e);
    spmm(c, c->pat[B2_PAT_VV], c->M.p, v.K, e, me, nullptr, nullptr, FIN_NONE, 0, B2_SPACE_V);
    B2_LAUNCH(c, k_dot_all, pgrid(c, S.n_owned), 256, S.n_owned, v.K, (int)nl, me, e, c->d_sums, c->partials.p, c->d_counter);
    allreduce_sum(c, c->d_sums, 1);
    read_sums(c, 1);
    *out = c->h_sums[0];
  });
}

int b2_l2_error_quadrature(b2_ctx* c, int vec, int64_t n_cells, int n_q, const double* ref_points, const double* weights,
                           const double* exact, double* out) {
  return guarded(c, [&] {
    require_ready(c);
    auto it = c->vecs.find(vec);
    B2_REQUIRE(it != c->vecs.end(), "unknown vector id");
    DVec& v = it->second;
    const Space& S = c->sp[v.space];
    B2_REQUIRE(n_cells >= 0 && n_cells <= c->n_cells && n_q > 0, "bad cell / point count");
    halo_forward(c, v.space, v.buf.p, v.K);
    const int d = c->gdim;
    DBuf<double> dp, dw, dex;
    dp.alloc((int64_t)n_q * d);
    dw.alloc(n_q);
    dex.alloc(n_cells * n_q * v.K);
    B2_CUDA(cudaMemcpyAsync(dp.p, ref_points, sizeof(double) * n_q * d, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dw.p, weights, sizeof(double) * n_q, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dex.p, exact, sizeof(double) * n_cells * n_q * v.K, cudaMemcpyHostToDevice, c->stream));
    c->stats.bytes_h2d += sizeof(double) * n_cells * n_q * v.K;
    const int grid = pgrid(c, n_cells, 128, 8);
    dispatch_elem(c, [&](auto e) {
      using E = decltype(e);
      if (v.space == B2_SPACE_V)
        B2_LAUNCH(c, (k_l2_error<E::D, E::DEG, true>), grid, 128, n_cells, c->x.p, c->cell_nodes.p, S.cell_dofs.p, v.K,
                  (int)S.n_local(), v.buf.p, n_q, dp.p, dw.p, dex.p, c->d_sums, c->partials.p, c->d_counter);
      else
        B2_LAUNCH(c, (k_l2_error<E::D, E::DEG, false>), grid, 128, n_cells, c->x.p, c->cell_nodes.p, S.cell_dofs.p, v.K,
                  (int)S.n_local(), v.buf.p, n_q, dp.p, dw.p, dex.p, c->d_sums, c->partials.p, c->d_counter);
    });
    allreduce_sum(c, c->d_sums, 1);
    read_sums(c, 1);
    *out = c->h_sums[0];
  });
}

// demo/assembly_strategies.py:56-152 on the device: the tentative-velocity right-hand side of the current U1 / UAB
// vectors by the matrix-vector strategy (into RHS1) and by the action strategy (into BFIRST), each timed over `reps`
// launches with CUDA events.  out[0..6] = ms convection assembly (untimed in the reference), ms matvec, ms action,
// algorithmic bytes of the three, in the same order.
int b2_bench_assembly_strategies(b2_ctx* c, double dt, double nu, int reps, double* out) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE(reps > 0, "reps must be positive");
    const int K = c->gdim;
    const Space& V = c->sp[B2_SPACE_V];
    const CSR& vv = c->pat[B2_PAT_VV];
    const int ld = (int)V.n_local();
    double *u1 = c->vec(B2_VEC_U1), *uab = c->vec(B2_VEC_UAB);
    halo_forward(c, B2_SPACE_V, u1, K);
    halo_forward(c, B2_SPACE_V, uab, K);
    DBuf<double> zero;
    zero.alloc((int64_t)ld * K);
    zero.zero(c->stream);
    cudaEvent_t e[2];
    for (auto& ev : e) B2_CUDA(cudaEventCreate(&ev));
    auto timed = [&](auto&& body) {
      body();  // warm-up
      B2_CUDA(cudaEventRecord(e[0], c->stream));
      for (int i = 0; i < reps; ++i) body();
      B2_CUDA(cudaEventRecord(e[1], c->stream));
      B2_CUDA(cudaEventSynchronize(e[1]));
      float ms = 0;
      B2_CUDA(cudaEventElapsedTime(&ms, e[0], e[1]));
      return (double)ms / reps;
    };
    const double inf = 1.0 / 0.0;
    // 1/2 C(uab) into A (1/dt = nu = 0): the matrix the reference assembles outside its timed block
    out[0] = timed([&] { first_cells(c, 1, inf, 0.0, u1, uab, zero.p, nullptr, c->A.p, c->vec(B2_VEC_BFIRST), c->dinvA.p); });
    const int grid = pgrid(c, vv.n_rows, 256, 4);
    out[1] = timed([&] {
      if (K == 2) B2_LAUNCH(c, (k_matvec_rhs<2, 8>), grid, 256, vv.n_rows, vv.slice_ptr.p, vv.scols.p, c->A.p, c->M.p, c->Kst.p, vv.order.p, 1.0 / dt, 0.5 * nu, u1, ld, (const double*)nullptr, c->vec(B2_VEC_RHS1));
      else B2_LAUNCH(c, (k_matvec_rhs<3, 8>), grid, 256, vv.n_rows, vv.slice_ptr.p, vv.scols.p, c->A.p, c->M.p, c->Kst.p, vv.order.p, 1.0 / dt, 0.5 * nu, u1, ld, (const double*)nullptr, c->vec(B2_VEC_RHS1));
    });
    out[2] = timed([&] { first_cells(c, 2, dt, nu, u1, uab, zero.p, nullptr, c->A.p, c->vec(B2_VEC_BFIRST), c->dinvA.p); });
    const double nV = (double)V.n_owned, nVc = (double)vv.n_cols, cells = (double)c->n_cells;
    const double nvp = (V.nd + 3) / 4 * 4;
    const double cell_bytes = 4.0 * (V.nd + c->gdim + 1);  // dofs + vertices: SURVEY.md 8(d) "cells * 56" for P2 tetrahedra
    out[3] = 24.0 * vv.nnz + cells * (cell_bytes + V.nd * nvp) + 8.0 * 3 * c->n_nodes + 8.0 * K * nVc;
    out[4] = 28.0 * vv.nnz + 4.0 * (nV + 1) + 8.0 * K * (nV + nVc);
    out[5] = cells * cell_bytes + 8.0 * 3 * c->n_nodes + 8.0 * K * (2 * nVc + nV);
    for (auto& ev : e) cudaEventDestroy(ev);
    c->cfg_version++;
  });
}

int b2_first_plan_info(b2_ctx* c, int64_t* out) {
  return guarded(c, [&] {
    out[0] = c->first.ready ? 1 : 0;
    out[1] = c->first.n_classes;
    out[2] = 1;  // slab thickness of the class interleaving, in reference lengths
    out[3] = c->n_cells;
  });
}

int b2_l2_error_trig(b2_ctx* c, int vec, int64_t n_cells, int n_q, const double* ref_points, const double* weights,
                     int n_terms, const double* terms, double* out) {
  return guarded(c, [&] {
    require_ready(c);
    auto it = c->vecs.find(vec);
    B2_REQUIRE(it != c->vecs.end(), "unknown vector id");
    DVec& v = it->second;
    const Space& S = c->sp[v.space];
    B2_REQUIRE(n_cells >= 0 && n_cells <= c->n_cells && n_q > 0 && n_terms >= 0, "bad cell / point / term count");
    halo_forward(c, v.space, v.buf.p, v.K);
    const int d = c->gdim;
    DBuf<double> dp, dw, dt;
    dp.alloc((int64_t)n_q * d);
    dw.alloc(n_q);
    dt.alloc(std::max(1, n_terms) * 12);
    B2_CUDA(cudaMemcpyAsync(dp.p, ref_points, sizeof(double) * n_q * d, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(dw.p, weights, sizeof(double) * n_q, cudaMemcpyHostToDevice, c->stream));
    if (n_terms) B2_CUDA(cudaMemcpyAsync(dt.p, terms, sizeof(double) * 12 * n_terms, cudaMemcpyHostToDevice, c->stream));
    c->stats.bytes_h2d += sizeof(double) * (12 * n_terms + n_q * (d + 1));
    const int grid = pgrid(c, n_cells, 128, 8);
    dispatch_elem(c, [&](auto e) {
      using E = decltype(e);
      if (v.space == B2_SPACE_V)
        B2_LAUNCH(c, (k_l2_error_trig<E::D, E::DEG, true>), grid, 128, n_cells, c->x.p, c->cell_nodes.p, S.cell_dofs.p, v.K,
                  (int)S.n_local(), v.buf.p, n_q, dp.p, dw.p, n_terms, dt.p, c->d_sums, c->partials.p, c->d_counter);
      else
        B2_LAUNCH(c, (k_l2_error_trig<E::D, E::DEG, false>), grid, 128, n_cells, c->x.p, c->cell_nodes.p, S.cell_dofs.p, v.K,
                  (int)S.n_local(), v.buf.p, n_q, dp.p, dw.p, n_terms, dt.p, c->d_sums, c->partials.p, c->d_counter);
    });
    allreduce_sum(c, c->d_sums, 1);
    read_sums(c, 1);
    *out = c->h_sums[0];
  });
}

int b2_get_stats(b2_ctx* c, b2_stats* out) {
  return guarded(c, [&] { *out = c->stats; });
}

int b2_synchronize(b2_ctx* c) {
  return guarded(c, [&] { B2_CUDA(cudaStreamSynchronize(c->stream)); });
}

int b2_set_tuning(b2_ctx* c, const char* key, int value) {
  return guarded(c, [&] {
    c->cfg_version++;
    std::string k(key);
    if (k == "mg_dense") c->mg_dense_on = value;
    else if (k == "first_order") {
      c->first_order = std::max(0, value);
      if (c->preassembled) build_first_plan(c);
    }
    else throw B2Error(-2, "unknown tuning key " + k);
  });
}

int b2_event_record(b2_ctx* c, int slot) {
  return guarded(c, [&] {
    B2_REQUIRE(slot >= 0 && slot < 8, "event slot out of range");
    B2_CUDA(cudaEventRecord(c->user_ev[slot], c->stream));
  });
}

int b2_event_elapsed_ms(b2_ctx* c, int a, int b, double* ms) {
  return guarded(c, [&] {
    B2_REQUIRE(a >= 0 && a < 8 && b >= 0 && b < 8, "event slot out of range");
    B2_CUDA(cudaEventSynchronize(c->user_ev[b]));
    float f = 0;
    B2_CUDA(cudaEventElapsedTime(&f, c->user_ev[a], c->user_ev[b]));
    *ms = f;
  });
}

int b2_bench_kernel(b2_ctx* c, int kernel, int reps, double* ms_per_launch, double* bytes_per_launch) {
  return guarded(c, [&] {
    require_ready(c);
    B2_REQUIRE(reps > 0, "reps must be positive");
    const int K = c->gdim;
    const CSR &vv = c->pat[B2_PAT_VV], &qq = c->pat[B2_PAT_QQ];
    const Space &V = c->sp[B2_SPACE_V];
    cudaEvent_t e0, e1;
    B2_CUDA(cudaEventCreate(&e0));
    B2_CUDA(cudaEventCreate(&e1));
    auto body = [&]() {
      switch (kernel) {
        case 0: spmm(c, vv, c->A.p, K, c->vec(B2_VEC_U), c->wv[2].p); break;
        case 3: spmm(c, vv, c->M.p, K, c->vec(B2_VEC_U), c->wv[2].p); break;
        case 4:  // with the fused dot products and the row scale of the BiCGStab products (state: a solve in progress that stores nothing)
        case 5:
          spmm(c, vv, c->M.p, K, c->vec(B2_VEC_U), c->wv[2].p, c->vec(B2_VEC_U1), c->d_st, FIN_STORE, kernel - 3, -1, c->dinvM.p);
          break;
        case 2: spmm(c, qq, c->Ap.p, 1, c->vec(B2_VEC_DP), c->wq[2].p); break;
        case 1: stage_assemble_first(c, c->last_dt > 0 ? c->last_dt : 0.005, 0.01); break;
        case 10: halo_forward(c, B2_SPACE_Q, c->vec(B2_VEC_DP), 1); break;          // latency of the collectives
        case 11: halo_forward(c, B2_SPACE_V, c->vec(B2_VEC_U), K); break;
        case 12: allreduce_sum(c, c->d_sums, 3); break;
        case 13:
          B2_REQUIRE(c->peer_on && c->pvs_ready, "vector-sum benchmark needs the peer path with a multigrid attached");
          B2_LAUNCH(c, k_peer_vecsum, std::min(PEER_GRID_MAX, blocks_for(c->mg[0].n, 1024)), 256, c->pvs, c->mg[0].b.p);
          break;
        default: throw B2Error(-2, "unknown bench kernel");
      }
    };
    if (kernel == 4 || kernel == 5) {
      std::memset(c->h_st, 0, sizeof(KryState));
      c->h_st->K = K;
      B2_CUDA(cudaMemcpyAsync(c->d_st, c->h_st, sizeof(KryState), cudaMemcpyHostToDevice, c->stream));
    }
    body();  // warm-up
    B2_CUDA(cudaEventRecord(e0, c->stream));
    for (int i = 0; i < reps; ++i) body();
    B2_CUDA(cudaEventRecord(e1, c->stream));
    B2_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    B2_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *ms_per_launch = ms / reps;
    double nV = (double)V.n_owned, nVc = (double)vv.n_cols;
    switch (kernel) {
      case 10: *bytes_per_launch = 8.0 * (c->halo[B2_SPACE_Q].send_off.empty() ? 0 : c->halo[B2_SPACE_Q].send_off.back()); break;
      case 11: *bytes_per_launch = 8.0 * K * (c->halo[B2_SPACE_V].send_off.empty() ? 0 : c->halo[B2_SPACE_V].send_off.back()); break;
      case 12: *bytes_per_launch = 24.0; break;
      case 13: *bytes_per_launch = 8.0 * (c->mg_hi - c->mg_lo) * (c->nranks - 1); break;
      case 0:
      case 4:
      case 5:
      case 3: *bytes_per_launch = 12.0 * vv.nnz + 4.0 * (nV + 1) + 8.0 * K * (nV + nVc); break;  // algorithmic: K (not KP) components
      case 2: *bytes_per_launch = 12.0 * qq.nnz + 4.0 * (qq.n_rows + 1) + 8.0 * (qq.n_rows + qq.n_cols); break;
      case 1: {  // k_first_cells: A written once (interface rows: zero-fill + read-modify-write on top), cell data
                 // (dofs, nodes, scatter table), coordinates, uab/u1 read, b0 read, b_first + dinv written, uab = 1.5 u1 - .5 u2
        const double nvp = (V.nd + 3) / 4 * 4;  // zero-fill (8 nnz) + read-modify-write of the reductions (16 nnz)
        *bytes_per_launch = 24.0 * vv.nnz + (double)c->n_cells * (4.0 * (V.nd + c->gdim + 1 + 1) + V.nd * nvp) +
                            8.0 * 3 * c->n_nodes + 8.0 * K * nVc * (2 + 3) + 8.0 * K * nV * 4 + 8.0 * nV;
        break;
      }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  });
}

}  // extern "C"
