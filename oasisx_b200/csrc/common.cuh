// common.cuh -- error handling, device buffers and reduction helpers shared by all kernels.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>

#define B2_MAXK 3  // at most 3 velocity components solved together

struct B2Error : std::runtime_error {
  int code;
  B2Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define B2_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      throw B2Error(-100, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                              ":" + std::to_string(__LINE__) + ")");                           \
  } while (0)

#define B2_REQUIRE(cond, msg)                      \
  do {                                             \
    if (!(cond)) throw B2Error(-1, std::string(msg)); \
  } while (0)

template <typename T>
struct DBuf {  // owning device buffer
  T* p = nullptr;
  int64_t n = 0;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DBuf& operator=(DBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  void alloc(int64_t count) {
    release();
    if (count > 0) B2_CUDA(cudaMalloc(&p, sizeof(T) * (size_t)count));
    n = count;
  }
  void zero(cudaStream_t s) {
    if (n) B2_CUDA(cudaMemsetAsync(p, 0, sizeof(T) * (size_t)n, s));
  }
};

// streaming loads for the matrix stream (values, columns): read-only path, do not allocate in L1, so that
// the lines of the gathered vector are what stays resident there
__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ int ld_stream(const int* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// SELL-32 slot of entry t of row `row` (the sliced-ELL layout: linalg.cuh, "storage")
__device__ __forceinline__ size_t sell_slot(const int* __restrict__ slice_ptr, int row, int t) {
  return (size_t)__ldg(slice_ptr + (row >> 5)) + ((size_t)t << 5) + (row & 31);
}

// ---- warp / block reductions ------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic grid-wide sum of N per-thread values.  Every block publishes its partial sums;
// the block that takes the last ticket re-reads all partials in a fixed order and returns true
// (in every thread of that block) with `total` valid in thread 0.  `counter` is reset for the
// next launch.  Requires blockDim.x to be a multiple of 32 and <= 1024.
template <int N>
__device__ __forceinline__ bool grid_reduce(double (&v)[N], double* __restrict__ partials,
                                            unsigned* __restrict__ counter, double (&total)[N]) {
  __shared__ double sm[N][32];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double s = warp_sum(v[i]);
    if (lane == 0) sm[i][warp] = s;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      double s = lane < nwarp ? sm[i][lane] : 0.0;
      s = warp_sum(s);
      if (lane == 0) partials[(size_t)blockIdx.x * N + i] = s;
    }
    if (lane == 0) {
      __threadfence();
      unsigned t = atomicAdd(counter, 1u);
      is_last = (t == gridDim.x - 1);
    }
  }
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
  double acc[N];
#pragma unroll
  for (int i = 0; i < N; ++i) acc[i] = 0.0;
  for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
#pragma unroll
    for (int i = 0; i < N; ++i) acc[i] += __ldcg(&partials[(size_t)b * N + i]);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double s = warp_sum(acc[i]);
    if (lane == 0) sm[i][warp] = s;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      double s = lane < nwarp ? sm[i][lane] : 0.0;
      s = warp_sum(s);
      total[i] = s;
    }
    if (lane == 0) *counter = 0u;
  }
  return true;
}

// ---- peer-memory communication between the ranks of one NVSwitch box -------------------------------
// Every rank owns one "arena" (cudaMalloc) that the other ranks map through CUDA IPC.  Collectives are done
// INSIDE the compute kernels by plain remote stores over NVLink; nothing waits across launches (a kernel only ever
// waits, inside its own launch, for the matching kernel of a peer, which does not depend on it), so the sequence is
// safe to capture into a CUDA graph and needs no NCCL call.  It replaces, per Krylov iteration, 2-3 ncclAllReduce of
// <= 9 doubles + 1-thread scalar kernels and 2-3 pack -> ncclSend/Recv -> unpack halo exchanges (SURVEY.md 5.8:
// "latency is everything").
//
// Wire format ("LL", as NCCL's low-latency protocol): a double travels as two 8-byte stores {low word, seq} and
// {high word, seq}; 8-byte stores are single-copy atomic, so a receiver that reads seq in both halves has the
// value -- no fence, no separate flag, one NVLink crossing per collective.  Buffers are double-buffered by the
// parity of the sequence number: a peer can be at most one collective ahead (its next one needs my next
// contribution, which I send only after consuming this one).
#define B2_MAXR 8        // ranks of one box
#define B2_RED_MAX 16    // doubles per fused scalar all-reduce
#define B2_PEER_TIMEOUT_NS 30000000000ull

struct __align__(16) LLSlot { unsigned lo, f0, hi, f1; };

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void ll_store(LLSlot* dst, double v, unsigned seq) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(dst), "r"((unsigned)b), "r"(seq) : "memory");
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"((char*)dst + 8), "r"((unsigned)(b >> 32)), "r"(seq) : "memory");
}
// spin until both halves carry `seq` (bounded by B2_PEER_TIMEOUT_NS of wall clock: a dead peer must not hang the GPU)
__device__ __forceinline__ double ll_load(const LLSlot* src, unsigned seq, unsigned long long* err) {
  unsigned lo, f0, hi, f1;
  unsigned long long t0 = 0;
  for (unsigned spin = 0;; ++spin) {
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(f0) : "l"(src) : "memory");
    asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(hi), "=r"(f1) : "l"((const char*)src + 8) : "memory");
    if (f0 == seq && f1 == seq) break;
    if ((spin & 255u) == 255u) {
      const unsigned long long now = global_timer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > B2_PEER_TIMEOUT_NS) {
        if (err != nullptr) atomicExch(err, 1ull);
        break;
      }
    }
  }
  return __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
}

struct PeerDev {
  int nranks, rank;
  unsigned long long* seq_red;        // local: number of scalar all-reduces done
  unsigned long long* err;            // local: set when a wait timed out (host checks after the step)
  LLSlot* slot_red;                   // local [2][B2_MAXR][B2_RED_MAX]
  LLSlot* peer_slot_red[B2_MAXR];     // the same array in each peer's arena
};

// Sum of `n` doubles over the ranks, called by ONE warp (all 32 lanes) of ONE block per rank; `v` is the local
// contribution in shared or global memory, the result overwrites it (every rank gets the same bits: summation in
// rank order).  Lane q sends to peer q; lane i then gathers entry i of every rank.
__device__ __forceinline__ void peer_allreduce_warp(const PeerDev* pr, double* v, int n) {
  const int lane = threadIdx.x & 31;
  const int R = pr->nranks, me = pr->rank;
  unsigned long long s = 0;
  if (lane == 0) s = *pr->seq_red + 1;
  s = __shfl_sync(0xffffffffu, s, 0);
  const unsigned seq = (unsigned)s;
  const size_t base = ((size_t)(s & 1ull) * B2_MAXR) * B2_RED_MAX;
  if (lane < R && lane != me) {
    LLSlot* dst = pr->peer_slot_red[lane] + base + (size_t)me * B2_RED_MAX;
    for (int i = 0; i < n; ++i) ll_store(dst + i, v[i], seq);
  }
  __syncwarp();
  double acc = 0.0;
  if (lane < n) {
    for (int q = 0; q < R; ++q)
      acc += (q == me) ? v[lane] : ll_load(pr->slot_red + base + (size_t)q * B2_RED_MAX + lane, seq, pr->err);
  }
  __syncwarp();
  if (lane < n) v[lane] = acc;
  __syncwarp();
  if (lane == 0) *pr->seq_red = s;
}

// halo plan of one space for the peer path (passed to the kernel by value)
struct PeerHalo {
  int n_neighbors, rank, n_owned;
  int nbr[B2_MAXR];                           // neighbour ranks
  long long send_off[B2_MAXR + 1], recv_off[B2_MAXR + 1];
  long long dst_off[B2_MAXR];                 // where my block starts in neighbour j's staging (in dofs)
  const int* send_idx;                        // local
  unsigned long long* seq;                    // local exchange counter of this space
  LLSlot* recv;                               // local staging [2][cap]
  long long cap;
  LLSlot* peer_recv[B2_MAXR];                 // by j: staging base of rank nbr[j]
  long long peer_cap[B2_MAXR];
  unsigned* counter;                          // local ticket counter (zero between launches)
  unsigned long long* err;
};

// Forward halo of K components in ONE kernel: my owned interface values go straight into the neighbours' staging
// buffers (remote LL stores over NVLink); their values are picked out of my staging as they arrive and written to my
// ghost slots.
__global__ void __launch_bounds__(256)
k_halo_peer(PeerHalo h, int K, int ld, double* __restrict__ v) {
  const unsigned long long s = *((volatile unsigned long long*)h.seq) + 1;
  const unsigned seq = (unsigned)s;
  const int par = (int)(s & 1ull);
  const long long ns = h.send_off[h.n_neighbors], nr = h.recv_off[h.n_neighbors];
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < ns * K; t += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(t / ns);
    const long long i = t - (long long)k * ns;
    int j = 0;
    while (j + 1 < h.n_neighbors && i >= h.send_off[j + 1]) ++j;
    const long long cnt = h.send_off[j + 1] - h.send_off[j];
    LLSlot* dst = h.peer_recv[j] + (size_t)par * h.peer_cap[j] + K * h.dst_off[j] + k * cnt + (i - h.send_off[j]);
    ll_store(dst, v[(size_t)k * ld + h.send_idx[i]], seq);
  }
  const LLSlot* src = h.recv + (size_t)par * h.cap;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nr * K; t += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(t / nr);
    const long long i = t - (long long)k * nr;
    int j = 0;
    while (j + 1 < h.n_neighbors && i >= h.recv_off[j + 1]) ++j;
    const long long cnt = h.recv_off[j + 1] - h.recv_off[j];
    v[(size_t)k * ld + h.n_owned + i] = ll_load(src + K * h.recv_off[j] + k * cnt + (i - h.recv_off[j]), seq, h.err);
  }
  // the exchange counter moves on once every block has read it (each block reads it before taking its ticket)
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(h.counter, 1u);
    if (t == gridDim.x - 1) {
      *h.counter = 0u;
      *h.seq = s;
    }
  }
}

// standalone scalar all-reduce (n <= B2_RED_MAX) of a device buffer: one warp
__global__ void k_peer_allreduce(const PeerDev* pr, double* v, int n) {
  __shared__ double sh[B2_RED_MAX];
  if (threadIdx.x < n) sh[threadIdx.x] = v[threadIdx.x];
  __syncwarp();
  peer_allreduce_warp(pr, sh, n);
  if (threadIdx.x < n) v[threadIdx.x] = sh[threadIdx.x];
}

// Sum over ranks of a replicated-level vector (the restricted multigrid right-hand side): every rank pushes the
// index range [lo, hi) its slab contributes to into every peer's staging and adds up, in rank order, the ranges
// that cover each entry as they arrive.
struct PeerVecSum {
  int nranks, rank, n;
  int lo[B2_MAXR], hi[B2_MAXR];
  unsigned long long* seq;
  LLSlot* stage;                             // local [2][nranks][n]
  LLSlot* peer_stage[B2_MAXR];
  unsigned* counter;
  unsigned long long* err;
};

__global__ void __launch_bounds__(256)
k_peer_vecsum(PeerVecSum h, double* __restrict__ v) {
  const unsigned long long s = *((volatile unsigned long long*)h.seq) + 1;
  const unsigned seq = (unsigned)s;
  const int par = (int)(s & 1ull);
  const int me = h.rank, lo = h.lo[me], hi = h.hi[me];
  const size_t mine = ((size_t)par * h.nranks + me) * h.n;
  for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
    const double x = v[i];
    for (int q = 0; q < h.nranks; ++q)
      if (q != me) ll_store(h.peer_stage[q] + mine + i, x, seq);
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h.n; i += gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int q = 0; q < h.nranks; ++q)
      if (i >= h.lo[q] && i < h.hi[q])  // my own partial is read in place; rank order kept
        acc += (q == me) ? v[i] : ll_load(h.stage + ((size_t)par * h.nranks + q) * h.n + i, seq, h.err);
    v[i] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(h.counter, 1u);
    if (t == gridDim.x - 1) {
      *h.counter = 0u;
      *h.seq = s;
    }
  }
}
