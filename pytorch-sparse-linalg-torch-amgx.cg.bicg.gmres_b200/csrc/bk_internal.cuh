// bk_internal.cuh — shared internals of libbk_krylov: handle, device state, deterministic
// reductions, pack loads.  sm_100a only (B200).  Not part of the public ABI (include/bk_krylov.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/bk_krylov.h"

#define BK_BLOCK 256          // threads per CTA of every persistent kernel
#define BK_WARPS (BK_BLOCK / 32)
#define BK_MAXB 2048          // upper bound on CTAs of a reducing grid (partials stride)
#define BK_NSLOT 4            // independent reduction scratch slots per handle
#define BK_SLOT_ROWS 8        // reductions per slot (fixed-R kernels use <= 8)

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
extern thread_local char bk_err_buf[512];
int bk_fail(int code, const char* fmt, ...);

#define BK_CUDA(expr)                                                                            \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return bk_fail(BK_ERR_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                  \
                     cudaGetErrorString(_e));                                                    \
  } while (0)

#define BK_TRY(expr)             \
  do {                           \
    int _r = (expr);             \
    if (_r != BK_OK) return _r;  \
  } while (0)

#define BK_KERNEL_CHECK() BK_CUDA(cudaGetLastError())

// ------------------------------------------------------------------------------------------
// device-resident solver state: every scalar of the recurrences lives here, written by the
// epilogue of the kernel that finishes the corresponding reduction, read by the next kernel.
// The host only ever reads it (async copy) to poll `done` and to build bk_result.
// ------------------------------------------------------------------------------------------
struct bk_dev_state {
  // loop control
  long long k;        // iterations (CG/BiCGStab) or restart cycles (GMRES) completed
  long long maxiter;
  long long matvecs;
  int done;           // 1 => every guarded kernel is an exact no-op
  int just_done;      // CG: `done` was set by THIS iteration's r-update, whose x/p-update kernel must still run once
  int status;         // enum bk_status
  int exit_early;     // BiCGStab: s.s < atol2 (:920)
  int parity;         // flips every iteration (sweep direction for the "snake" option)
  // tolerances
  double tol32;       // (double)(float)tol      — torch.tensor(tol) is fp32 (:816)
  double atol32;      // (double)(float)atol
  double tolsq32;     // (double)((float)tol*(float)tol)
  double atolsq32;
  double atol2;       // max(tol^2 * b.b, atol^2)  (:815-817, :870-872)
  double bs;          // b.b
  // CG
  double gamma, pAp, alpha, beta;
  double alpha_lag;   // CG, lagged-x cut: alpha of the previous (even) iteration, whose x += alpha p is still pending
  // BiCGStab
  double rho, omega, rho_new, rs, rhat_q, ss;
  // final check
  double rtrue2, xx;
  // GMRES (scalars; the small dense arrays live in bk_gmres_small)
  double g_atol, g_ptol, g_tol_eff, g_atol_eff;
  double g_bnorm, g_resnorm, g_vnorm0, g_err, g_scale;
  int g_kcur;         // Arnoldi steps taken in the current cycle
  int g_cycle_over;   // 1 => remaining Arnoldi kernels of this cycle are no-ops
  int g_use;          // normalisation flag of the last safe_normalize
  int g_method;
  int g_restart;
  int pad0;
};

struct bk_scratch {
  double* partials;       // [rows][stride]
  unsigned int* counter;  // self-resetting ticket (atomicInc wraps at gridDim.x-1)
  int stride;
};

// ------------------------------------------------------------------------------------------
// matrix object
// ------------------------------------------------------------------------------------------
struct bk_csr {
  bk_handle* h;
  int64_t n, nnz;
  int dtype;
  const int* rowptr;  // int32, device
  const int* col;     // int32, device
  const void* val;    // dtype, device
  void* own_rowptr;   // non-null when the library owns (converted / copied) arrays
  void* own_col;
  void* own_val;
  int kernel;         // 0 row-stream (LDG staged), 1 sub-warp vector, 2 row-stream with TMA-staged tiles, 3 = 2 + 8-bit column
                      // codes, 4 long rows split into virtual rows, 5 = 2 with 8-bit (offset, value) pair codes
  int lanes_per_row;
  int cap;            // row-stream: shared-memory products per warp
  int tma_cap;        // TMA row-stream: entries per pipeline stage (multiple of 4)
  int tma_stages;     // TMA row-stream: pipeline depth
  void* tail_val;     // TMA row-stream: the last nnz%4 entries, zero-padded to 4 (own)
  int* tail_col;
  // compressed index stream (kernel 3): 8-bit codes into per-block dictionaries of (column - row) offsets
  unsigned char* codes;      // nnz (+ padding) bytes, own
  int* dict;                 // nblk * 32 offsets, own
  void* tail_val16;          // last nnz%16 entries zero-padded to 16 (own)
  unsigned char* tail_code16;
  int cmp_cap;               // entries per stage for the compressed variant
  // pair-coded stream (kernel 5, bk_spmv_pair.cuh): 8-bit codes into per-block dictionaries of (column - row, value)
  // pairs, stored SELL-32-4; the SpMV reads neither val, col nor rowptr
  unsigned char* pcodes;     // code stream, own
  void* pdict;               // nblk * 32 bk_pair_entry (16 B each), own
  int* pbptr;                // [n/256 + 1] byte offset of every 256-row block span in pcodes, own
  int pair_cap;              // code bytes per pipeline stage
  // row-bitmask stream (kernel 6, bk_spmv_mask.cuh): one presence byte per row over its 32-row chunk's pattern of
  // (column - row, value) pairs, one pattern-table slot per chunk
  unsigned char* mmasks;     // [nchunks * 32], own
  int* mpids;                // [nchunks], own
  void* mptab;               // BK_MASK_HT * 8 bk_pair_entry, own
  int* mdeferred;            // multi-GPU: chunks with ghost entries (processed after the halo arrived), own
  int n_mdeferred;
  int mask_patterns;         // distinct patterns in the table
  // kernel 7 (two rows per lane, patterns as kernel parameters): tile summaries + the host copy of the parameter block
  unsigned short* musum;     // [n / 64, whole groups] step summaries of kernel 7 (nullptr: fp32 / no common offset set / ghosts), own
  unsigned char* mumasks;    // [nchunks * 32] presence bits in union numbering, own
  int mu_len, mu_odd;        // union entries, bit mask of the odd offsets
  int mu_center;             // 1: the union holds -1, 0, +1 at positions len/2 - 1, len/2, len/2 + 1
  int64_t mu_bytes;          // matrix-side bytes kernel 7 reads per SpMV
  unsigned char mctab[1024]; // bk_mask_utab
  int mw_win;                // kernel 6W: half-width W of the near window (0: no window plan)
  int mw_nfar;               // kernel 6W: far windows
  int mw_far[2];             // their offsets
  int64_t n_cols;            // columns (== n except for the extended local+ghost matrix of a row partition)
  const long long* reg_ghost_gid;  // registration only (n_cols > n): global ids of the ghost columns
  long long reg_row_begin;         // registration only: global id of row 0
  int64_t bytes_stream;      // actual matrix-side bytes the selected kernel reads per SpMV (bk_csr_info)
  int max_row_nnz;
  double mean_row_nnz;
  bk_csr* transpose;  // cached, owned
  bk_sgs* sgs;        // multicolor symmetric Gauss-Seidel set-up (bk_sgs_create), cached, owned
  // long-row splitting (skewed matrices): `split` views the same col/val arrays through a finer row pointer in which
  // every row longer than BK_SPLIT_LEN is cut into virtual rows; vstart[r] = first virtual row of real row r
  bk_csr* split;      // owned (its rowptr only)
  int* vstart;        // n+1, own
  void* yv;           // nv partial sums of the virtual rows, own
  int is_view;        // this object borrows col/val/tails from a parent (do not free them)
  uint64_t uid;       // unique id for graph-cache keys
};

// multicolor symmetric Gauss-Seidel (bk_sgs.cu): the coloring of A's pattern and its rows grouped by color.  The
// sweeps read rowptr / col / val of `A` at every application, so an in-place update of the values is picked up.
struct bk_sgs {
  const bk_csr* A;
  int ncolors, rounds;
  unsigned char* colors;  // [n], own
  int* rows;              // [n] rows sorted by color (stable: ascending within a color), own
  int* offs;              // host [ncolors + 1]: rows of color c are rows[offs[c] .. offs[c+1])
};
void bk_sgs_free(bk_sgs* S);
// z = M r: the forward sweep over colors 0..C-1, then the backward sweep over C-2..0 (2C-1 kernels).  Every kernel
// returns at once when bk_guard_skip(st, guard) holds.  r and z must not alias.
int bk_sgs_run(bk_handle* h, const bk_sgs* S, const void* r, void* z, int guard, cudaStream_t s);
static inline int bk_sgs_launches(const bk_sgs* S) { return 2 * S->ncolors - 1; }
// the checks every bk_*_sgs entry shares: S belongs to h and fits A_sys (order, dtype)
int bk_sgs_args_check(const char* who, bk_handle* h, const bk_csr* A, const bk_sgs* S);

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct bk_graph_entry {
  cudaGraphExec_t exec;
  uint64_t key[6];
  int valid;
};

struct bk_handle {
  int device;
  int num_sms;
  int64_t l2_bytes;
  int64_t mem_bytes;
  // options
  int grid_mult_vec;   // CTAs/SM of elementwise kernels
  int grid_mult_spmv;  // CTAs/SM of SpMV kernels
  int tma_ctas;        // CTAs/SM of the TMA row-stream SpMV (2..4)
  int pair_ctas;       // CTAs/SM of the pair-coded SpMV (2..6)
  int mask_ctas;       // CTAs/SM of the row-bitmask SpMV (kernel 6; 2..6)
  int mask_group;      // kernel 6: consecutive 256-row blocks dealt to a CTA at a time
  int mask_prefetch;   // kernel 6: L2 bulk prefetch of the x range of a CTA's next group
  int mask_window;     // kernel 6W: gathers from TMA-staged shared-memory windows of x (1) instead of LDG (0)
  int mask_wgroup;     // kernel 6W: consecutive 256-row blocks per stage
  int nvtx;            // emit NVTX ranges around the phases of every solve (BK_NVTX=1)
  int last_loop_mode;  // how the last iteration loop actually ran (bk_result.loop_mode_used)
  int dist_fuse_push;  // multi-GPU CG, peer path: fold the halo push into the kernel that produces p (1)
  int dist_fold;       // multi-GPU, peer path: ONE SpMV kernel over [local | ghost] (kernel 6) instead of local + boundary rows
  int tma_stages;      // 0 = fill shared memory, else cap on the pipeline depth
  int use_tma;         // allow the TMA row-stream kernel
  int prefetch_x;      // kernel 3: L2 bulk prefetch of the forward-diagonal x ranges
  int persistent;      // CG: run small systems in ONE cooperative persistent kernel (grid barriers instead of launches)
  int persistent_max_n;
  int persistent_cluster;  // persistent GMRES: run systems of <= 16384 rows as ONE thread-block cluster (hardware barrier)
  int use_split;       // split very long rows into virtual rows (skewed matrices)
  int use_compress;    // 0 off | 1 8-bit dictionary-coded column stream (kernel 3) | 2 also try (offset, value) pair codes (kernel 5)
  int dist_p2p;        // multi-GPU: use the peer-memory path (halo push + one-shot all-reduce) when it is connected
  int loop_mode;
  int chunk;
  int fuse_xpay;
  int snake;
  int mask_cctas;  // kernel 7: CTAs per SM (4..6)
  int mask2_prefetch;  // kernel 7: L2 bulk prefetch of the next group's x range (measured: no gain on 3-D stencils; off)
  int mask_const;  // kernel 7 (two rows per lane, patterns in the kernel's parameter block) when the matrix has <= 12 patterns
  int cg_lag_x;  // CG (3-kernel cut): x is updated every second iteration with both pending terms (9n instead of 10n per 2)
  int l2_hints;  // bit 0: K2 streams Ap | bit 1: K3 streams x | bit 2: K3 streams r | bit 3: SpMV streams masks
  // reduction scratch
  double* partials;        // BK_NSLOT * BK_SLOT_ROWS * BK_MAXB
  unsigned int* counters;  // BK_NSLOT (+ spare)
  // device state + pinned mirror
  bk_dev_state* st;        // device
  bk_dev_state* st_host;   // pinned, 4 entries (poll ring + final)
  // work vectors (elements of the largest dtype requested so far)
  void* ws;
  size_t ws_bytes;
  // GMRES small arrays (device)
  double* gm_small;
  size_t gm_small_bytes;
  double* gm_partials;     // (restart+1) x BK_MAXB partial sums for the multi-dot
  size_t gm_partials_bytes;
  // poll events
  cudaEvent_t ev[4];
  cudaEvent_t ev_t0, ev_t1;  // device time of a solve (bk_result.device_ms)
  unsigned long long* cksum; // device scratch of bk_checksum
  // graph cache
  bk_graph_entry graphs[8];
  cudaStream_t cap_stream;
  cudaStream_t io_stream;   // bk_solve_host: H2D / solve / D2H
  void* stage;              // bk_solve_host: cached device staging area
  size_t stage_bytes;
  uint64_t next_uid;
  // multi-GPU: the NCCL communicator is created once per handle and shared by every row-partitioned matrix
  // registered with the same (rank, nranks) — ncclCommInitRank costs 0.1-1 s (bk_dist.cu)
  void* dist_comm;
  int dist_comm_rank, dist_comm_nranks;
};

static inline bk_scratch bk_slot(bk_handle* h, int slot) {
  bk_scratch s;
  s.partials = h->partials + (size_t)slot * BK_SLOT_ROWS * BK_MAXB;
  s.counter = h->counters + slot;
  s.stride = BK_MAXB;
  return s;
}

// Matrix-side allocations (index copies, coded columns, tails, transposes) come from the device's stream-ordered
// memory pool (cudaMallocAsync) with the release threshold raised, so registering / dropping a matrix costs
// microseconds instead of the milliseconds cudaMalloc/cudaFree take for hundreds of megabytes.
cudaError_t bk_pool_alloc(void** p, size_t bytes, cudaStream_t s);
void bk_pool_free(void* p);
int bk_ws_reserve(bk_handle* h, size_t bytes);  // grows h->ws (invalidates cached graphs)
void bk_graphs_invalidate(bk_handle* h);
void bk_dist_release_comm(bk_handle* h);  // bk_dist.cu
void bk_state_fill_tol(bk_dev_state* v, double tol, double atol);
// bracket of every solver entry: NVTX range + start event | stop event (enqueue before the final stream sync) |
// after the sync: device_ms, loop_mode_used, NVTX pop
void bk_call_begin(bk_handle* h, cudaStream_t s, const char* name);
void bk_call_mark(bk_handle* h, const char* phase);  // NVTX only: closes the previous phase range, opens `phase`
void bk_call_stop(bk_handle* h, cudaStream_t s);
void bk_call_finish(bk_handle* h, bk_result* res);
void bk_fill_result_isolve(const bk_dev_state* st, bk_result* res, int64_t matvecs);
void bk_convert_i64_i32(bk_handle* h, const void* in, void* out, long long n, cudaStream_t s);
int bk_exclusive_scan_u32(unsigned int* data, long long n, cudaStream_t s);
int bk_sort_pairs_i32(bk_handle* h, int* k0, int* k1, int* v0, int* v1, long long n, int bits, cudaStream_t s,
                      int** ks, int** vs);
void bk_lower_bound_i32(bk_handle* h, const int* keys, long long count, long long n, int* out, cudaStream_t s);
void bk_iota_i32(bk_handle* h, int* out, long long n, cudaStream_t s);
#define BK_SPLIT_LEN 256
int bk_csr_finish_plan(bk_handle* h, bk_csr* A, cudaStream_t s);
int bk_csr_plan_mask(bk_handle* h, bk_csr* A, const long long* ghost_gid, long long row_begin, cudaStream_t s);
int bk_solver_args_check(const char* who, bk_handle* h, const bk_csr* A, const void* b, void* x, bk_result* res);

static inline int bk_grid_vec(const bk_handle* h) {
  int g = h->num_sms * h->grid_mult_vec;
  return g > BK_MAXB ? BK_MAXB : g;
}
static inline int bk_grid_spmv(const bk_handle* h) {
  int g = h->num_sms * h->grid_mult_spmv;
  return g > BK_MAXB ? BK_MAXB : g;
}
// Small problems: do not launch more CTAs than there is work for (cheaper launch, fewer partials in the final
// reduction).  Depends only on the problem size, so the summation order stays a function of (n, grid options).
static inline int bk_grid_vec_n(const bk_handle* h, long long n, int elems_per_thread) {
  const int g = bk_grid_vec(h);
  long long need = (n + (long long)BK_BLOCK * elems_per_thread - 1) / ((long long)BK_BLOCK * elems_per_thread);
  if (need < 1) need = 1;
  return need < g ? (int)need : g;
}
static inline int bk_grid_rows(int g, long long n, int rows_per_cta) {
  long long need = (n + rows_per_cta - 1) / rows_per_cta;
  if (need < 1) need = 1;
  return need < g ? (int)need : g;
}
static inline size_t bk_dtype_size(int dtype) { return dtype == BK_F32 ? 4 : 8; }
static inline bool bk_aligned16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// round-to-nearest mul/add that the compiler may NOT contract into an FMA: the reference
// evaluates x + alpha*p as two separately rounded torch ops (_add/_mul :165-173).
__device__ __forceinline__ double bk_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double bk_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double bk_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float bk_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float bk_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float bk_sub(float a, float b) { return __fsub_rn(a, b); }

template <typename T, int W>
struct bk_vec {
  T v[W];
};

template <typename T>
struct bk_native_w {
  static constexpr int value = 16 / sizeof(T);
};

// 16-byte vector load/store when W is the native pack width, scalar otherwise.
template <typename T, int W>
__device__ __forceinline__ bk_vec<T, W> bk_ld(const T* __restrict__ p) {
  bk_vec<T, W> r;
  if constexpr (W == 1) {
    r.v[0] = *p;
  } else if constexpr (sizeof(T) == 8) {
    static_assert(W == 2, "fp64 pack is 2 wide");
    double2 t = *reinterpret_cast<const double2*>(p);
    r.v[0] = t.x;
    r.v[1] = t.y;
  } else {
    static_assert(W == 4, "fp32 pack is 4 wide");
    float4 t = *reinterpret_cast<const float4*>(p);
    r.v[0] = t.x;
    r.v[1] = t.y;
    r.v[2] = t.z;
    r.v[3] = t.w;
  }
  return r;
}

template <typename T, int W>
__device__ __forceinline__ void bk_st(T* __restrict__ p, const bk_vec<T, W>& r) {
  if constexpr (W == 1) {
    *p = r.v[0];
  } else if constexpr (sizeof(T) == 8) {
    double2 t;
    t.x = r.v[0];
    t.y = r.v[1];
    *reinterpret_cast<double2*>(p) = t;
  } else {
    float4 t;
    t.x = r.v[0];
    t.y = r.v[1];
    t.z = r.v[2];
    t.w = r.v[3];
    *reinterpret_cast<float4*>(p) = t;
  }
}

// The same with the streaming ("evict first") cache operator: for operands that nobody reads again before the L2 has
// turned over, so that the vector the NEXT kernel of the iteration starts with keeps its place in the 126 MB L2.
template <typename T, int W>
__device__ __forceinline__ bk_vec<T, W> bk_ld_cs(const T* __restrict__ p) {
  bk_vec<T, W> r;
  if constexpr (W == 1) {
    r.v[0] = __ldcs(p);
  } else if constexpr (sizeof(T) == 8) {
    double2 t = __ldcs(reinterpret_cast<const double2*>(p));
    r.v[0] = t.x;
    r.v[1] = t.y;
  } else {
    float4 t = __ldcs(reinterpret_cast<const float4*>(p));
    r.v[0] = t.x;
    r.v[1] = t.y;
    r.v[2] = t.z;
    r.v[3] = t.w;
  }
  return r;
}

template <typename T, int W>
__device__ __forceinline__ void bk_st_cs(T* __restrict__ p, const bk_vec<T, W>& r) {
  if constexpr (W == 1) {
    __stcs(p, r.v[0]);
  } else if constexpr (sizeof(T) == 8) {
    double2 t;
    t.x = r.v[0];
    t.y = r.v[1];
    __stcs(reinterpret_cast<double2*>(p), t);
  } else {
    float4 t;
    t.x = r.v[0];
    t.y = r.v[1];
    t.z = r.v[2];
    t.w = r.v[3];
    __stcs(reinterpret_cast<float4*>(p), t);
  }
}

// ... and with an L2 "evict last" policy: the vector a kernel hands to the next kernel of the iteration.
__device__ __forceinline__ unsigned long long bk_policy_evict_last() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bk_st_hint1(double* p, double v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void bk_st_hint1(float* p, float v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
template <typename T, int W>
__device__ __forceinline__ void bk_st_keep(T* __restrict__ p, const bk_vec<T, W>& r, unsigned long long pol) {
  if constexpr (W == 1) {
    bk_st_hint1(p, r.v[0], pol);
  } else if constexpr (sizeof(T) == 8) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(r.v[0]), "d"(r.v[1]), "l"(pol)
                 : "memory");
  } else {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
                 "f"(r.v[2]), "f"(r.v[3]), "l"(pol)
                 : "memory");
  }
}

// Block-level sum of R values over NW warps; result valid in thread 0.  Fixed shuffle tree => the
// summation order depends only on (NW, R), never on scheduling.
template <int R, int NW = BK_WARPS>
__device__ __forceinline__ void bk_block_reduce(double (&v)[R], double* sh /* R*NW */) {
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
#pragma unroll
  for (int r = 0; r < R; ++r) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[r] += __shfl_down_sync(0xffffffffu, v[r], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < R; ++r) sh[r * NW + wid] = v[r];
  }
  __syncthreads();
  if (wid == 0) {
    constexpr int TOP = NW <= 2 ? 1 : (NW <= 4 ? 2 : (NW <= 8 ? 4 : (NW <= 16 ? 8 : 16)));
#pragma unroll
    for (int r = 0; r < R; ++r) {
      double t = (lane < NW) ? sh[r * NW + lane] : 0.0;
#pragma unroll
      for (int o = TOP; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
      v[r] = t;
    }
  }
  __syncthreads();
}

// Grid-level deterministic sum: every CTA parks its partial in slot [r][blockIdx.x]; the CTA
// that draws the last ticket adds the partials in index order with the same fixed tree and
// runs `epi(sums)` on its thread 0 (this is where alpha/beta/stop flags are computed, so no
// scalar kernels and no host round trip exist).  Bitwise reproducible for a fixed grid size.
template <int R, typename Epi, int NW = BK_WARPS>
__device__ __forceinline__ void bk_grid_reduce(double (&v)[R], const bk_scratch sc, Epi epi) {
  __shared__ double sh[R * NW];
  __shared__ int s_last;
  bk_block_reduce<R, NW>(v, sh);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int r = 0; r < R; ++r) __stcg(&sc.partials[(size_t)r * sc.stride + blockIdx.x], v[r]);
    __threadfence();
    const unsigned int t = atomicInc(sc.counter, gridDim.x - 1);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    double acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      double a = 0.0;
      for (int i = threadIdx.x; i < (int)gridDim.x; i += NW * 32)
        a += __ldcg(&sc.partials[(size_t)r * sc.stride + i]);
      acc[r] = a;
    }
    bk_block_reduce<R, NW>(acc, sh);
    if (threadIdx.x == 0) epi(acc);
  }
}

#endif  // __CUDACC__
