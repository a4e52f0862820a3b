// bk_gmres.cu — restarted GMRES with a device-resident restart cycle.
// Replaces gmres (reference torch_sparse_linalg.py:641-784), _gmres_solve_with_method (:788-803),
// _gmres_batched (:431-493), _gmres_incremental (:557-638), _kth_arnoldi_iteration (:331-388),
// _iterative_classical_gram_schmidt (:284-328), _givens_rotation (:508-518), _safe_normalize (:217-273).
//
// Layout: Krylov basis V stored vector-major, (restart+1) x ldv, each vector contiguous (the reference
// keeps N x (restart+1) with the basis index fastest and clones it every step, :363-368, :448-452).
//
// One Arnoldi step j (the reference's single classical Gram-Schmidt pass, SURVEY §8a-G3):
//   A1  w = A v_j              fused with ||w||^2        -> v_norm_0 (safe_normalize, thresh eps)   (:350-352)
//   A2  h_i = v_i . w, i<=j    tall-skinny multi-dot: w is read once per 8 basis vectors           (:279, :302)
//   A3  w -= sum_i h_i v_i     fused with ||w||^2 ; its epilogue does ALL the small dense work of the
//       step on device: breakdown threshold eps*v_norm_0 (:358-359), H column, the stored Givens
//       rotations, the new rotation (:508-518), the rotated rhs g and the residual estimate |g_{j+1}|
//       (:599-623), and decides whether the cycle continues ('incremental': err > ptol, :591).
//   A4  v_{j+1} = w / ||w||  (or 0 on breakdown)                                               (:359, :363-368)
// End of cycle:  y = R^-1 g (one warp, back substitution; 'batched' uses the same QR instead of the
// reference's normal equations + Cholesky, :407-421 — SURVEY compatibility ledger, <= 7e-15 effect),
// x += V[:, :k] y (:488/:631), r = b - A x fused with ||r||^2 (:489-492), v_0 = r/||r||, and the
// restart test `k < maxiter and ||r|| > atol` (:798) — all flags on device, one host poll per cycle.
#include "bk_internal.cuh"
#include "bk_loop.cuh"
#include "bk_spmv.cuh"
#include "bk_sys.cuh"
#include "bk_dist.cuh"
#include "bk_vec.cuh"

#define BK_GM_MAXM 256  // largest supported restart

struct bk_gm_small {  // device arrays of the small dense problem (all fp64)
  double* R;     // (m+1) x m, column-major, leading dimension m+1
  double* cs;    // m
  double* sn;    // m
  double* g;     // m+1   rotated right-hand side (beta e1)
  double* y;     // m
  double* hcol;  // m+1   projection coefficients of the current step
  int m;
};

template <typename T>
struct bk_gm_eps {
  static constexpr double value = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
};

// ---- scalar epilogues ------------------------------------------------------------------------------
struct bk_epi_gm_tol {  // ||b|| -> atol, ptol   (:729-753)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    const double bs = s[0];
    st->bs = bs;
    const double bnorm = sqrt(fmax(bs, 0.0));
    st->g_bnorm = bnorm;
    const double atol = fmax(st->g_tol_eff * bnorm, st->g_atol_eff);
    st->g_atol = atol;
    st->g_ptol = bnorm * fmin(1.0, atol / bnorm);
  }
};

// after r = b - A x: safe_normalize(r) (thresh eps), restart test, reset of the cycle state
template <typename T>
__device__ __forceinline__ void bk_gm_after_residual(bk_dev_state* st, const bk_gm_small sm, double rr, int is_init) {
  const double norm = sqrt(fmax(rr, 0.0));
  const int use = norm > bk_gm_eps<T>::value;
  const double resnorm = use ? norm : 0.0;
  st->rtrue2 = rr;
  st->g_resnorm = resnorm;
  st->g_scale = norm;
  st->g_use = use;
  if (!is_init) st->k += 1;
  st->g_kcur = 0;
  st->g_err = resnorm;
  sm.g[0] = resnorm;
  const bool go = (st->k < st->maxiter) && (resnorm > st->g_atol);
  if (!go) {
    st->done = 1;
    st->status = (resnorm > st->g_atol) ? BK_ST_MAXITER : BK_ST_CONVERGED;
  }
  // 'incremental' enters the Arnoldi loop only while err > ptol (:591)
  st->g_cycle_over = (st->g_method == BK_GMRES_INCREMENTAL && !(resnorm > st->g_ptol)) ? 1 : 0;
}

template <typename T>
struct bk_epi_gm_resid {
  bk_dev_state* st;
  bk_gm_small sm;
  int is_init;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->matvecs += 1;
    bk_gm_after_residual<T>(st, sm, s[0], is_init);
  }
};

template <typename T>
__global__ void bk_gm_resid_from_bs_kernel(bk_dev_state* st, const bk_gm_small sm) {
  bk_gm_after_residual<T>(st, sm, st->bs, 1);  // x0 = 0: r0 = b exactly
}

template <typename T>
struct bk_epi_gm_vnorm0 {  // _, v_norm_0 = safe_normalize(A v_j)   (:352)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    const double norm = sqrt(fmax(s[0], 0.0));
    st->g_vnorm0 = (norm > bk_gm_eps<T>::value) ? norm : 0.0;
    st->matvecs += 1;
  }
};

struct bk_epi_gm_ignore {
  __device__ __forceinline__ void operator()(const double*) const {}
};
struct bk_epi_gm_ptol {  // Jacobi: ptol = ||M b|| * min(1, atol / ||b||)   (:750-753); s[0] = ||M b||^2
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->g_ptol = sqrt(fmax(s[0], 0.0)) * fmin(1.0, st->g_atol / st->g_bnorm);
  }
};
template <typename T>
struct bk_epi_gm_resid0 {  // Jacobi, x0 = 0: r0 = M b (no matvec to count)
  bk_dev_state* st;
  bk_gm_small sm;
  __device__ __forceinline__ void operator()(const double* s) const { bk_gm_after_residual<T>(st, sm, s[0], 1); }
};
struct bk_epi_gm_xx {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->xx = s[0]; }
};

// ---- A2: h_i = v_i . w for i < count ---------------------------------------------------------------
// Tall-skinny multi-vector GEMV: one pass over w per group of 8 basis vectors, 9 independent 16-byte
// loads in flight per thread; per-CTA partials land in fixed slots, the last CTA adds them in index
// order (one warp per output) => bitwise reproducible.
template <typename T, int W>
__global__ void __launch_bounds__(BK_BLOCK, 3)
bk_multidot_kernel(const T* __restrict__ V, const size_t ldv, const int count, const T* __restrict__ w, const long long n,
                   double* __restrict__ partials, unsigned int* counter, bk_dev_state* st,
                   double* __restrict__ hout, const bk_gsum gs) {
  if (st->done || st->g_cycle_over) return;
  constexpr int NV = 8;
  __shared__ double sh[NV * BK_WARPS];
  __shared__ int s_last;
  const long long npack = n / W;
  const long long stride = (long long)gridDim.x * BK_BLOCK;
  const long long tid = (long long)blockIdx.x * BK_BLOCK + threadIdx.x;
  for (int g0 = 0; g0 < count; g0 += NV) {
    const int nv = (count - g0 < NV) ? count - g0 : NV;
    double acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = 0.0;
    for (long long i = tid; i < npack; i += stride) {
      const bk_vec<T, W> wv = bk_ld<T, W>(w + i * W);
      bk_vec<T, W> vv[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v)
        if (v < nv) vv[v] = bk_ld<T, W>(V + (size_t)(g0 + v) * ldv + i * W);
#pragma unroll
      for (int v = 0; v < NV; ++v)
        if (v < nv) {
#pragma unroll
          for (int j = 0; j < W; ++j) acc[v] += (double)vv[v].v[j] * (double)wv.v[j];
        }
    }
    if (W > 1) {
      const long long t = npack * W + tid;
      if (t < n) {
        const double wv = (double)w[t];
        for (int v = 0; v < nv; ++v) acc[v] += (double)V[(size_t)(g0 + v) * ldv + t] * wv;
      }
    }
    bk_block_reduce<NV>(acc, sh);
    if (threadIdx.x == 0) {
      for (int v = 0; v < nv; ++v) __stcg(&partials[(size_t)(g0 + v) * BK_MAXB + blockIdx.x], acc[v]);
    }
  }
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int t = atomicInc(counter, gridDim.x - 1);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int r = wid; r < count; r += BK_WARPS) {
      double a = 0.0;
      for (int i = lane; i < (int)gridDim.x; i += 32) a += __ldcg(&partials[(size_t)r * BK_MAXB + i]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
      if (lane == 0) hout[r] = a;
    }
    if (gs.mode == 1) {  // peer memory: make the coefficients global right here (mode 2: ncclAllReduce follows)
      __syncthreads();
      const unsigned int seq = gs.p2p.counters[5] + 1u;
      bk_p2p_allreduce_vec(gs.p2p, seq, hout, hout, count, threadIdx.x, BK_BLOCK);
      __syncthreads();
      if (threadIdx.x == 0) {
        gs.p2p.counters[5] = seq;
        if (gs.p2p.counters[4]) {
          st->done = 1;
          st->status = BK_ST_COMM_TIMEOUT;
        }
      }
    }
  }
}

// reference _givens_rotation (:508-518)
__device__ __forceinline__ void bk_givens(double a, double b, double& cs, double& sn) {
  if (fabs(b) == 0.0) {
    cs = 1.0;
    sn = 0.0;
    return;
  }
  const bool a_lt_b = fabs(a) < fabs(b);
  const double t = -(a_lt_b ? a : b) / (a_lt_b ? b : a);
  const double r = 1.0 / sqrt(1.0 + fabs(t) * fabs(t));
  cs = a_lt_b ? r * t : r;
  sn = a_lt_b ? r : r * t;
}

// The small dense work of Arnoldi step j, on ONE thread: hc = h_0..h_j (shared), s_c/s_s = the stored rotations,
// ww = GLOBAL ||w||^2 after the projection.
template <typename T>
__device__ __forceinline__ void bk_gm_dense_step(bk_dev_state* st, const bk_gm_small& sm, const int j, const double ww,
                                                 double* hc, const double* s_c, const double* s_s) {
  const double eps = bk_gm_eps<T>::value;
  const int m = sm.m;
  const double norm1 = sqrt(fmax(ww, 0.0));
  const double thresh = eps * st->g_vnorm0;  // tol = eps * v_norm_0   (:358)
  const int use = norm1 > thresh;
  const double vnorm1 = use ? norm1 : 0.0;
  st->g_scale = norm1;
  st->g_use = use;
  const bool breakdown = (vnorm1 == 0.0);  // :387
  // new Hessenberg column (h_0..h_j, v_norm_1), rotated by the stored Givens rotations (:599-603)
  hc[j + 1] = vnorm1;
  for (int i = 0; i < j; ++i) {
    const double t = s_c[i] * hc[i] - s_s[i] * hc[i + 1];
    hc[i + 1] = s_s[i] * hc[i] + s_c[i] * hc[i + 1];
    hc[i] = t;
  }
  double c_new, s_new;
  bk_givens(hc[j], hc[j + 1], c_new, s_new);  // :606
  sm.cs[j] = c_new;
  sm.sn[j] = s_new;
  hc[j] = c_new * hc[j] - s_new * hc[j + 1];  // :611
  hc[j + 1] = 0.0;
  double* Rcol = sm.R + (size_t)j * (m + 1);
  for (int i = 0; i <= j; ++i) Rcol[i] = hc[i];  // :615
  const double gj = sm.g[j], gj1 = sm.g[j + 1];
  const double t = c_new * gj - s_new * gj1;  // :618-620
  const double gnext = s_new * gj + c_new * gj1;
  sm.g[j] = t;
  sm.g[j + 1] = gnext;
  const double err = fabs(gnext);
  st->g_err = err;
  const int kcur = j + 1;
  st->g_kcur = kcur;
  bool over = breakdown || (kcur >= m);
  if (st->g_method == BK_GMRES_INCREMENTAL && !(err > st->g_ptol)) over = true;  // :591
  st->g_cycle_over = over ? 1 : 0;
}

#include "bk_gmres_persist.cuh"

// ---- A3 (MODE 0): w -= sum_i h_i v_i, ||w||^2, then the step's small dense update
// ---- C2 (MODE 1): x += sum_{i<kcur} y_i v_i
template <typename T, int W, int MODE>
__global__ void __launch_bounds__(BK_BLOCK, 3)
bk_multiaxpy_kernel(const T* __restrict__ V, const size_t ldv, const int count_arg, T* __restrict__ w, const long long n,
                    const bk_scratch sc, bk_dev_state* st, const bk_gm_small sm, const int step, const bk_gsum gs) {
  if (st->done) return;
  if (MODE == 0 && st->g_cycle_over) return;
  __shared__ double s_coef[BK_GM_MAXM + 1];
  __shared__ double s_c[BK_GM_MAXM];
  __shared__ double s_s[BK_GM_MAXM];
  __shared__ double sh[BK_WARPS];
  __shared__ int s_last;
  const int count = (MODE == 0) ? count_arg : st->g_kcur;
  const double* coef = (MODE == 0) ? sm.hcol : sm.y;
  for (int i = threadIdx.x; i < count; i += BK_BLOCK) s_coef[i] = coef[i];
  __syncthreads();
  const long long npack = n / W;
  const long long stride = (long long)gridDim.x * BK_BLOCK;
  const long long tid = (long long)blockIdx.x * BK_BLOCK + threadIdx.x;
  double acc1[1] = {0.0};
  if (count > 0) {
    for (long long i = tid; i < npack; i += stride) {
      bk_vec<T, W> wv = bk_ld<T, W>(w + i * W);
      T a[W];
#pragma unroll
      for (int j = 0; j < W; ++j) a[j] = T(0);
      int c = 0;
      for (; c + 4 <= count; c += 4) {
        bk_vec<T, W> vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) vv[u] = bk_ld<T, W>(V + (size_t)(c + u) * ldv + i * W);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const T hc = (T)s_coef[c + u];
#pragma unroll
          for (int j = 0; j < W; ++j) a[j] = fma(hc, vv[u].v[j], a[j]);
        }
      }
      for (; c < count; ++c) {
        const bk_vec<T, W> vv = bk_ld<T, W>(V + (size_t)c * ldv + i * W);
        const T hc = (T)s_coef[c];
#pragma unroll
        for (int j = 0; j < W; ++j) a[j] = fma(hc, vv.v[j], a[j]);
      }
#pragma unroll
      for (int j = 0; j < W; ++j) {
        wv.v[j] = (MODE == 0) ? bk_sub(wv.v[j], a[j]) : bk_add(wv.v[j], a[j]);
        if (MODE == 0) acc1[0] += (double)wv.v[j] * (double)wv.v[j];
      }
      bk_st<T, W>(w + i * W, wv);
    }
    if (W > 1) {
      const long long t = npack * W + tid;
      if (t < n) {
        T a = T(0);
        for (int c = 0; c < count; ++c) a = fma((T)s_coef[c], V[(size_t)c * ldv + t], a);
        const T o = (MODE == 0) ? bk_sub(w[t], a) : bk_add(w[t], a);
        w[t] = o;
        if (MODE == 0) acc1[0] += (double)o * (double)o;
      }
    }
  }
  if (MODE == 1) return;

  // ---- deterministic ||w||^2 + the small dense step, on the last CTA -------------------------------
  bk_block_reduce<1>(acc1, sh);
  if (threadIdx.x == 0) {
    __stcg(&sc.partials[blockIdx.x], acc1[0]);
    __threadfence();
    const unsigned int t = atomicInc(sc.counter, gridDim.x - 1);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double tot[1] = {0.0};
  for (int i = threadIdx.x; i < (int)gridDim.x; i += BK_BLOCK) tot[0] += __ldcg(&sc.partials[i]);
  bk_block_reduce<1>(tot, sh);
  // stage the rotations of the earlier steps (s_coef already holds h_0..h_j)
  const int j = step;
  for (int i = threadIdx.x; i < j; i += BK_BLOCK) {
    s_c[i] = sm.cs[i];
    s_s[i] = sm.sn[i];
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double ww[1];
  if (!bk_gsum_finish<1>(gs, st, tot, ww)) return;  // NCCL path: bk_gm_step_kernel finishes the step
  bk_gm_dense_step<T>(st, sm, j, ww[0], s_coef, s_c, s_s);
}

// NCCL path: the dense step after ncclAllReduce of ||w||^2 (red[0])
template <typename T>
__global__ void __launch_bounds__(BK_BLOCK) bk_gm_step_kernel(bk_dev_state* st, const bk_gm_small sm, const int j,
                                                            const double* red) {
  if (st->done || st->g_cycle_over) return;
  __shared__ double s_coef[BK_GM_MAXM + 1];
  __shared__ double s_c[BK_GM_MAXM];
  __shared__ double s_s[BK_GM_MAXM];
  for (int i = threadIdx.x; i <= j; i += BK_BLOCK) s_coef[i] = sm.hcol[i];
  for (int i = threadIdx.x; i < j; i += BK_BLOCK) {
    s_c[i] = sm.cs[i];
    s_s[i] = sm.sn[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) bk_gm_dense_step<T>(st, sm, j, red[0], s_coef, s_c, s_s);
}

// ---- C1: y = R[:k,:k]^-1 g[:k] (back substitution on one warp), then clear g[1..m] for the next cycle
__global__ void bk_gm_solve_kernel(bk_dev_state* st, const bk_gm_small sm) {
  if (st->done) return;
  const int lane = threadIdx.x;
  const int k = st->g_kcur;
  const int m = sm.m;
  const int ld = m + 1;
  for (int i = k - 1; i >= 0; --i) {
    double a = 0.0;
    for (int c = i + 1 + lane; c < k; c += 32) a += sm.R[(size_t)c * ld + i] * sm.y[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) sm.y[i] = (sm.g[i] - a) / sm.R[(size_t)i * ld + i];
    __syncwarp();
  }
  __syncwarp();
  for (int i = 1 + lane; i <= m; i += 32) sm.g[i] = 0.0;
}

template <typename T, typename Sys>
static int bk_gmres_t(const Sys& sys, const void* b, void* x_user, int has_x0, double tol_eff, double atol_eff,
                      int restart, int64_t maxiter, int method, bk_result* res, cudaStream_t s,
                      const T* diag = nullptr, const bk_sgs* S = nullptr) {
  bk_handle* h = sys.h;
  const long long n = sys.n();
  const int m = restart;
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  BK_TRY(bk_ws_reserve(h, (size_t)(m + (S ? 5 : 4)) * npad * sizeof(T)));
  T* V = (T*)h->ws;
  T* w = V + (size_t)(m + 1) * npad;
  T* x = w + npad;
  T* bw = x + npad;  // private copy of b: keeps the cached cycle graph independent of the caller's pointer
  T* u = bw + npad;  // SGS: the A-product the sweeps read (they cannot work in place)
  bk_dev_state* st = h->st;
  const size_t vbytes = (size_t)n * sizeof(T);
  constexpr int NW = bk_native_w<T>::value;
  const bk_gsum gs = sys.gsum();
  bk_call_begin(h, s, "bk_gmres");

  // small dense arrays
  const size_t small_doubles = (size_t)(m + 1) * m + 2 * (size_t)m + 2 * (size_t)(m + 1) + m + 16;
  if (h->gm_small_bytes < small_doubles * sizeof(double)) {
    bk_graphs_invalidate(h);
    if (h->gm_small) {
      BK_CUDA(cudaDeviceSynchronize());
      cudaFree(h->gm_small);
      h->gm_small = nullptr;
      h->gm_small_bytes = 0;
    }
    if (cudaMalloc(&h->gm_small, small_doubles * sizeof(double)) != cudaSuccess) {
      cudaGetLastError();
      return bk_fail(BK_ERR_ALLOC, "bk_gmres: small-array allocation failed");
    }
    h->gm_small_bytes = small_doubles * sizeof(double);
  }
  const size_t part_bytes = (size_t)(m + 4) * BK_MAXB * sizeof(double);  // (+3 rows: the persistent kernel's norms)
  if (h->gm_partials_bytes < part_bytes) {
    bk_graphs_invalidate(h);
    if (h->gm_partials) {
      BK_CUDA(cudaDeviceSynchronize());
      cudaFree(h->gm_partials);
      h->gm_partials = nullptr;
      h->gm_partials_bytes = 0;
    }
    if (cudaMalloc(&h->gm_partials, part_bytes) != cudaSuccess) {
      cudaGetLastError();
      return bk_fail(BK_ERR_ALLOC, "bk_gmres: partials allocation failed");
    }
    h->gm_partials_bytes = part_bytes;
  }
  bk_gm_small sm;
  sm.m = m;
  sm.R = h->gm_small;
  sm.cs = sm.R + (size_t)(m + 1) * m;
  sm.sn = sm.cs + m;
  sm.g = sm.sn + m;
  sm.y = sm.g + (m + 1);
  sm.hcol = sm.y + m;
  BK_CUDA(cudaMemsetAsync(h->gm_small, 0, small_doubles * sizeof(double), s));

  bk_dev_state init;
  memset(&init, 0, sizeof(init));
  init.maxiter = maxiter < 0 ? 10 * sys.n_global() : maxiter;
  init.status = BK_ST_MAXITER;
  init.g_tol_eff = tol_eff;
  init.g_atol_eff = atol_eff;
  init.g_method = method;
  init.g_restart = m;
  bk_state_set_kernel<<<1, 1, 0, s>>>(st, init);
  BK_KERNEL_CHECK();

  const int grid = bk_grid_vec_n(h, n, 2 * NW);
  auto normalize = [&](const T* src, T* dst, int guard, cudaStream_t cs) -> int {
    bk_op_normalize<T> op;
    op.w = src;
    op.v = dst;
    op.st = st;
    op.guard = guard;
    return sys.template ew<T>(op, true, 3, cs);
  };

  // ---- set-up: ||b||, tolerances, r0, v_0 ----------------------------------------------------------
  BK_CUDA(cudaMemcpyAsync(bw, b, vbytes, cudaMemcpyDeviceToDevice, s));
  b = bw;
  BK_TRY((sys.template dot<T>(b, b, bk_epi_gm_tol{st}, 1, s)));
  const bool dal = diag && bk_aligned16(diag);
  // left Jacobi preconditioning (diag != nullptr): every A-product is followed by an in-place division by d that also
  // carries the norm the unpreconditioned path fuses into the SpMV
  auto scale_sq = [&](T* vec, auto epi, int guard, cudaStream_t cs) -> int {
    bk_op_scale_sq<T, decltype(epi)> op;
    op.w = vec;
    op.d = diag;
    op.epi = epi;
    op.st = st;
    op.guard = guard;
    return sys.template ew<T>(op, dal, 1, cs);
  };
  // left symmetric Gauss-Seidel preconditioning (S != nullptr): the A-product goes to u, the sweeps write w = M u and
  // a guarded reduction carries the norm
  auto sgs_sq = [&](const T* src, auto epi, int guard, cudaStream_t cs) -> int {
    BK_TRY(bk_sgs_run(h, S, src, w, guard, cs));
    bk_op_dot_epi<T, decltype(epi)> op;
    op.x = w;
    op.y = w;
    op.epi = epi;
    op.st = st;
    op.guard = guard;
    return sys.template ew<T>(op, true, 1, cs);
  };
  if (diag) {
    BK_CUDA(cudaMemcpyAsync(w, b, vbytes, cudaMemcpyDeviceToDevice, s));
    BK_TRY(scale_sq(w, bk_epi_gm_ptol{st}, 0, s));  // w = M b (also r0 when x0 = 0)
  } else if (S) {
    BK_TRY(sgs_sq((const T*)b, bk_epi_gm_ptol{st}, 0, s));
  }
  if (has_x0) {
    BK_CUDA(cudaMemcpyAsync(x, x_user, vbytes, cudaMemcpyDeviceToDevice, s));
    if (diag) {
      BK_TRY((sys.template matvec<T, 1, 2>(x, w, nullptr, b, 0, bk_epi_gm_ignore{}, s)));
      BK_TRY(scale_sq(w, bk_epi_gm_resid<T>{st, sm, 1}, 0, s));
    } else if (S) {
      BK_TRY((sys.template matvec<T, 1, 2>(x, u, nullptr, b, 0, bk_epi_gm_ignore{}, s)));
      BK_TRY(sgs_sq(u, bk_epi_gm_resid<T>{st, sm, 1}, 0, s));
    } else {
      BK_TRY((sys.template matvec<T, 1, 2>(x, w, nullptr, b, 0, bk_epi_gm_resid<T>{st, sm, 1}, s)));
    }
  } else {
    BK_CUDA(cudaMemsetAsync(x, 0, vbytes, s));
    if (diag || S) {  // w already holds M b; its norm is ||M b|| = sqrt of what the ptol pass summed: recompute cheaply
      BK_TRY((sys.template dot<T>(w, w, bk_epi_gm_resid0<T>{st, sm}, 1, s)));
    } else {
      BK_CUDA(cudaMemcpyAsync(w, b, vbytes, cudaMemcpyDeviceToDevice, s));
      bk_gm_resid_from_bs_kernel<T><<<1, 1, 0, s>>>(st, sm);
      BK_KERNEL_CHECK();
    }
  }
  BK_TRY(normalize(w, V, 0, s));

  // ---- one restart cycle ------------------------------------------------------------------------
  auto enqueue_cycle = [&](cudaStream_t cs) -> int {
    for (int j = 0; j < m; ++j) {
      if (diag) {
        BK_TRY((sys.template matvec<T, 0, 2>(V + (size_t)j * npad, w, nullptr, nullptr, 2, bk_epi_gm_ignore{}, cs)));
        BK_TRY(scale_sq(w, bk_epi_gm_vnorm0<T>{st}, 2, cs));
      } else if (S) {
        BK_TRY((sys.template matvec<T, 0, 2>(V + (size_t)j * npad, u, nullptr, nullptr, 2, bk_epi_gm_ignore{}, cs)));
        BK_TRY(sgs_sq(u, bk_epi_gm_vnorm0<T>{st}, 2, cs));
      } else {
        BK_TRY((sys.template matvec<T, 0, 2>(V + (size_t)j * npad, w, nullptr, nullptr, 2, bk_epi_gm_vnorm0<T>{st}, cs)));
      }
      bk_multidot_kernel<T, NW><<<grid, BK_BLOCK, 0, cs>>>(V, npad, j + 1, w, n, h->gm_partials, h->counters + 4, st,
                                                            sm.hcol, gs);
      BK_KERNEL_CHECK();
      if (gs.mode == 2) BK_TRY(sys.allreduce(sm.hcol, j + 1, cs));
      bk_multiaxpy_kernel<T, NW, 0><<<grid, BK_BLOCK, 0, cs>>>(V, npad, j + 1, w, n, bk_slot(h, 1), st, sm, j, gs);
      BK_KERNEL_CHECK();
      if (gs.mode == 2) {
        BK_TRY(sys.allreduce(gs.red, 1, cs));
        bk_gm_step_kernel<T><<<1, BK_BLOCK, 0, cs>>>(st, sm, j, gs.red);
        BK_KERNEL_CHECK();
      }
      BK_TRY(normalize(w, V + (size_t)(j + 1) * npad, 2, cs));
    }
    bk_gm_solve_kernel<<<1, 32, 0, cs>>>(st, sm);
    BK_KERNEL_CHECK();
    bk_multiaxpy_kernel<T, NW, 1><<<grid, BK_BLOCK, 0, cs>>>(V, npad, 0, x, n, bk_slot(h, 1), st, sm, 0, gs);
    BK_KERNEL_CHECK();
    if (diag) {
      BK_TRY((sys.template matvec<T, 1, 2>(x, w, nullptr, b, 1, bk_epi_gm_ignore{}, cs)));
      BK_TRY(scale_sq(w, bk_epi_gm_resid<T>{st, sm, 0}, 1, cs));
    } else if (S) {
      BK_TRY((sys.template matvec<T, 1, 2>(x, u, nullptr, b, 1, bk_epi_gm_ignore{}, cs)));
      BK_TRY(sgs_sq(u, bk_epi_gm_resid<T>{st, sm, 0}, 1, cs));
    } else {
      BK_TRY((sys.template matvec<T, 1, 2>(x, w, nullptr, b, 1, bk_epi_gm_resid<T>{st, sm, 0}, cs)));
    }
    BK_TRY(normalize(w, V, 1, cs));
    return BK_OK;
  };
  const bool use_graph = h->loop_mode != BK_LOOP_STREAM;
  uint64_t key[6] = {3 /*gmres*/, sys.uid(), (uint64_t)(uintptr_t)h->ws, (uint64_t)n,
                     (uint64_t)sys.dtype() | ((uint64_t)m << 8) | ((uint64_t)method << 24),
                     (uint64_t)bk_grid_spmv(h) | ((uint64_t)bk_grid_vec(h) << 32)};
  if (diag) key[1] ^= (uint64_t)(uintptr_t)diag * 0x9e3779b97f4a7c15ull;  // its address is baked into the graph
  if (S) key[1] ^= (uint64_t)(uintptr_t)S * 0xc2b2ae3d27d4eb4full;
  int64_t chunks = 0;
  bk_call_mark(h, "loop");
  bool persistent = false;
  if constexpr (!Sys::kDist) {
    // launch-bound (L2-resident) systems: the whole solve in ONE cooperative kernel (bk_gmres_persist.cuh)
    const bk_csr* A = sys.A;
    if (S == nullptr && A->rowptr && A->col) {
      bk_gp_args ga;
      ga.rowptr = A->rowptr;
      ga.col = A->col;
      ga.val = A->val;
      ga.diag = diag;
      ga.n = n;
      ga.V = V;
      ga.ldv = npad;
      ga.w = w;
      ga.x = x;
      ga.b = b;
      ga.st = st;
      ga.R = sm.R;
      ga.y = sm.y;
      ga.partials = h->gm_partials;
      ga.m = m;
      BK_TRY(bk_launch_persistent(h, bk_gmres_persistent_kernel<T, true>, bk_gmres_persistent_kernel<T, false>, ga, n, s,
                                  &persistent));
    }
  }
  if (!persistent) BK_TRY(bk_run_loop(h, s, use_graph, key, enqueue_cycle, &chunks));
  bk_call_mark(h, "final");

  // ---- final check (:766-773): the last residual pass already holds ||b - A x||; add ||x|| --------
  BK_TRY((sys.template dot<T>(x, x, bk_epi_gm_xx{st}, 1, s)));
  BK_CUDA(cudaMemcpyAsync(x_user, x, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(&h->st_host[3], st, sizeof(bk_dev_state), cudaMemcpyDeviceToHost, s));
  bk_call_stop(h, s);
  BK_CUDA(cudaStreamSynchronize(s));
  const bk_dev_state* fin = &h->st_host[3];
  bk_call_finish(h, res);
  res->iterations = fin->k;
  res->matvecs = fin->matvecs;
  res->kernel_launches = (persistent ? 1 : chunks * (4 * (int64_t)m + 4)) + 5;
  if (S)  // every A-product is followed by the sweeps and the norm: m + 1 per cycle, 2 (3 with x0) in the set-up
    res->kernel_launches += (chunks * (m + 1) + 2 + (has_x0 ? 1 : 0)) * (int64_t)(bk_sgs_launches(S) + 1);
  res->status = fin->status;
  res->final_residual = sqrt(fmax(fin->rtrue2, 0.0));
  res->b_norm = fin->g_bnorm;
  res->x_norm = sqrt(fmax(fin->xx, 0.0));
  res->threshold = 10.0 * fin->g_atol;  // "Allow 10x tolerance for convergence check" (:769)
  res->rr_last = fin->g_resnorm;
  const bool failed = (res->x_norm != res->x_norm) || (res->final_residual > res->threshold);
  res->info = failed ? -1 : 0;
  return sys.check_comm(fin, "gmres");
}

static int bk_gmres_args_check(const char* who, int restart, int method);

/* GMRES with the built-in symmetric Gauss-Seidel preconditioner applied from the left (v = M(A v), r = M(b - A x),
 * ptol from ||M b||, final check on ||M(b - A x)||), as bk_gmres_jacobi. */
extern "C" int bk_gmres_sgs(bk_handle* h, const bk_csr* A, const bk_sgs* S, const void* b, void* x, int has_x0,
                            double tol_eff, double atol_eff, int restart, int64_t maxiter, int method, bk_result* result,
                            void* stream) {
  BK_TRY(bk_solver_args_check("bk_gmres_sgs", h, A, b, x, result));
  BK_TRY(bk_gmres_args_check("bk_gmres_sgs", restart, method));
  BK_TRY(bk_sgs_args_check("bk_gmres_sgs", h, A, S));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_gmres_t<double>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                              (cudaStream_t)stream, nullptr, S);
  return bk_gmres_t<float>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                           (cudaStream_t)stream, nullptr, S);
}

static int bk_gmres_args_check(const char* who, int restart, int method) {
  if (restart < 1 || restart > BK_GM_MAXM)
    return bk_fail(BK_ERR_UNSUPPORTED, "%s: restart must be in [1, %d], got %d", who, BK_GM_MAXM, restart);
  if (method != BK_GMRES_BATCHED && method != BK_GMRES_INCREMENTAL)
    return bk_fail(BK_ERR_ARG, "%s: unknown method %d", who, method);
  return BK_OK;
}

extern "C" int bk_gmres(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol_eff,
                        double atol_eff, int restart, int64_t maxiter, int method, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_gmres", h, A, b, x, result));
  BK_TRY(bk_gmres_args_check("bk_gmres", restart, method));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_gmres_t<double>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                              (cudaStream_t)stream);
  return bk_gmres_t<float>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                           (cudaStream_t)stream);
}

/* GMRES with the built-in Jacobi preconditioner applied from the left exactly as the reference does with a callable M:
 * v = M(A v) in every Arnoldi step (:351), r = M(b - A x) at every restart (:491/:636/:791), ptol from ||M b|| (:750),
 * final check on ||M(b - A x)|| (:766). */
extern "C" int bk_gmres_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0,
                               double tol_eff, double atol_eff, int restart, int64_t maxiter, int method,
                               bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_gmres_jacobi", h, A, b, x, result));
  BK_TRY(bk_gmres_args_check("bk_gmres_jacobi", restart, method));
  if (!diag && A->n > 0) return bk_fail(BK_ERR_ARG, "bk_gmres_jacobi: null diagonal");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_gmres_t<double>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                              (cudaStream_t)stream, (const double*)diag);
  return bk_gmres_t<float>(sys, b, x, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                           (cudaStream_t)stream, (const float*)diag);
}

// Row-partitioned GMRES: the basis is partitioned like every vector; V^T w is one all-reduce of j+1 doubles and the
// small dense problem is replicated (identical on every rank because the all-reduced sums are) — SURVEY §8e.
extern "C" int bk_dist_gmres(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol_eff,
                             double atol_eff, int restart, int64_t maxiter, int method, int64_t n_global,
                             bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_gmres: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local)) return bk_fail(BK_ERR_ARG, "bk_dist_gmres: null vector");
  BK_TRY(bk_gmres_args_check("bk_dist_gmres", restart, method));
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global};
  if (D->dtype == BK_F64)
    return bk_gmres_t<double>(sys, b_local, x_local, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                              (cudaStream_t)stream);
  return bk_gmres_t<float>(sys, b_local, x_local, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                           (cudaStream_t)stream);
}

extern "C" int bk_dist_gmres_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local, void* x_local,
                                    int has_x0, double tol_eff, double atol_eff, int restart, int64_t maxiter,
                                    int method, int64_t n_global, bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_gmres_jacobi: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local || !diag_local))
    return bk_fail(BK_ERR_ARG, "bk_dist_gmres_jacobi: null vector");
  BK_TRY(bk_gmres_args_check("bk_dist_gmres_jacobi", restart, method));
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global};
  if (D->dtype == BK_F64)
    return bk_gmres_t<double>(sys, b_local, x_local, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                              (cudaStream_t)stream, (const double*)diag_local);
  return bk_gmres_t<float>(sys, b_local, x_local, has_x0, tol_eff, atol_eff, restart, maxiter, method, result,
                           (cudaStream_t)stream, (const float*)diag_local);
}
