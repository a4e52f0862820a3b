// bk_cg.cu — conjugate gradient with a device-resident loop.
// Replaces _cg_solve (reference torch_sparse_linalg.py:806-856) and its wrapper _isolve (:967-1016).
//
// Per iteration (recurrences and operation order exactly the reference's, :843-853):
//   K1  Ap = A p            fused with p.Ap ; epilogue: alpha = gamma / p.Ap
//   K2  r -= alpha Ap ; fused with r.r ; epilogue: beta = gamma'/gamma, k += 1,
//       stop test `k >= maxiter or gamma' <= atol2` (:841) for the next iteration
//   K3  x += alpha p ; p = r + beta p      (x rides along with the p-update: both read p_k; 8n instead of 9n)
// With option fuse_xpay K3 disappears: K1 gathers r[c] + beta p_old[c] on the fly (bitwise the
// same value K3 would have stored) and writes the new p for its own rows (double-buffered p).
// Algorithmic HBM bytes per iteration (the reference-equivalent plan): nnz*(8+4) + (n+1)*4 + 11*n*8  (SURVEY §8d).
#include "bk_internal.cuh"
#include "bk_loop.cuh"
#include "bk_spmv.cuh"
#include "bk_sys.cuh"
#include "bk_dist.cuh"
#include "bk_vec.cuh"

// ---- epilogues ---------------------------------------------------------------------------------
struct bk_epi_cg_pAp {  // alpha = gamma / (p . Ap)   (:845)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->pAp = s[0];
    st->alpha_lag = st->alpha;  // lagged-x cut: in an odd iteration the previous alpha is still owed to x
    st->alpha = st->gamma / s[0];
  }
};

struct bk_epi_set_gamma {  // gamma0 = r0 . r0  (:826)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->gamma = s[0]; }
};

struct bk_epi_cg_init {  // bs = b.b ; atol2 = max(tol^2 bs, atol^2) (:815-817) ; first stop test
  bk_dev_state* st;
  int has_x0;
  __device__ __forceinline__ void operator()(const double* s) const {
    const double bs = s[0];
    st->bs = bs;
    st->atol2 = fmax(st->tolsq32 * bs, st->atolsq32);
    if (!has_x0) st->gamma = bs;  // r0 = b - A*0 = b exactly
    if (st->maxiter <= 0) {
      st->done = 1;
      st->status = BK_ST_MAXITER;
    }
    if (st->gamma <= st->atol2) {
      st->done = 1;
      st->status = BK_ST_CONVERGED;
    }
  }
};

struct bk_epi_final_r {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->rtrue2 = s[0]; }
};
struct bk_epi_final_x {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->xx = s[0]; }
};

// Shared by all solvers: tolerance fields with the reference's fp32 rounding of torch.tensor(tol).
void bk_state_fill_tol(bk_dev_state* v, double tol, double atol) {
  const float t = (float)tol, a = (float)atol;
  v->tol32 = (double)t;
  v->atol32 = (double)a;
  v->tolsq32 = (double)(t * t);    // torch.square on an fp32 0-dim tensor
  v->atolsq32 = (double)(a * a);
}

// Shared: final true-residual check of _isolve (:1008-1016) from the device state copy.
void bk_fill_result_isolve(const bk_dev_state* st, bk_result* res, int64_t matvecs) {
  res->iterations = st->k;
  res->matvecs = matvecs;
  res->status = st->status;
  res->final_residual = sqrt(fmax(st->rtrue2, 0.0));
  res->b_norm = sqrt(fmax(st->bs, 0.0));
  res->x_norm = sqrt(fmax(st->xx, 0.0));
  res->threshold = fmax(st->tol32 * res->b_norm, st->atol32);
  const bool failed = (res->x_norm != res->x_norm) || (res->final_residual > res->threshold);
  res->info = failed ? -1 : 0;
}

// ---- persistent cooperative CG for launch-latency-bound (small) systems ------------------------------------
// One cooperative kernel runs the WHOLE iteration loop: three grid-wide barriers per iteration replace three
// kernel launches (which cost ~5 us each at n = 65k even inside a CUDA graph).  Every CTA re-adds the per-CTA
// partials of a dot product in the same fixed order after the barrier, so all threads hold bitwise identical
// alpha/beta/gamma and take the reference's stop test (`k >= maxiter or gamma <= atol2`, :841) uniformly — the
// convergence flag never leaves the device.  Thread-per-row SpMV is fine here: the matrix and vectors are L2
// resident at these sizes.  Same recurrences and rounding (separate mul/add) as the multi-kernel path.
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

__device__ __forceinline__ double bk_sum_partials(const double* partials, int count, double* sh) {
  // executed by all threads of the CTA; result identical in every CTA (fixed order)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (wid == 0) {
    double a = 0.0;
    for (int i = lane; i < count; i += 32) a += __ldcg(partials + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
    if (lane == 0) sh[0] = a;
  }
  __syncthreads();
  const double r = sh[0];
  __syncthreads();
  return r;
}

#define BK_PERSIST_BLOCK 1024
#define BK_PERSIST_WARPS (BK_PERSIST_BLOCK / 32)

// Two grid barriers per iteration: the p-update is folded into the SpMV gather (p_new[c] = r[c] + beta p_old[c] is
// recomputed on the fly with the same two roundings the stand-alone update would use, and stored once per owned row
// into the other p buffer), so only the two dot products need a barrier.  1024-thread CTAs keep the barrier small.
template <typename T>
__global__ void __launch_bounds__(BK_PERSIST_BLOCK, 1)
bk_cg_persistent_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const T* __restrict__ val,
                        T* x, T* r, T* p0, T* p1, T* ap, const long long n, bk_dev_state* st, double* partials) {
  cg::grid_group grid = cg::this_grid();
  __shared__ double sh_red[BK_PERSIST_WARPS];
  __shared__ double sh_one[1];
  const long long tid = (long long)blockIdx.x * BK_PERSIST_BLOCK + threadIdx.x;
  const long long nth = (long long)gridDim.x * BK_PERSIST_BLOCK;
  double gamma = st->gamma;
  const double atol2 = st->atol2;
  const long long maxiter = st->maxiter;
  long long k = 0;
  int status = BK_ST_MAXITER;
  if (st->done) return;  // uniform: set by the init epilogue (zero rhs / maxiter 0)
  T beta = T(0);         // p_{-1} = 0 (buffer p0 is zero-filled), so the first gather forms p_0 = r_0 exactly
  T* pold = p0;
  T* pnew = p1;
  for (;;) {
    if (k >= maxiter) {
      status = BK_ST_MAXITER;
      break;
    }
    if (gamma <= atol2) {
      status = BK_ST_CONVERGED;
      break;
    }
    // phase 1: p_new = r + beta p_old (own rows), Ap = A p_new, partial p.Ap
    double acc[1] = {0.0};
    for (long long row = tid; row < n; row += nth) {
      T sum = T(0);
      for (int e = rowptr[row]; e < rowptr[row + 1]; ++e) {
        const int c = col[e];
        sum = fma(val[e], bk_add(r[c], bk_mul(beta, pold[c])), sum);
      }
      const T pr = bk_add(r[row], bk_mul(beta, pold[row]));
      pnew[row] = pr;
      ap[row] = sum;
      acc[0] += (double)pr * (double)sum;
    }
    bk_block_reduce<1, BK_PERSIST_WARPS>(acc, sh_red);
    if (threadIdx.x == 0) __stcg(partials + blockIdx.x, acc[0]);
    grid.sync();
    const double pAp = bk_sum_partials(partials, (int)gridDim.x, sh_one);
    const T alpha = (T)(gamma / pAp);
    // phase 2: x += alpha p ; r -= alpha Ap ; partial r.r
    acc[0] = 0.0;
    for (long long row = tid; row < n; row += nth) {
      x[row] = bk_add(x[row], bk_mul(alpha, pnew[row]));
      const T rn = bk_sub(r[row], bk_mul(alpha, ap[row]));
      r[row] = rn;
      acc[0] += (double)rn * (double)rn;
    }
    bk_block_reduce<1, BK_PERSIST_WARPS>(acc, sh_red);
    if (threadIdx.x == 0) __stcg(partials + BK_MAXB + blockIdx.x, acc[0]);
    grid.sync();  // also publishes the new r (and p_new) to the next iteration's gathers
    const double gamma_new = bk_sum_partials(partials + BK_MAXB, (int)gridDim.x, sh_one);
    beta = (T)(gamma_new / gamma);
    gamma = gamma_new;
    ++k;
    T* t = pold;
    pold = pnew;
    pnew = t;
  }
  if (tid == 0) {
    st->k = k;
    st->gamma = gamma;
    st->done = 1;
    st->status = status;
  }
}

template <typename T>
static int bk_cg_try_persistent(bk_handle* h, const bk_csr* A, T* x, T* r, T* p0, T* p1, T* ap, cudaStream_t s,
                                bool* used) {
  *used = false;
  if (!h->persistent || A->n > (long long)h->persistent_max_n) return BK_OK;
  int coop = 0;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device);
  if (!coop) return BK_OK;
  int per_sm = 0;
  BK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bk_cg_persistent_kernel<T>, BK_PERSIST_BLOCK, 0));
  long long grid = (A->n + BK_PERSIST_BLOCK - 1) / BK_PERSIST_BLOCK;
  const long long cap = (long long)per_sm * h->num_sms;
  if (grid > cap) grid = cap;
  if (grid > BK_MAXB) grid = BK_MAXB;
  if (grid < 1) return BK_OK;
  const int* rowptr = A->rowptr;
  const int* col = A->col;
  const T* val = (const T*)A->val;
  long long n = A->n;
  bk_dev_state* st = h->st;
  double* partials = h->partials;  // slots 0 and 1 (BK_MAXB apart)
  void* args[] = {(void*)&rowptr, (void*)&col, (void*)&val, (void*)&x,  (void*)&r,       (void*)&p0,
                  (void*)&p1,     (void*)&ap,  (void*)&n,   (void*)&st, (void*)&partials};
  BK_CUDA(cudaLaunchCooperativeKernel((const void*)bk_cg_persistent_kernel<T>, dim3((unsigned)grid),
                                      dim3(BK_PERSIST_BLOCK), args, 0, s));
  *used = true;
  return BK_OK;
}

template <typename T>
struct bk_cg_vecs {
  T* x;
  T* r;
  T* p[2];
  T* ap;
};

template <typename T>
static int bk_cg_enqueue_iter(bk_handle* h, const bk_csr* A, const bk_cg_vecs<T>& v, int it, bool fuse, bool lag,
                              cudaStream_t s) {
  const long long n = A->n;
  bk_dev_state* st = h->st;
  const T* pcur;
  if (fuse) {
    const T* pold = v.p[it & 1];
    T* pnew = v.p[(it + 1) & 1];
    bk_spmv_args a = bk_spmv_base(A, st);
    a.x = v.r;
    a.x2 = pold;
    a.xout = pnew;
    a.y = v.ap;
    a.guard = 1;
    a.use_parity = h->snake;
    bk_epi_cg_pAp epi{st};
    BK_TRY((bk_launch_spmv<0, 1, 1>(h, A, a, bk_slot(h, 0), epi, s)));
    pcur = pnew;
  } else {
    pcur = lag ? v.p[it & 1] : v.p[0];  // lagged-x cut: p ping-pongs (chunks are even-sized and start at an even k)
    bk_spmv_args a = bk_spmv_base(A, st);
    a.x = pcur;
    a.w = pcur;
    a.y = v.ap;
    a.guard = 1;
    a.use_parity = h->snake;
    a.l2_hints = h->l2_hints;
    bk_epi_cg_pAp epi{st};
    BK_TRY((bk_launch_spmv<0, 1, 0>(h, A, a, bk_slot(h, 0), epi, s)));
  }
  if (fuse) {
    bk_op_cg_update<T> op;
    op.p = pcur;
    op.ap = v.ap;
    op.x = v.x;
    op.r = v.r;
    op.st = st;
    op.snake = h->snake;
    BK_TRY(bk_launch_ew<T>(h, op, n, true, bk_slot(h, 1), s));
  } else {
    {
      bk_op_cg_r<T> op;
      op.ap = v.ap;
      op.r = v.r;
      op.st = st;
      op.snake = h->snake;
      op.hints = h->l2_hints;
      BK_TRY(bk_launch_ew<T>(h, op, n, true, bk_slot(h, 1), s));
    }
    if (!lag) {
      bk_op_cg_xp<T> op;
      op.x = v.x;
      op.p = v.p[0];
      op.r = v.r;
      op.st = st;
      op.snake = h->snake;
      op.hints = h->l2_hints;
      BK_TRY(bk_launch_ew<T>(h, op, n, true, bk_slot(h, 2), s));
    } else if ((it & 1) == 0) {
      bk_op_cg_p_lag<T> op;
      op.x = v.x;
      op.pcur = v.p[0];
      op.pnext = v.p[1];
      op.r = v.r;
      op.st = st;
      op.snake = h->snake;
      BK_TRY(bk_launch_ew<T>(h, op, n, true, bk_slot(h, 2), s));
    } else {
      bk_op_cg_xp_lag<T> op;
      op.x = v.x;
      op.pprev = v.p[0];
      op.pcur = v.p[1];
      op.r = v.r;
      op.st = st;
      op.snake = h->snake;
      BK_TRY(bk_launch_ew<T>(h, op, n, true, bk_slot(h, 2), s));
    }
  }
  return BK_OK;
}

template <typename T>
static int bk_cg_t(bk_handle* h, const bk_csr* A, const void* b, void* x_user, int has_x0, double tol, double atol,
                   int64_t maxiter, bk_result* res, cudaStream_t s) {
  const long long n = A->n;
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  // fused p-update: 2 kernels per iteration instead of 3 — a win while the iteration is launch-latency bound
  // (measured: -17 % at n = 65k, +13 % at n = 1M), so 'auto' (-1) enables it for small systems only
  const bool persist_ok = h->persistent && n <= (long long)h->persistent_max_n;  // one cooperative kernel runs the loop
  const bool fuse = !persist_ok && A->kernel != 1 && A->split == nullptr && (h->fuse_xpay > 0 || (h->fuse_xpay < 0 && n <= 300000));
  const bool lag = !fuse && !persist_ok && h->cg_lag_x != 0;
  BK_TRY(bk_ws_reserve(h, (size_t)5 * npad * sizeof(T)));
  bk_cg_vecs<T> v;
  v.x = (T*)h->ws;
  v.r = v.x + npad;
  v.p[0] = v.r + npad;
  v.p[1] = v.p[0] + npad;
  v.ap = v.p[1] + npad;
  bk_dev_state* st = h->st;
  const size_t vbytes = (size_t)n * sizeof(T);
  bk_call_begin(h, s, "bk_cg");

  bk_dev_state init;
  memset(&init, 0, sizeof(init));
  init.maxiter = maxiter < 0 ? 10 * n : maxiter;
  init.status = BK_ST_MAXITER;
  bk_state_fill_tol(&init, tol, atol);
  bk_state_set_kernel<<<1, 1, 0, s>>>(st, init);
  BK_KERNEL_CHECK();

  if (has_x0) {
    BK_CUDA(cudaMemcpyAsync(v.x, x_user, vbytes, cudaMemcpyDeviceToDevice, s));
    bk_spmv_args a = bk_spmv_base(A, st);  // r0 = b - A x0, gamma0 = r0.r0   (:820, :826)
    a.x = v.x;
    a.y = v.r;
    a.b = b;
    bk_epi_set_gamma epi{st};
    BK_TRY((bk_launch_spmv<1, 2, 0>(h, A, a, bk_slot(h, 0), epi, s)));
  } else {
    BK_CUDA(cudaMemsetAsync(v.x, 0, vbytes, s));
    BK_CUDA(cudaMemcpyAsync(v.r, b, vbytes, cudaMemcpyDeviceToDevice, s));
  }
  {
    bk_epi_cg_init epi{st, has_x0};
    BK_TRY((bk_dot_epi<T>(h, n, b, b, epi, 1, s)));
  }
  if (fuse || persist_ok) {
    // p_{-1} = 0, beta = 0  =>  the first fused SpMV forms p_0 = r_0 + 0*0 = r_0  (:821)
    BK_CUDA(cudaMemsetAsync(v.p[0], 0, vbytes, s));
  } else {
    BK_CUDA(cudaMemcpyAsync(v.p[0], v.r, vbytes, cudaMemcpyDeviceToDevice, s));
  }

  const double bytes_iter = (double)A->nnz * (sizeof(T) + 4) + 4.0 * (n + 1) + 11.0 * n * sizeof(T);
  const int chunk = bk_pick_chunk(h, bytes_iter, fuse ? 2 : 3);
  const bool use_graph = h->loop_mode != BK_LOOP_STREAM;
  uint64_t key[6] = {1 /*cg*/, A->uid, (uint64_t)(uintptr_t)h->ws, (uint64_t)n,
                     (uint64_t)A->dtype | ((uint64_t)fuse << 8) | ((uint64_t)h->snake << 9) | ((uint64_t)(h->l2_hints & 31) << 10) | ((uint64_t)lag << 15) | ((uint64_t)chunk << 16),
                     (uint64_t)bk_grid_spmv(h) | ((uint64_t)bk_grid_vec(h) << 32)};
  auto enqueue_chunk = [&](cudaStream_t cs) -> int {
    for (int it = 0; it < chunk; ++it) BK_TRY(bk_cg_enqueue_iter<T>(h, A, v, it, fuse, lag, cs));
    return BK_OK;
  };
  int64_t chunks = 0;
  bool persistent = false;
  bk_call_mark(h, "loop");
  BK_TRY(bk_cg_try_persistent<T>(h, A, v.x, v.r, v.p[0], v.p[1], v.ap, s, &persistent));
  if (persistent) h->last_loop_mode = 3;
  if (!persistent) {
    if (persist_ok)  // cooperative launch unavailable after all: the unfused loop expects p = r0
      BK_CUDA(cudaMemcpyAsync(v.p[0], v.r, vbytes, cudaMemcpyDeviceToDevice, s));
    BK_TRY(bk_run_loop(h, s, use_graph, key, enqueue_chunk, &chunks));
  }

  bk_call_mark(h, "final");
  {  // final true residual  ||b - A x||  and  ||x||   (_isolve :1008-1013)
    bk_spmv_args a = bk_spmv_base(A, st);
    a.x = v.x;
    a.y = v.ap;
    a.b = b;
    bk_epi_final_r epi{st};
    BK_TRY((bk_launch_spmv<1, 2, 0>(h, A, a, bk_slot(h, 0), epi, s)));
    bk_epi_final_x epx{st};
    BK_TRY((bk_dot_epi<T>(h, n, v.x, v.x, epx, 1, s)));
  }
  BK_CUDA(cudaMemcpyAsync(x_user, v.x, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(&h->st_host[3], st, sizeof(bk_dev_state), cudaMemcpyDeviceToHost, s));
  bk_call_stop(h, s);
  BK_CUDA(cudaStreamSynchronize(s));
  const bk_dev_state* fin = &h->st_host[3];
  bk_fill_result_isolve(fin, res, fin->k + (has_x0 ? 1 : 0));
  res->rr_last = fin->gamma;
  res->kernel_launches = (persistent ? 1 : chunks * chunk * (fuse ? 2 : 3)) + 2 /*state, b.b*/ + (has_x0 ? 1 : 0) + 2 /*final*/;
  bk_call_finish(h, res);
  return BK_OK;
}

int bk_solver_args_check(const char* who, bk_handle* h, const bk_csr* A, const void* b, void* x, bk_result* res) {
  if (!h || !A || !res) return bk_fail(BK_ERR_ARG, "%s: null handle/matrix/result", who);
  if (A->n > 0 && (!b || !x)) return bk_fail(BK_ERR_ARG, "%s: null vector", who);
  if (A->h != h) return bk_fail(BK_ERR_ARG, "%s: matrix belongs to another handle", who);
  memset(res, 0, sizeof(*res));
  return BK_OK;
}

extern "C" int bk_cg(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol, double atol,
                     int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_cg", h, A, b, x, result));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  if (A->dtype == BK_F64) return bk_cg_t<double>(h, A, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
  return bk_cg_t<float>(h, A, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
}

// ---- Jacobi-preconditioned CG (SURVEY §8f-1: a built-in M so that preconditioning need not leave the device) ------
struct bk_epi_pcg_bs {  // bs = b.b ; atol2 (:815-817)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->bs = s[0];
    st->atol2 = fmax(st->tolsq32 * s[0], st->atolsq32);
  }
};
struct bk_epi_ignore {
  __device__ __forceinline__ void operator()(const double*) const {}
};
// Symmetric Gauss-Seidel CG (M = bk_sgs_run, z stored): K2 is the unpreconditioned bk_op_cg_r (r -= alpha Ap and the
// stop test on r.r, which it leaves in gamma); the r.z reduction after the sweeps then sets beta = r.z / rho and puts r.z
// into both rho and gamma, so the next SpMV's epilogue forms alpha = r.z / p.Ap.
struct bk_epi_sgs_rr0 {  // first stop test on r0.r0 (:841) — atol2 was set by the b.b reduction
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->rs = s[0];
    if (st->maxiter <= 0) {
      st->done = 1;
      st->status = BK_ST_MAXITER;
    }
    if (s[0] <= st->atol2) {
      st->done = 1;
      st->status = BK_ST_CONVERGED;
    }
  }
};
struct bk_epi_sgs_rz {  // init: gamma = r0.z0 ; in the loop: beta = r.z / rho, gamma = r.z   (:826, :850-851)
  bk_dev_state* st;
  int init;
  __device__ __forceinline__ void operator()(const double* s) const {
    if (!init) st->beta = s[0] / st->rho;
    st->rho = s[0];
    st->gamma = s[0];
  }
};

// Preconditioned CG.  M is either Jacobi (d = diag(A), S = nullptr: z = r / d formed on the fly inside the BLAS-1
// kernels) or symmetric Gauss-Seidel (S != nullptr, d unused: z = M r stored by the sweeps).
template <typename T, typename Sys>
static int bk_pcg_t(const Sys& sys, const T* d, const void* b, void* x_user, int has_x0, double tol,
                    double atol, int64_t maxiter, bk_result* res, cudaStream_t s, const bk_sgs* S = nullptr) {
  bk_handle* h = sys.h;
  const long long n = sys.n();
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  BK_TRY(bk_ws_reserve(h, (size_t)(S ? 5 : 4) * npad * sizeof(T)));
  T* x = (T*)h->ws;
  T* r = x + npad;
  T* p = r + npad;
  T* ap = p + npad;
  T* z = ap + npad;  // SGS only
  bk_dev_state* st = h->st;
  const size_t vbytes = (size_t)n * sizeof(T);
  bk_call_begin(h, s, S ? "bk_cg_sgs" : "bk_cg_jacobi");

  bk_dev_state init;
  memset(&init, 0, sizeof(init));
  init.maxiter = maxiter < 0 ? 10 * sys.n_global() : maxiter;
  init.status = BK_ST_MAXITER;
  bk_state_fill_tol(&init, tol, atol);
  bk_state_set_kernel<<<1, 1, 0, s>>>(st, init);
  BK_KERNEL_CHECK();

  BK_TRY((sys.template dot<T>(b, b, bk_epi_pcg_bs{st}, 1, s)));
  if (has_x0) {
    BK_CUDA(cudaMemcpyAsync(x, x_user, vbytes, cudaMemcpyDeviceToDevice, s));
    BK_TRY((sys.template matvec<T, 1, 2>(x, r, nullptr, b, 0, bk_epi_ignore{}, s)));  // r0 = b - A x0 (:820)
  } else {
    BK_CUDA(cudaMemsetAsync(x, 0, vbytes, s));
    BK_CUDA(cudaMemcpyAsync(r, b, vbytes, cudaMemcpyDeviceToDevice, s));
  }
  if (S) {  // z0 = M r0 ; p0 = z0 ; rho = r0.z0 ; the stop test on r0.r0
    BK_TRY(bk_sgs_run(h, S, r, z, 0, s));
    BK_CUDA(cudaMemcpyAsync(p, z, vbytes, cudaMemcpyDeviceToDevice, s));
    BK_TRY((sys.template dot<T>(r, r, bk_epi_sgs_rr0{st}, 1, s)));
    BK_TRY((sys.template dot<T>(r, z, bk_epi_sgs_rz{st, 1}, 1, s)));
  } else {
    bk_op_pcg_init<T> op;
    op.r = r;
    op.d = d;
    op.p = p;
    op.st = st;
    BK_TRY(sys.template ew<T>(op, bk_aligned16(d), 1, s));
  }
  const bool al = S ? true : bk_aligned16(d);
  auto enqueue_iter = [&](cudaStream_t cs) -> int {
    BK_TRY((sys.template matvec<T, 0, 1>(p, ap, p, nullptr, 1, bk_epi_cg_pAp{st}, cs)));
    if (S) {
      bk_op_cg_r<T> opr;
      opr.ap = ap;
      opr.r = r;
      opr.st = st;
      opr.snake = 0;
      BK_TRY(sys.template ew<T>(opr, true, 1, cs));
      BK_TRY(bk_sgs_run(h, S, r, z, 1, cs));
      bk_op_dot_epi<T, bk_epi_sgs_rz> opd;  // gamma = r.z in the fixed order of the grid reduction
      opd.x = r;
      opd.y = z;
      opd.epi = bk_epi_sgs_rz{st, 0};
      opd.st = st;
      opd.guard = 1;
      BK_TRY(sys.template ew<T>(opd, true, 1, cs));
      bk_op_cg_xp<T> opx;  // x += alpha p ; p = z + beta p
      opx.x = x;
      opx.p = p;
      opx.r = z;
      opx.st = st;
      opx.snake = 0;
      BK_TRY(sys.template ew<T>(opx, true, 2, cs));
      return BK_OK;
    }
    {
      bk_op_pcg_r<T> op;
      op.ap = ap;
      op.r = r;
      op.d = d;
      op.st = st;
      BK_TRY(sys.template ew<T>(op, al, 1, cs));
    }
    {
      bk_op_pcg_xp<T> op;
      op.x = x;
      op.p = p;
      op.r = r;
      op.d = d;
      op.st = st;
      BK_TRY(sys.template ew<T>(op, al, 2, cs));
    }
    return BK_OK;
  };
  const int kernels_iter = S ? 4 + bk_sgs_launches(S) : 3;
  const double bytes_iter = (S ? 3.0 : 1.0) * sys.matrix_bytes() + 13.0 * n * sizeof(T);
  const int chunk = bk_pick_chunk(h, bytes_iter, kernels_iter);
  const bool use_graph = h->loop_mode != BK_LOOP_STREAM;
  uint64_t key[6] = {S ? 6ull /*sgs cg*/ : 5ull /*jacobi cg*/, sys.uid(), (uint64_t)(uintptr_t)h->ws, (uint64_t)n,
                     (uint64_t)sys.dtype() | ((uint64_t)chunk << 16) | ((uint64_t)al << 8),
                     (uint64_t)bk_grid_spmv(h) | ((uint64_t)bk_grid_vec(h) << 32)};
  // the diagonal's address is baked into the captured graph: make it part of the key
  key[1] ^= (uint64_t)(uintptr_t)(S ? (const void*)S : (const void*)d) * 0x9e3779b97f4a7c15ull;
  auto enqueue_chunk = [&](cudaStream_t cs) -> int {
    for (int it = 0; it < chunk; ++it) BK_TRY(enqueue_iter(cs));
    return BK_OK;
  };
  int64_t chunks = 0;
  bk_call_mark(h, "loop");
  BK_TRY(bk_run_loop(h, s, use_graph, key, enqueue_chunk, &chunks));
  bk_call_mark(h, "final");

  // final check of _isolve: || M (b - A x) || against max(tol ||b||, atol) (:1008-1013)
  BK_TRY((sys.template matvec<T, 1, 2>(x, ap, nullptr, b, 0, bk_epi_ignore{}, s)));
  if (S) {
    BK_TRY(bk_sgs_run(h, S, ap, z, 0, s));
    BK_TRY((sys.template dot<T>(z, z, bk_epi_final_r{st}, 1, s)));
  } else {
    bk_op_scaled_sq<T, bk_epi_final_r> op;
    op.t = ap;
    op.d = d;
    op.epi = bk_epi_final_r{st};
    BK_TRY(sys.template ew<T>(op, al, 1, s));
  }
  BK_TRY((sys.template dot<T>(x, x, bk_epi_final_x{st}, 1, s)));
  BK_CUDA(cudaMemcpyAsync(x_user, x, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(&h->st_host[3], st, sizeof(bk_dev_state), cudaMemcpyDeviceToHost, s));
  bk_call_stop(h, s);
  BK_CUDA(cudaStreamSynchronize(s));
  const bk_dev_state* fin = &h->st_host[3];
  bk_fill_result_isolve(fin, res, fin->k + (has_x0 ? 1 : 0));
  if (S) {
    res->rr_last = fin->k > 0 ? fin->gamma : fin->rs;  // the loop's last K2 left r.r in gamma
    res->kernel_launches = chunks * chunk * kernels_iter + 4 + (has_x0 ? 1 : 0) + 2 * bk_sgs_launches(S) + 3;
  } else {
    res->rr_last = fin->rs;
    res->kernel_launches = chunks * chunk * 3 + 4 + (has_x0 ? 1 : 0) + 3;
  }
  bk_call_finish(h, res);
  return sys.check_comm(fin, S ? "cg_sgs" : "cg_jacobi");
}

extern "C" int bk_cg_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0,
                            double tol, double atol, int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_cg_jacobi", h, A, b, x, result));
  if (!diag && A->n > 0) return bk_fail(BK_ERR_ARG, "bk_cg_jacobi: null diagonal");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_pcg_t<double>(sys, (const double*)diag, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
  return bk_pcg_t<float>(sys, (const float*)diag, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
}

extern "C" int bk_cg_sgs(bk_handle* h, const bk_csr* A, const bk_sgs* S, const void* b, void* x, int has_x0,
                         double tol, double atol, int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_cg_sgs", h, A, b, x, result));
  BK_TRY(bk_sgs_args_check("bk_cg_sgs", h, A, S));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_pcg_t<double>(sys, nullptr, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream, S);
  return bk_pcg_t<float>(sys, nullptr, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream, S);
}

// diag[r] = A[r][r] (sum of the stored entries with col == r; 0 when the row has none)
template <typename T>
__global__ void bk_csr_diag_kernel(const int* __restrict__ rowptr, const int* __restrict__ col,
                                   const T* __restrict__ val, long long n, T* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
    T dsum = T(0);
    for (int k = rowptr[r]; k < rowptr[r + 1]; ++k)
      if (col[k] == (int)r) dsum += val[k];
    out[r] = dsum;
  }
}

extern "C" int bk_csr_diagonal(bk_handle* h, const bk_csr* A, void* out, void* stream) {
  if (!h || !A || (!out && A->n > 0)) return bk_fail(BK_ERR_ARG, "bk_csr_diagonal: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const int g = bk_grid_rows(h->num_sms * 8, A->n, 256);
  if (A->dtype == BK_F64)
    bk_csr_diag_kernel<double><<<g, 256, 0, (cudaStream_t)stream>>>(A->rowptr, A->col, (const double*)A->val, A->n,
                                                                    (double*)out);
  else
    bk_csr_diag_kernel<float><<<g, 256, 0, (cudaStream_t)stream>>>(A->rowptr, A->col, (const float*)A->val, A->n,
                                                                   (float*)out);
  BK_KERNEL_CHECK();
  return BK_OK;
}

// ---- row-partitioned CG (SURVEY §8e) --------------------------------------------------------------------------
// The 3-kernel iteration above on the distributed system: K1's halo exchange overlaps the local-block SpMV, p.Ap and
// r.r become global sums (peer path: inside the epilogues of the boundary-row kernel and of K2; NCCL path:
// ncclAllReduce + a one-thread scalar kernel each).
template <typename T>
static int bk_dist_cg_t(const bk_sys_dist& sys, const void* b, void* x_user, int has_x0, double tol, double atol,
                        int64_t maxiter, bk_result* res, cudaStream_t s) {
  bk_handle* h = sys.h;
  const long long n = sys.n();
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  BK_TRY(bk_ws_reserve(h, (size_t)5 * npad * sizeof(T)));
  T* x = (T*)h->ws;
  T* r = x + npad;
  T* p = r + npad;
  T* ap = p + npad;
  T* p2 = ap + npad;  // second p buffer of the lagged-x cut
  bk_dev_state* st = h->st;
  const size_t vbytes = (size_t)n * sizeof(T);
  bk_call_begin(h, s, "bk_dist_cg");

  bk_dev_state init;
  memset(&init, 0, sizeof(init));
  init.maxiter = maxiter < 0 ? 10 * sys.n_global() : maxiter;
  init.status = BK_ST_MAXITER;
  bk_state_fill_tol(&init, tol, atol);
  bk_state_set_kernel<<<1, 1, 0, s>>>(st, init);
  BK_KERNEL_CHECK();

  if (has_x0) {
    BK_CUDA(cudaMemcpyAsync(x, x_user, vbytes, cudaMemcpyDeviceToDevice, s));
    BK_TRY((sys.matvec<T, 1, 2>(x, r, nullptr, b, 0, bk_epi_set_gamma{st}, s)));  // r0 = b - A x0, gamma0 (:820, :826)
  } else {
    BK_CUDA(cudaMemsetAsync(x, 0, vbytes, s));
    BK_CUDA(cudaMemcpyAsync(r, b, vbytes, cudaMemcpyDeviceToDevice, s));
  }
  BK_TRY((sys.dot<T>(b, b, bk_epi_cg_init{st, has_x0}, 1, s)));
  BK_CUDA(cudaMemcpyAsync(p, r, vbytes, cudaMemcpyDeviceToDevice, s));
  // peer path on slab-like partitions: K3 itself pushes the new p into the neighbours (no push kernel in the loop);
  // p0 goes out here, guarded so that a solve that ends before its first iteration pushes nothing
  const bool fuse_push = sys.can_fuse_push() && h->dist_fuse_push;
  if (fuse_push) BK_TRY(sys.halo_begin<T>(p, 1, true, s));

  // lagged-x cut (see bk_op_cg_p_lag): x is updated every second iteration, p ping-pongs between p and p2
  const bool lag = fuse_push && h->cg_lag_x != 0;
  auto enqueue_iter = [&](int it, cudaStream_t cs) -> int {
    T* pcur = (lag && (it & 1)) ? p2 : p;
    T* pnext = (lag && !(it & 1)) ? p2 : p;
    BK_TRY((sys.matvec<T, 0, 1>(pcur, ap, pcur, nullptr, 1, bk_epi_cg_pAp{st}, cs, fuse_push)));
    {
      bk_op_cg_r<T> op;
      op.ap = ap;
      op.r = r;
      op.st = st;
      op.snake = sys.snake ? 1 : 0;
      BK_TRY(sys.ew<T>(op, true, 1, cs));
    }
    if (fuse_push) {
      BK_TRY(sys.cg_xp_push<T>(x, pcur, pnext, r, lag ? 1 + (it & 1) : 0, cs));
    } else {
      bk_op_cg_xp<T> op;
      op.x = x;
      op.p = p;
      op.r = r;
      op.st = st;
      op.snake = sys.snake ? 1 : 0;
      BK_TRY(sys.ew<T>(op, true, 2, cs));
    }
    return BK_OK;
  };
  const double bytes_iter = sys.matrix_bytes() + 11.0 * n * sizeof(T);
  const int chunk = bk_pick_chunk(h, bytes_iter, 8);
  const bool use_graph = h->loop_mode != BK_LOOP_STREAM;  // NCCL calls are captured into the iteration graph too
  uint64_t key[6] = {4 /*dist cg*/, sys.uid(), (uint64_t)(uintptr_t)h->ws, (uint64_t)n,
                     (uint64_t)sys.dtype() | ((uint64_t)fuse_push << 8) | ((uint64_t)sys.snake << 9) | ((uint64_t)lag << 10) | ((uint64_t)chunk << 16),
                     (uint64_t)bk_grid_spmv(h) | ((uint64_t)bk_grid_vec(h) << 32)};
  auto enqueue_chunk = [&](cudaStream_t cs) -> int {
    for (int it = 0; it < chunk; ++it) BK_TRY(enqueue_iter(it, cs));
    return BK_OK;
  };
  int64_t chunks = 0;
  bk_call_mark(h, "loop");
  BK_TRY(bk_run_loop(h, s, use_graph, key, enqueue_chunk, &chunks));
  bk_call_mark(h, "final");

  // final true residual and ||x|| (global)
  BK_TRY((sys.matvec<T, 1, 2>(x, ap, nullptr, b, 0, bk_epi_final_r{st}, s)));
  BK_TRY((sys.dot<T>(x, x, bk_epi_final_x{st}, 1, s)));
  BK_CUDA(cudaMemcpyAsync(x_user, x, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(&h->st_host[3], st, sizeof(bk_dev_state), cudaMemcpyDeviceToHost, s));
  bk_call_stop(h, s);
  BK_CUDA(cudaStreamSynchronize(s));
  const bk_dev_state* fin = &h->st_host[3];
  bk_fill_result_isolve(fin, res, fin->k + (has_x0 ? 1 : 0));
  res->rr_last = fin->gamma;
  res->kernel_launches = chunks * chunk * (sys.p2p ? (fuse_push ? 4 : 5) : 7) + 12;
  bk_call_finish(h, res);
  return sys.check_comm(fin, "bk_dist_cg");
}

extern "C" int bk_dist_cg(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol,
                          double atol, int64_t maxiter, int64_t n_global, bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_cg: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local)) return bk_fail(BK_ERR_ARG, "bk_dist_cg: null vector");
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global, h->snake != 0};
  if (D->dtype == BK_F64)
    return bk_dist_cg_t<double>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
  return bk_dist_cg_t<float>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
}

extern "C" int bk_dist_cg_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local, void* x_local,
                                 int has_x0, double tol, double atol, int64_t maxiter, int64_t n_global,
                                 bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_cg_jacobi: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local || !diag_local)) return bk_fail(BK_ERR_ARG, "bk_dist_cg_jacobi: null vector");
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global, false};
  if (D->dtype == BK_F64)
    return bk_pcg_t<double>(sys, (const double*)diag_local, b_local, x_local, has_x0, tol, atol, maxiter, result,
                            (cudaStream_t)stream);
  return bk_pcg_t<float>(sys, (const float*)diag_local, b_local, x_local, has_x0, tol, atol, maxiter, result,
                         (cudaStream_t)stream);
}
