// bk_bicgstab.cu — BiCGStab with a device-resident loop.
// Replaces _bicgstab_solve (reference torch_sparse_linalg.py:859-964) + _isolve (:967-1016).
//
// Per iteration (the reference's recurrences, operation order and breakdown tests):
//   K1  p = r + beta (p - omega q)                                              (:906-907)
//   K2  q = A p  fused with rhat.q ; epilogue alpha = rho'/(rhat.q), |alpha| < eps -> -11  (:909-915)
//   K3  s = r - alpha q  fused with s.s ; epilogue exit_early = s.s < atol2      (:917-920)
//   K4  t = A s  fused with t.s, t.t ; epilogue omega (guarded), omega breakdown -> -11 (:923-936)
//       (skipped when exit_early: neither x nor r depends on t then — SURVEY compatibility ledger)
//   K5  x += alpha p (+ omega s) ; r = s (- omega t)  fused with r.r and rhat.r ; epilogue: k += 1,
//       stop tests of the next iteration (:893-904), beta                         (:942-962)
// The reference pays 5 host syncs per iteration for these tests; here there are none.
// Algorithmic HBM bytes per iteration: 2*[nnz*(8+4) + (n+1)*4] + 19*n*8  (SURVEY §8d).
#include "bk_internal.cuh"
#include "bk_loop.cuh"
#include "bk_spmv.cuh"
#include "bk_sys.cuh"
#include "bk_dist.cuh"
#include "bk_vec.cuh"
#include "bk_bicgstab_persist.cuh"

template <typename T>
struct bk_eps_of {
  static constexpr double value = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
};

template <typename T>
struct bk_epi_bicg_alpha {  // alpha = rho' / (rhat . q)
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    st->rhat_q = s[0];
    const double alpha = st->rho_new / s[0];
    st->alpha = alpha;
    if (fabs(alpha) < bk_eps_of<T>::value) {
      st->done = 1;
      st->status = BK_ST_BREAKDOWN_AW;
    }
  }
};

template <typename T>
struct bk_epi_bicg_omega {  // sums: [0] t.s  [1] t.t
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const {
    const double eps = bk_eps_of<T>::value;
    const double omega = (fabs(s[1]) < eps) ? 0.0 : s[0] / s[1];
    st->omega = omega;
    if (fabs(omega) < eps && !st->exit_early) {
      st->done = 1;
      st->status = BK_ST_BREAKDOWN_AW;
    }
  }
};

// top-of-loop tests of iteration 0 from r0.r0 (rhat = r0 so rho' = r0.r0); rho = alpha = omega = 1 (:884-890)
template <typename T>
struct bk_epi_bicg_init {
  bk_dev_state* st;
  int has_x0;
  __device__ __forceinline__ void operator()(const double* s) const {
    // called from the b.b reduction; r0.r0 already sits in st->rs when has_x0, else equals b.b
    const double bs = s[0];
    st->bs = bs;
    st->atol2 = fmax(st->tolsq32 * bs, st->atolsq32);
    if (!has_x0) st->rs = bs;
    const double rs = st->rs;
    st->rho = 1.0;
    st->alpha = 1.0;
    st->omega = 1.0;
    st->rho_new = rs;
    if (st->maxiter <= 0) {
      st->done = 1;
      st->status = BK_ST_MAXITER;
      return;
    }
    if (rs <= st->atol2) {
      st->done = 1;
      st->status = BK_ST_CONVERGED;
      return;
    }
    if (fabs(rs) < bk_eps_of<T>::value * 1.0) {
      st->done = 1;
      st->status = BK_ST_BREAKDOWN_RHO;
      return;
    }
    st->beta = rs / 1.0 * 1.0 / 1.0;
  }
};

struct bk_epi_set_rs {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->rs = s[0]; }
};
struct bk_epi_final_r2 {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->rtrue2 = s[0]; }
};
struct bk_epi_final_x2 {
  bk_dev_state* st;
  __device__ __forceinline__ void operator()(const double* s) const { st->xx = s[0]; }
};

template <typename T>
struct bk_bicg_vecs {
  T *x, *r, *rhat, *p, *q, *s, *t;
  T *phat, *shat;  // Jacobi: the preconditioned copies the SpMVs gather from
  const T* d;      // Jacobi: diag(A); nullptr = unpreconditioned
  const bk_sgs* S; // symmetric Gauss-Seidel: phat = M p, shat = M s by the sweeps (d unused)
};

template <typename T, typename Sys>
static int bk_bicg_enqueue_iter(const Sys& sys, const bk_bicg_vecs<T>& v, cudaStream_t s) {
  bk_dev_state* st = sys.h->st;
  const bool jac = v.d != nullptr;
  const bool pc = jac || v.S;
  const bool al = !jac || bk_aligned16(v.d);
  if (jac) {
    bk_op_bicg_p_pc<T> op;
    op.r = v.r;
    op.p = v.p;
    op.q = v.q;
    op.st = st;
    op.d = v.d;
    op.phat = v.phat;
    BK_TRY(sys.template ew<T>(op, al, 2, s));
  } else {
    bk_op_bicg_p<T> op;
    op.r = v.r;
    op.p = v.p;
    op.q = v.q;
    op.st = st;
    BK_TRY(sys.template ew<T>(op, true, 2, s));
    if (v.S) BK_TRY(bk_sgs_run(sys.h, v.S, v.p, v.phat, 1, s));
  }
  BK_TRY((sys.template matvec<T, 0, 1>(pc ? v.phat : v.p, v.q, v.rhat, nullptr, 1, bk_epi_bicg_alpha<T>{st}, s)));
  if (jac) {
    bk_op_bicg_s_pc<T> op;
    op.r = v.r;
    op.q = v.q;
    op.s = v.s;
    op.st = st;
    op.d = v.d;
    op.shat = v.shat;
    BK_TRY(sys.template ew<T>(op, al, 1, s));
  } else {
    bk_op_bicg_s<T> op;
    op.r = v.r;
    op.q = v.q;
    op.s = v.s;
    op.st = st;
    BK_TRY(sys.template ew<T>(op, true, 1, s));
    if (v.S) BK_TRY(bk_sgs_run(sys.h, v.S, v.s, v.shat, 3, s));
  }
  // t = A shat ; the dots are t.s and t.t with the UNpreconditioned s (:926-930)
  BK_TRY((sys.template matvec<T, 0, 3>(pc ? v.shat : v.s, v.t, v.s, nullptr, 3, bk_epi_bicg_omega<T>{st}, s)));
  if (pc) {
    bk_op_bicg_xr_pc<T> op;
    op.x = v.x;
    op.p = v.phat;
    op.s = v.s;
    op.t = v.t;
    op.rhat = v.rhat;
    op.r = v.r;
    op.st = st;
    op.shat = v.shat;
    BK_TRY(sys.template ew<T>(op, true, 1, s));
  } else {
    bk_op_bicg_xr<T> op;
    op.x = v.x;
    op.p = v.p;
    op.s = v.s;
    op.t = v.t;
    op.rhat = v.rhat;
    op.r = v.r;
    op.st = st;
    BK_TRY(sys.template ew<T>(op, true, 1, s));
  }
  return BK_OK;
}

template <typename T, typename Sys>
static int bk_bicgstab_t(const Sys& sys, const void* b, void* x_user, int has_x0, double tol, double atol,
                         int64_t maxiter, bk_result* res, cudaStream_t s, const T* diag = nullptr,
                         const bk_sgs* S = nullptr) {
  bk_handle* h = sys.h;
  const long long n = sys.n();
  const size_t npad = ((size_t)n + 63) & ~(size_t)63;
  BK_TRY(bk_ws_reserve(h, (size_t)9 * npad * sizeof(T)));
  bk_bicg_vecs<T> v;
  v.x = (T*)h->ws;
  v.r = v.x + npad;
  v.rhat = v.r + npad;
  v.p = v.rhat + npad;
  v.q = v.p + npad;
  v.s = v.q + npad;
  v.t = v.s + npad;
  v.phat = v.t + npad;
  v.shat = v.phat + npad;
  v.d = diag;
  v.S = S;
  bk_dev_state* st = h->st;
  const size_t vbytes = (size_t)n * sizeof(T);
  bk_call_begin(h, s, "bk_bicgstab");

  bk_dev_state init;
  memset(&init, 0, sizeof(init));
  init.maxiter = maxiter < 0 ? 10 * sys.n_global() : maxiter;
  init.status = BK_ST_MAXITER;
  bk_state_fill_tol(&init, tol, atol);
  bk_state_set_kernel<<<1, 1, 0, s>>>(st, init);
  BK_KERNEL_CHECK();

  if (has_x0) {
    BK_CUDA(cudaMemcpyAsync(v.x, x_user, vbytes, cudaMemcpyDeviceToDevice, s));
    // r0 = b - A x0 ; rs = r0.r0   (:875)
    BK_TRY((sys.template matvec<T, 1, 2>(v.x, v.r, nullptr, b, 0, bk_epi_set_rs{st}, s)));
  } else {
    BK_CUDA(cudaMemsetAsync(v.x, 0, vbytes, s));
    BK_CUDA(cudaMemcpyAsync(v.r, b, vbytes, cudaMemcpyDeviceToDevice, s));
  }
  BK_TRY((sys.template dot<T>(b, b, bk_epi_bicg_init<T>{st, has_x0}, 1, s)));
  // rhat = p = q = r0   (:876, :890)
  BK_CUDA(cudaMemcpyAsync(v.rhat, v.r, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(v.p, v.r, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(v.q, v.r, vbytes, cudaMemcpyDeviceToDevice, s));

  const int kernels_iter = 5 + (S ? 2 * bk_sgs_launches(S) : 0);
  const double bytes_iter = (S ? 6.0 : 2.0) * sys.matrix_bytes() + (diag || S ? 25.0 : 19.0) * n * sizeof(T);
  const int chunk = bk_pick_chunk(h, bytes_iter, kernels_iter);
  const bool use_graph = h->loop_mode != BK_LOOP_STREAM;
  uint64_t key[6] = {2 /*bicgstab*/, sys.uid(), (uint64_t)(uintptr_t)h->ws, (uint64_t)n,
                     (uint64_t)sys.dtype() | ((uint64_t)chunk << 16),
                     (uint64_t)bk_grid_spmv(h) | ((uint64_t)bk_grid_vec(h) << 32)};
  if (diag) key[1] ^= (uint64_t)(uintptr_t)diag * 0x9e3779b97f4a7c15ull;  // its address is baked into the graph
  if (S) key[1] ^= (uint64_t)(uintptr_t)S * 0xc2b2ae3d27d4eb4full;
  auto enqueue_chunk = [&](cudaStream_t cs) -> int {
    for (int it = 0; it < chunk; ++it) BK_TRY((bk_bicg_enqueue_iter<T, Sys>(sys, v, cs)));
    return BK_OK;
  };
  int64_t chunks = 0;
  bk_call_mark(h, "loop");
  bool persistent = false;
  if constexpr (!Sys::kDist) {
    // launch-bound (L2-resident) systems: the whole loop in ONE persistent kernel (bk_bicgstab_persist.cuh);
    // phat / shat (unused without a preconditioner) serve as the second p / q buffers
    const bk_csr* A = sys.A;
    if (diag == nullptr && S == nullptr && A->rowptr && A->col) {
      bk_bp_args ga;
      ga.rowptr = A->rowptr;
      ga.col = A->col;
      ga.val = A->val;
      ga.n = n;
      ga.x = v.x;
      ga.r = v.r;
      ga.rhat = v.rhat;
      ga.p0 = v.p;
      ga.p1 = v.phat;
      ga.q0 = v.q;
      ga.q1 = v.shat;
      ga.s = v.s;
      ga.t = v.t;
      ga.st = st;
      ga.partials = h->partials;
      BK_TRY(bk_launch_persistent(h, bk_bicgstab_persistent_kernel<T, true>, bk_bicgstab_persistent_kernel<T, false>, ga,
                                  n, s, &persistent));
    }
  }
  if (!persistent) BK_TRY(bk_run_loop(h, s, use_graph, key, enqueue_chunk, &chunks));
  bk_call_mark(h, "final");

  BK_TRY((sys.template matvec<T, 1, 2>(v.x, v.t, nullptr, b, 0, bk_epi_final_r2{st}, s)));
  if (diag) {  // _isolve checks || M (b - A x) || (:1008)
    bk_op_scaled_sq<T, bk_epi_final_r2> op;
    op.t = v.t;
    op.d = diag;
    op.epi = bk_epi_final_r2{st};
    BK_TRY(sys.template ew<T>(op, bk_aligned16(diag), 1, s));
  }
  if (S) {
    BK_TRY(bk_sgs_run(h, S, v.t, v.phat, 0, s));
    BK_TRY((sys.template dot<T>(v.phat, v.phat, bk_epi_final_r2{st}, 1, s)));
  }
  BK_TRY((sys.template dot<T>(v.x, v.x, bk_epi_final_x2{st}, 1, s)));
  BK_CUDA(cudaMemcpyAsync(x_user, v.x, vbytes, cudaMemcpyDeviceToDevice, s));
  BK_CUDA(cudaMemcpyAsync(&h->st_host[3], st, sizeof(bk_dev_state), cudaMemcpyDeviceToHost, s));
  bk_call_stop(h, s);
  BK_CUDA(cudaStreamSynchronize(s));
  const bk_dev_state* fin = &h->st_host[3];
  bk_fill_result_isolve(fin, res, 2 * fin->k + (has_x0 ? 1 : 0));
  res->rr_last = fin->rs;
  res->kernel_launches = (persistent ? 1 : chunks * chunk * kernels_iter) + 2 + (has_x0 ? 1 : 0) + 2 +
                         (S ? bk_sgs_launches(S) + 1 : 0);
  bk_call_finish(h, res);
  return sys.check_comm(fin, "bicgstab");
}

extern "C" int bk_bicgstab(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol, double atol,
                           int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_bicgstab", h, A, b, x, result));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_bicgstab_t<double>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
  return bk_bicgstab_t<float>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
}

/* BiCGStab with the built-in Jacobi preconditioner (right preconditioning, _bicgstab_solve :907-946 with
 * M = (v -> v / diag)); see bk_cg_jacobi. */
extern "C" int bk_bicgstab_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0,
                                  double tol, double atol, int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_bicgstab_jacobi", h, A, b, x, result));
  if (!diag && A->n > 0) return bk_fail(BK_ERR_ARG, "bk_bicgstab_jacobi: null diagonal");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_bicgstab_t<double>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream,
                                 (const double*)diag);
  return bk_bicgstab_t<float>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream,
                              (const float*)diag);
}

/* BiCGStab with the built-in symmetric Gauss-Seidel preconditioner: the right preconditioning of bk_bicgstab_jacobi
 * with phat = M p and shat = M s computed by the sweeps. */
extern "C" int bk_bicgstab_sgs(bk_handle* h, const bk_csr* A, const bk_sgs* S, const void* b, void* x, int has_x0,
                               double tol, double atol, int64_t maxiter, bk_result* result, void* stream) {
  BK_TRY(bk_solver_args_check("bk_bicgstab_sgs", h, A, b, x, result));
  BK_TRY(bk_sgs_args_check("bk_bicgstab_sgs", h, A, S));
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  const bk_sys_local sys{h, A};
  if (A->dtype == BK_F64)
    return bk_bicgstab_t<double>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream, nullptr, S);
  return bk_bicgstab_t<float>(sys, b, x, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream, nullptr, S);
}

// Row-partitioned BiCGStab: same driver, every reduction made global (SURVEY §8e: "BiCGStab: 3 allreduce points").
extern "C" int bk_dist_bicgstab(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol,
                                double atol, int64_t maxiter, int64_t n_global, bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_bicgstab: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local)) return bk_fail(BK_ERR_ARG, "bk_dist_bicgstab: null vector");
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global};
  if (D->dtype == BK_F64)
    return bk_bicgstab_t<double>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
  return bk_bicgstab_t<float>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream);
}

extern "C" int bk_dist_bicgstab_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local,
                                       void* x_local, int has_x0, double tol, double atol, int64_t maxiter,
                                       int64_t n_global, bk_result* result, void* stream) {
  if (!h || !D || !result) return bk_fail(BK_ERR_ARG, "bk_dist_bicgstab_jacobi: null handle/matrix/result");
  if (D->n_local > 0 && (!b_local || !x_local || !diag_local))
    return bk_fail(BK_ERR_ARG, "bk_dist_bicgstab_jacobi: null vector");
  memset(result, 0, sizeof(*result));
  BK_CUDA(cudaSetDevice(h->device));
  const bk_sys_dist sys{h, D, D->p2p_enabled && h->dist_p2p, n_global};
  if (D->dtype == BK_F64)
    return bk_bicgstab_t<double>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream,
                                 (const double*)diag_local);
  return bk_bicgstab_t<float>(sys, b_local, x_local, has_x0, tol, atol, maxiter, result, (cudaStream_t)stream,
                              (const float*)diag_local);
}
