/*
 * bk_krylov.h — C ABI of the B200-native Krylov inner loop (libbk_krylov.so).
 *
 * This is the drop-in boundary underneath the reference's Python API
 * (pytorch_sparse_solver.module_a.cg / bicgstab / gmres).  The reference has no
 * native boundary of its own (it is 100 % Python on torch ops), so every entry
 * point below cites the reference *Python* function whose per-iteration work it
 * replaces (paths relative to the reference checkout,
 * src/pytorch_sparse_solver/module_a/torch_sparse_linalg.py unless noted).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every function returns 0 on success or a negative bk_error code and never
 *     throws; bk_last_error() returns a human-readable message for the calling
 *     thread's last failure.
 *   - "device pointer" arguments are borrowed for the duration of the call,
 *     except the three CSR arrays given to bk_csr_create with copy==0, which
 *     must stay alive until bk_csr_destroy.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *     All work is enqueued on it; solver entry points synchronise that stream
 *     once, at the end, to hand back bk_result (the reference's `info` is a
 *     Python int, so one sync per solve is part of its contract).
 *   - a bk_handle is bound to one CUDA device and is not thread-safe.
 *   - there is NO CPU fallback anywhere in this library.
 */
#ifndef BK_KRYLOV_H
#define BK_KRYLOV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BK_VERSION 200 /* 0.2.0 */

typedef struct bk_handle bk_handle; /* per-device context: scratch, workspaces, graph cache */
typedef struct bk_csr bk_csr;       /* a registered CSR matrix + its kernel plan */
typedef struct bk_dist bk_dist;     /* row-partitioned (multi-GPU) matrix + halo plan */
typedef struct bk_sgs bk_sgs;       /* multicolor symmetric Gauss-Seidel preconditioner of a registered matrix */

enum bk_error {
  BK_OK = 0,
  BK_ERR_ARG = -1,         /* invalid argument (message says which) */
  BK_ERR_CUDA = -2,        /* a CUDA runtime call failed */
  BK_ERR_ALLOC = -3,       /* device or host allocation failed */
  BK_ERR_UNSUPPORTED = -4, /* valid request this build cannot serve */
  BK_ERR_NCCL = -5         /* NCCL missing or a collective failed */
};

enum bk_dtype { BK_F64 = 0, BK_F32 = 1 };

/* Device-side loop status, reported in bk_result.status.  The breakdown codes
 * are the reference's own (k = -10 / -11 at :903, :914, :935). */
enum bk_status {
  BK_ST_CONVERGED = 0,       /* recurrence residual met the stop test */
  BK_ST_MAXITER = 1,         /* maxiter reached */
  BK_ST_BREAKDOWN_RHO = -10, /* BiCGStab |rho'| < eps |rho|            (:902-904) */
  BK_ST_BREAKDOWN_AW = -11   /* BiCGStab alpha or omega breakdown      (:913-915, :934-936) */
};

enum bk_gmres_method { BK_GMRES_BATCHED = 0, BK_GMRES_INCREMENTAL = 1 };

/* How the iteration loop is driven (all variants keep the stop test on the device). */
enum bk_loop_mode {
  BK_LOOP_AUTO = 0,
  BK_LOOP_STREAM = 1, /* plain stream launches, flag polled every `chunk` iterations */
  BK_LOOP_GRAPH = 2   /* CUDA graph of `chunk` flag-guarded iterations, polled per graph launch */
};

typedef struct bk_result {
  int64_t iterations;    /* CG/BiCGStab: iterations done; GMRES: restart cycles done */
  int64_t matvecs;       /* SpMV launches that did work (excludes the final check) */
  int64_t kernel_launches; /* kernels of this library enqueued by the call (graph nodes included; guarded
                            no-op launches after convergence included) */
  int32_t info;          /* the reference's `info`: 0 = final TRUE residual within tolerance, -1 otherwise
                            (_isolve :1008-1016, gmres :766-773) */
  int32_t status;        /* enum bk_status */
  double final_residual; /* || b - A x ||_2, recomputed from scratch */
  double threshold;      /* what final_residual was compared against */
  double b_norm;         /* || b ||_2 */
  double x_norm;         /* || x ||_2 (NaN check of the reference) */
  double rr_last;        /* last recurrence value: CG gamma = r.r, BiCGStab r.r, GMRES residual norm */
  int32_t loop_mode_used;/* how the iteration loop actually ran: 1 plain stream launches, 2 CUDA graph of chunks,
                            3 one persistent cooperative kernel (a failed graph capture shows up here as 1) */
  int32_t reserved0;
  double device_ms;      /* device time of the whole call (CUDA events on `stream`: set-up, loop, final check) */
} bk_result;

typedef struct bk_csr_info {
  int64_t n, nnz;
  int32_t dtype;        /* enum bk_dtype */
  int32_t kernel;       /* 0 row-stream (LDG-staged) | 1 sub-warp vector | 2 row-stream, TMA-staged tiles, int32 columns |
                           3 = 2 with 8-bit dictionary-coded columns | 4 long rows split into virtual rows (skewed
                           matrices) + ordered per-row reduction | 5 = 2 with 8-bit codes of (column - row, value)
                           PAIRS and no value stream (constant-coefficient stencils; lossless, bit-identical) |
                           6 = one presence BITMASK per row over its 32-row chunk's pattern of (column - row, value)
                           pairs; the pattern lives in registers (stencils with <= 8 pairs per chunk; bit-identical) |
                           7 = kernel 6's plan served by the stencil fast path: every pattern is a sub-pattern of one
                           offset set (7-point 3-D / 5-point 2-D), a lane owns two rows and gathers with 128-bit
                           loads, offsets and values are constant-bank operands, one summary per 64 rows replaces the
                           mask bytes of complete rows (fp64; bit-identical) */
  int32_t lanes_per_row;/* for kernel 1 */
  int32_t max_row_nnz;
  double mean_row_nnz;
  int64_t bytes_matrix; /* ALGORITHMIC bytes one SpMV reads for the matrix: nnz*(sizeof val + 4) + (n+1)*4 (CSR, int32) */
  int64_t bytes_stream; /* ACTUAL matrix-side bytes the selected kernel streams per SpMV (coded streams, dictionaries,
                           headers, row pointers ... counted at registration; equals bytes_matrix for kernels 0/1/2) */
} bk_csr_info;

/* ---- library / handle ------------------------------------------------------------ */
int bk_version(void);
const char* bk_last_error(void);
/* device: CUDA ordinal.  The handle owns reduction scratch (fixed slots => bitwise
 * reproducible sums), solver work vectors and cached CUDA graphs. */
int bk_create(int device, bk_handle** out);
int bk_destroy(bk_handle* h);
/* Tunables (all also readable from the environment at bk_create, BK_<UPPERCASE KEY>; unknown keys -> BK_ERR_ARG):
 *   loop_mode      0 auto (= graph) | 1 plain stream launches | 2 CUDA graph of `chunk` flag-guarded iterations
 *   chunk          iterations per graph / poll (0 = sized for ~2 ms of GPU work)
 *   use_tma        1: short-row matrices use the TMA-staged row-stream SpMV (kernel 2/3), 0: LDG-staged (kernel 0)
 *   dist_fuse_push 1: multi-GPU CG on the peer path folds the halo push into the p-update kernel when the partition allows it
 *   use_split      1: matrices with a short mean row but a few very long rows are run on a virtual-row view (kernel 4)
 *   use_compress   0: off | 1: stream column indices as 8-bit dictionary codes when the matrix allows it (kernel 3)
 *                  | 2 (default): first try 8-bit codes of (column - row, value) pairs (kernel 5), then kernel 3
 *                  | 3: first the row-bitmask plan (kernels 6 / 7)
 *   mask_const     1 (default): matrices that qualify run kernel 7 instead of kernel 6;  mask_cctas: its CTAs per SM (4..6)
 *   cg_lag_x       1 (default): CG on large systems updates x every second iteration with both pending terms (bit-identical)
 *   tma_ctas       CTAs per SM of the TMA SpMV (2..4), tma_stages: cap on its pipeline depth (0 = fill shared memory)
 *   prefetch_x     kernel 3: L2 bulk prefetch of the forward-diagonal x ranges (experiment, default 0)
 *   grid_mult_vec / grid_mult_spmv   CTAs per SM of the BLAS-1 kernels / the non-TMA SpMV kernels
 *   fuse_xpay      CG: fold p = r + beta p into the next SpMV's gather (-1 auto: only for launch-bound small systems)
 *   snake          CG: alternate the sweep direction of consecutive kernels so the tail of one is still in L2
 *   persistent     CG: run systems with n <= persistent_max_n (200000) in one cooperative persistent kernel
 *   dist_p2p       multi-GPU: use the peer-memory path when it is connected (0 = NCCL path)
 * Registration-time options (use_tma, use_compress, use_split) apply to matrices registered afterwards. */
int bk_set_option(bk_handle* h, const char* key, int64_t value);
int64_t bk_get_option(bk_handle* h, const char* key);
int bk_device_info(bk_handle* h, int32_t* num_sms, int64_t* l2_bytes, int64_t* mem_bytes);

/* ---- matrix registration ----------------------------------------------------------
 * Replaces: _normalize_matvec :176-208 (tensor branch; torch.matmul(CSR, v) at :191).
 * rowptr/col: device arrays of int32 (idx_bits=32) or int64 (idx_bits=64, converted to an
 * internal int32 copy; n and nnz must be < 2^31).  val: device array of `dtype`.
 * copy != 0 makes the library keep private copies of all three arrays. */
int bk_csr_create(bk_handle* h, int64_t n, int64_t nnz, const void* rowptr, const void* col,
                  int idx_bits, const void* val, int dtype, int copy, void* stream, bk_csr** out);
int bk_csr_destroy(bk_csr* A);
/* Other layouts -> the library's CSR, on the device, with the library owning all arrays (SURVEY section 8f-2: the
 * reference's tests and LDC example pass DENSE matrices to _normalize_matvec, torch_sparse_linalg.py:176-208).
 * bk_csr_from_dense: row-major n x n device matrix, row stride `ld` elements; entries != 0 are kept, columns ascending
 *   (the structure of torch's A.to_sparse_csr()).  Two passes over the matrix: count, ordered compaction.
 * bk_csr_from_coo: device triplets (rows, cols: int32 or int64 per idx_bits; vals), any order, duplicates allowed:
 *   stably sorted by (row, col) and equal positions summed in input order (torch's coalesce()).
 * in_dtype: dtype of the given values; dtype: dtype of the registered matrix (fp32 inputs may be widened). */
int bk_csr_from_dense(bk_handle* h, int64_t n, const void* dense, int64_t ld, int in_dtype, int dtype, void* stream,
                      bk_csr** out);
int bk_csr_from_coo(bk_handle* h, int64_t n, int64_t nnz, const void* rows, const void* cols, int idx_bits,
                    const void* val, int in_dtype, int dtype, void* stream, bk_csr** out);
int bk_csr_get_info(const bk_csr* A, bk_csr_info* out);
/* Cached transpose (CSC of A == CSR of A^T) built on the device by a stable LSD radix
 * sort on the column index — deterministic.  Replaces `A_matrix.T` in
 * ImplicitAdjointFunction.backward :1245 (which raises for CSR on torch 2.11).
 * The returned matrix is owned by A and freed with it. */
int bk_csr_transpose(bk_handle* h, bk_csr* A, void* stream, bk_csr** out);
/* out_vals[k] = -g[row(k)] * x[col[k]] for every stored entry k: the gradient of a loss with respect to the
 * entries of A on its sparsity pattern, given g = A^-T dL/dx (the adjoint solve) and the solution x.
 * No reference counterpart in Module A (it returns None for A, :1248); SURVEY §8f-3. */
int bk_csr_grad_pattern(bk_handle* h, const bk_csr* A, const void* g, const void* x, void* out_vals, void* stream);
/* 64-bit position-dependent checksum of `nbytes` of device memory (nbytes % 4 == 0), written to *out_host after a
 * stream synchronisation.  Integer arithmetic only => deterministic.  The Python front end uses it to validate a cached
 * registration of a BORROWED value array: torch gives no reliable way to notice that a user updated `vals` in place
 * (the wrapper's version counter does not move), and a stale pair dictionary would silently solve the wrong system. */
int bk_checksum(bk_handle* h, const void* data, int64_t nbytes, void* stream, uint64_t* out_host);
/* Export the arrays of a registered matrix (int32 rowptr/col): device pointers, borrowed. */
int bk_csr_arrays(const bk_csr* A, const void** rowptr, const void** col, const void** val);

/* ---- building blocks (deterministic; also used by the callable-A route) ------------
 * y = A x                                         (matrix_mv :185-205)            */
int bk_spmv(bk_handle* h, const bk_csr* A, const void* x, void* y, void* stream);
/* y = A x and *dot_out(device, fp64) = w . y      (SpMV fused with p.Ap, _cg_solve :844-845) */
int bk_spmv_dot(bk_handle* h, const bk_csr* A, const void* x, void* y, const void* w,
                double* dot_out, void* stream);
/* *out(device, fp64) = x . y                      (_vdot :86-91, _vdot_real_part :100-127) */
int bk_dot(bk_handle* h, int64_t n, int dtype, const void* x, const void* y, double* out, void* stream);
/* *out(device, fp64) = sqrt(max(x.x, 0))          (_norm :154-162) */
int bk_nrm2(bk_handle* h, int64_t n, int dtype, const void* x, double* out, void* stream);
/* z = a x + b y  (z may alias x or y)             (_add/_sub/_mul :165-173) */
int bk_axpby(bk_handle* h, int64_t n, int dtype, double a, const void* x, double b, const void* y,
             void* z, void* stream);
/* z = (sa * *a_dev) x + (sb * *b_dev) y with the scalars read from DEVICE memory (fp64; a null pointer stands for 1):
 * the callable-A route keeps alpha / beta of _cg_solve (:845, :851) on the device, one host sync per iteration
 * (the stop test, as in the reference :841) instead of one per dot product. */
int bk_axpby_dev(bk_handle* h, int64_t n, int dtype, double sa, const double* a_dev, const void* x, double sb,
                 const double* b_dev, const void* y, void* z, void* stream);
/* z = blockdiag(inv) r: block-Jacobi preconditioner application (SURVEY section 8f-1; what users of the reference write as
 * M = lambda r: (Binv @ r.view(-1, bs, 1)).view(-1)).  inv: device [ceil(n/bs)][bs][bs] row-major inverses of the
 * diagonal blocks, dtype as the vectors.  r and z must not alias. */
int bk_block_apply(bk_handle* h, int64_t n, int bs, int dtype, const void* inv, const void* r, void* z, void* stream);
/* complex128 vectors stored as interleaved (re, im) doubles, 16-byte aligned (what torch.view_as_real gives):
 * bk_cdot: out2[0] + i out2[1] = sum conj(x_k) y_k (device, fp64 x 2) — torch.vdot, reference _vdot :86-91;
 * bk_caxpby: z = (ar + i ai) x + (br + i bi) y.  With the complex matrix registered as its real-equivalent 2n x 2n CSR
 * ([[re, -im], [im, re]] blocks; module_a/complex_route.py) these serve the reference's complex code path (:100-127,
 * :1220) on the device. */
int bk_cdot(bk_handle* h, int64_t n_complex, const void* x, const void* y, double* out2, void* stream);
int bk_caxpby(bk_handle* h, int64_t n_complex, double ar, double ai, const void* x, double br, double bi,
              const void* y, void* z, void* stream);
/* z = x / d — true division, the reference's `y / norm` (_safe_normalize :266-272) */
int bk_div_scalar(bk_handle* h, int64_t n, int dtype, const void* x, double d, void* z, void* stream);

/* ---- solvers ------------------------------------------------------------------------
 * b: device vector (read only).  x: device vector, in = initial guess when has_x0 != 0
 * (ignored otherwise: x0 = 0 as in _isolve :975-976), out = solution.
 * tol/atol are the caller's Python floats; the fp32 rounding of torch.tensor(tol)
 * (:816, :871, :1010) is reproduced inside.  maxiter < 0 means the default 10*n (:982-984).
 *
 * bk_cg       replaces _cg_solve :806-856 + _isolve :967-1016
 * bk_bicgstab replaces _bicgstab_solve :859-964 + _isolve
 */
int bk_cg(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol, double atol,
          int64_t maxiter, bk_result* result, void* stream);
int bk_bicgstab(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol,
                double atol, int64_t maxiter, bk_result* result, void* stream);
/* Jacobi-preconditioned CG: _cg_solve with M = (r -> r / diag), :820-853 — z = M r, gamma = r.z, the stop test on
 * rs = r.r (:838), p = z + beta p — and _isolve's final check on ||M (b - A x)|| (:1008).  `diag`: device vector of
 * A's dtype (bk_csr_diagonal extracts it).  What the reference does through a user-supplied Python callable
 * `M = lambda r: r / d`, kept on the device (SURVEY section 8f-1).  Same result fields as bk_cg. */
int bk_cg_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0, double tol,
                 double atol, int64_t maxiter, bk_result* result, void* stream);
/* BiCGStab with the same built-in M: right preconditioning exactly as _bicgstab_solve :907-946 (phat = M p,
 * q = A phat, shat = M s, t = A shat, x += alpha phat + omega shat; residuals, dots and breakdown tests in residual
 * space) and the M-weighted final check (:1008). */
int bk_bicgstab_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0,
                       double tol, double atol, int64_t maxiter, bk_result* result, void* stream);
/* GMRES with the same built-in M applied from the left, as the reference does with a callable M: v = M(A v) in every
 * Arnoldi step (:351), r = M(b - A x) at every restart (:491, :636, :791), ptol from ||M b|| (:750-753), final check on
 * ||M(b - A x)|| (:766).  Arguments as bk_gmres. */
int bk_gmres_jacobi(bk_handle* h, const bk_csr* A, const void* diag, const void* b, void* x, int has_x0,
                    double tol_eff, double atol_eff, int restart, int64_t maxiter, int method, bk_result* result,
                    void* stream);
/* ---- multicolor symmetric Gauss-Seidel preconditioner (AMGX's MULTICOLOR_GS, one symmetric sweep) -------------
 * No reference counterpart: what users of the reference write as a callable M, kept on the device.
 * bk_sgs_create colors A's pattern deterministically (Jones-Plassmann rounds over the neighbours j != i with (i, j) or
 *   (j, i) stored, priority (fmix32(i) << 32) | i, smallest color no earlier-colored neighbour holds) and groups the rows
 *   by color.  Every row must store a nonzero diagonal (the sum of its col == row entries): otherwise BK_ERR_ARG, naming
 *   the row.  More than 255 colors: BK_ERR_UNSUPPORTED.  The result is cached, owned by A and freed with it.
 * bk_sgs_get_info: the number of colors C and of coloring rounds.  bk_sgs_colors: the colors, copied to a device
 *   uint8[n].
 * bk_sgs_apply: z = M r with z = 0, a forward sweep over colors 0..C-1 and a backward sweep over C-2..0, every row
 *   z_i = (r_i - sum_{j != i} a_ij z_j) / a_ii summed in CSR order (2C-1 kernels; bitwise reproducible).  The sweeps
 *   read A's rowptr / col / val at every call, so an in-place update of the (borrowed) values is picked up by the next
 *   application; only the coloring depends on the pattern.  (bk_*_jacobi, by contrast, take the diagonal the caller
 *   extracted.)  r and z must not alias.
 * bk_cg_sgs / bk_bicgstab_sgs / bk_gmres_sgs: arguments, recurrences and result fields of bk_cg_jacobi /
 *   bk_bicgstab_jacobi / bk_gmres_jacobi with M = bk_sgs_apply.  A_sys may differ from the matrix S was built from
 *   (same order and dtype): the adjoint solve runs on A^T with the M of A. */
int bk_sgs_create(bk_handle* h, bk_csr* A, void* stream, bk_sgs** out);
int bk_sgs_get_info(const bk_sgs* S, int32_t* ncolors, int32_t* rounds);
int bk_sgs_colors(const bk_sgs* S, void* out, void* stream);
int bk_sgs_apply(bk_handle* h, const bk_sgs* S, const void* r, void* z, void* stream);
int bk_cg_sgs(bk_handle* h, const bk_csr* A_sys, const bk_sgs* S, const void* b, void* x, int has_x0, double tol,
              double atol, int64_t maxiter, bk_result* result, void* stream);
int bk_bicgstab_sgs(bk_handle* h, const bk_csr* A_sys, const bk_sgs* S, const void* b, void* x, int has_x0, double tol,
                    double atol, int64_t maxiter, bk_result* result, void* stream);
int bk_gmres_sgs(bk_handle* h, const bk_csr* A_sys, const bk_sgs* S, const void* b, void* x, int has_x0,
                 double tol_eff, double atol_eff, int restart, int64_t maxiter, int method, bk_result* result,
                 void* stream);
/* out[r] = A[r][r] (0 when the row stores no diagonal entry); out: device vector of A's dtype */
int bk_csr_diagonal(bk_handle* h, const bk_csr* A, void* out, void* stream);
/* bk_gmres replaces gmres :641-784, _gmres_solve_with_method :788-803, _gmres_batched :431-493,
 * _gmres_incremental :557-638, _kth_arnoldi_iteration :331-388, _iterative_classical_gram_schmidt
 * :284-328, _givens_rotation :508-518, _safe_normalize :217-273.
 * tol_eff  = the reference's `adaptive_tol` after its torch.tensor() rounding (:739-747),
 * atol_eff = max(float32(atol), float32(base_atol)) (:746-748); the device computes
 * atol = max(tol_eff*||b||, atol_eff) and ptol = ||b|| * min(1, atol/||b||) (:750-753).
 * maxiter = maximum number of restart cycles (< 0: 10*n, :719-721). */
int bk_gmres(bk_handle* h, const bk_csr* A, const void* b, void* x, int has_x0, double tol_eff,
             double atol_eff, int restart, int64_t maxiter, int method, bk_result* result, void* stream);

/* ---- host-buffer entry (end-to-end path: H2D copies + solve + D2H inside) -----------
 * All pointers are HOST memory (pinned or pageable).  idx_bits 32/64.  method: 0 cg, 1 bicgstab,
 * 2 gmres (restart/gmres_method used only then).  tol/atol: for cg/bicgstab the caller's Python floats; for gmres
 * they are forwarded unchanged to bk_gmres, i.e. they must be tol_eff / atol_eff as documented there (the caller
 * applies the reference's device-dependent constants of :737-748; the Python front end does, with the 'cpu'
 * constants because the tensors it was given live on the CPU).  x_inout: x0 in (if has_x0) / x out. */
int bk_solve_host(bk_handle* h, int method, int64_t n, int64_t nnz, const void* rowptr, const void* col,
                  int idx_bits, const void* val, int dtype, const void* b, void* x_inout, int has_x0,
                  double tol, double atol, int64_t maxiter, int restart, int gmres_method,
                  bk_result* result);

/* ---- multi-GPU (one process per GPU; 1-D row partition; SURVEY §8e) ------------------
 * No reference counterpart (the reference is single-device).  The caller (Python, torch.distributed) owns
 * rendezvous and the set-up index work: rank 0 calls bk_dist_unique_id and broadcasts the 128 bytes; every rank
 * splits its rows into a LOCAL block (columns inside its slab, renumbered from 0) and a GHOST block (columns owned
 * by peers, renumbered into a compact ghost vector ordered by owner rank) and passes both here, all index arrays
 * int32 on the device:
 *   local block : CSR n_local x n_local                      (loc_rowptr, loc_col, loc_val)
 *   ghost block : CSR over the n_brows boundary rows         (brow_ids = their local row ids, gh_rowptr[n_brows+1],
 *                                                             gh_col = index into the ghost vector, gh_val)
 *   halo plan   : peer_ranks/send_counts/recv_counts (HOST arrays, npeers entries; receives land in the ghost
 *                 vector in peer order), send_idx (DEVICE int32: local indices to send, concatenated per peer).
 * Run time: boundary entries are packed, exchanged with ncclSend/ncclRecv on a side stream overlapped with the
 * local-block SpMV, the ghost rows are added afterwards; the scalar dots go through ncclAllReduce. */
int bk_dist_unique_id(void* id128);
int bk_dist_create(bk_handle* h, const void* id128, int rank, int nranks, int64_t n_local, int64_t nnz_loc,
                   const void* loc_rowptr, const void* loc_col, const void* loc_val, int64_t n_brows,
                   const void* brow_ids, int64_t nnz_gh, const void* gh_rowptr, const void* gh_col,
                   const void* gh_val, int64_t n_ghost, int npeers, const int32_t* peer_ranks,
                   const int64_t* send_counts, const int64_t* recv_counts, const void* send_idx, int dtype,
                   void* stream, bk_dist** out);
int bk_dist_destroy(bk_dist* D);
/* Optional: the rows of this rank as ONE matrix over the extended vector [ local entries | ghost vector ] — CSR with
 * n_local rows, columns < n_local + n_ghost (ghost entry g has column n_local + g), entries in the order of the GLOBAL
 * matrix's rows.  When the row-bitmask plan (kernel 6) fits it, the peer-memory path runs ONE SpMV kernel per matvec:
 * interior chunks first, the chunks that gather ghost entries last, after polling the neighbours' arrival flags — the
 * separate boundary-row kernel and the correction of the dot partials disappear.  ghost_gid: device int64[n_ghost],
 * global ids of the ghost entries; row_begin: global id of local row 0 (pattern entries are ordered by global offset,
 * like the single-GPU matrix).  ext_val may be the array the local/ghost blocks were split from.  The arrays are only
 * read during this call.  *folded = 1 when the plan was built (2: its interior steps also qualify for kernel 7), else 0
 * and the two-kernel path stays in use. */
int bk_dist_set_extended(bk_dist* D, int64_t nnz_ext, const void* ext_rowptr, const void* ext_col, const void* ext_val,
                         const void* ghost_gid, int64_t row_begin, void* stream, int32_t* folded);
/* Peer-memory path (NVLink/NVSwitch, CUDA IPC).  Each rank exports the 64-byte IPC handle of its communication
 * window (all-reduce slots, halo flags, ghost vector); the caller gathers all handles and every rank maps them.
 * remote_ghost_offsets[i] = element offset inside halo peer i's ghost vector where this rank's entries land.
 * Once connected, bk_dist_cg pushes boundary entries straight into the neighbours' ghost vectors from a kernel and
 * all-reduces the two scalar dots with a one-shot peer-store exchange inside the reducing kernels' epilogues
 * (no NCCL call and no extra kernel per iteration).  Returns BK_ERR_UNSUPPORTED when peers cannot be mapped; the
 * NCCL path then stays in use. */
int bk_dist_p2p_export(bk_dist* D, void* handle64);
int bk_dist_p2p_connect(bk_dist* D, const void* handles, const int64_t* remote_ghost_offsets);
/* y_local = (A x)_local */
int bk_dist_spmv(bk_handle* h, bk_dist* D, const void* x_local, void* y_local, void* stream);
/* distributed CG (same recurrences / stop test / info as bk_cg; n_global sets the default maxiter = 10 n) */
int bk_dist_cg(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol,
               double atol, int64_t maxiter, int64_t n_global, bk_result* result, void* stream);
/* the same three with the built-in Jacobi preconditioner (diag_local: this rank's slice of diag(A); the diagonal of a
 * row partition is local).  Recurrences as bk_cg_jacobi / bk_bicgstab_jacobi / bk_gmres_jacobi. */
int bk_dist_cg_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local, void* x_local, int has_x0,
                      double tol, double atol, int64_t maxiter, int64_t n_global, bk_result* result, void* stream);
int bk_dist_bicgstab_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local, void* x_local,
                            int has_x0, double tol, double atol, int64_t maxiter, int64_t n_global, bk_result* result,
                            void* stream);
int bk_dist_gmres_jacobi(bk_handle* h, bk_dist* D, const void* diag_local, const void* b_local, void* x_local,
                         int has_x0, double tol_eff, double atol_eff, int restart, int64_t maxiter, int method,
                         int64_t n_global, bk_result* result, void* stream);
/* distributed BiCGStab / GMRES: the single-GPU drivers (bk_bicgstab, bk_gmres — same recurrences, breakdown codes,
 * restart logic and info) run on the row-partitioned matrix; every dot product becomes a global sum (NCCL path:
 * ncclAllReduce + a one-thread scalar kernel; peer-memory path: all-reduced inside the reducing kernel's epilogue,
 * GMRES's projection coefficients V^T w as one vector all-reduce of j+1 doubles).  The GMRES small dense problem is
 * replicated on every rank.  Reference: _bicgstab_solve :859-964, gmres :641-784; SURVEY section 8e. */
int bk_dist_bicgstab(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol,
                     double atol, int64_t maxiter, int64_t n_global, bk_result* result, void* stream);
int bk_dist_gmres(bk_handle* h, bk_dist* D, const void* b_local, void* x_local, int has_x0, double tol_eff,
                  double atol_eff, int restart, int64_t maxiter, int method, int64_t n_global, bk_result* result,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BK_KRYLOV_H */
