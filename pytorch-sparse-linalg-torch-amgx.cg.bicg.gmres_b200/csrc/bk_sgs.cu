// bk_sgs.cu — multicolor symmetric Gauss-Seidel preconditioner (AMGX's MULTICOLOR_GS with one symmetric sweep).
//
// Set-up (bk_sgs_create, deterministic):
//   neighbours  j != i with (i, j) or (j, i) stored — the rows of A plus the rows of the cached transpose
//   priority    prio(i) = (fmix32(i) << 32) | i
//   rounds      Jones-Plassmann: an uncolored row whose priority exceeds that of every uncolored neighbour takes the
//               smallest color no neighbour colored in an EARLIER round holds.  A round reads a snapshot: a row
//               colored in round t still counts as uncolored for the decisions of round t, so the result does not
//               depend on scheduling (two rows colored in the same round are never neighbours).
//   row lists   a stable radix sort by color
// Application z = M r: z = 0, forward sweep over colors 0..C-1, backward sweep over C-2..0, each row
//   z_i = (r_i - sum_{j != i} a_ij z_j) / a_ii   summed in CSR order by one thread.
// No two rows of one color are neighbours, so every sweep is race-free and the result bitwise reproducible.
#include "bk_internal.cuh"
#include "bk_spmv.cuh"

#include <stdlib.h>

#define BK_SGS_MAXC 255  // colors are stored as uint8

__device__ __forceinline__ unsigned long long bk_sgs_prio(unsigned int i) {
  unsigned int h = i;
  h ^= h >> 16;
  h *= 0x85ebca6bu;
  h ^= h >> 13;
  h *= 0xc2b2ae35u;
  h ^= h >> 16;
  return ((unsigned long long)h << 32) | i;
}

// state[i] = -1 (uncolored) or color | (round << 8)
__device__ __forceinline__ bool bk_sgs_unc(int st, int round) { return st < 0 || (st >> 8) == round; }

__global__ void bk_sgs_round_kernel(const int* __restrict__ rp, const int* __restrict__ ci,
                                    const int* __restrict__ trp, const int* __restrict__ tci, long long n, int round,
                                    int* __restrict__ state, unsigned int* __restrict__ remaining,
                                    int* __restrict__ overflow) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (state[i] >= 0) continue;
    const unsigned long long pi = bk_sgs_prio((unsigned int)i);
    unsigned long long used[4] = {0ull, 0ull, 0ull, 0ull};
    bool top = true;
    for (int pass = 0; pass < 2 && top; ++pass) {
      const int* p = pass ? trp : rp;
      const int* c = pass ? tci : ci;
      for (int k = p[i]; k < p[i + 1]; ++k) {
        const int j = c[k];
        if (j == (int)i) continue;
        const int sj = state[j];
        if (bk_sgs_unc(sj, round)) {
          if (bk_sgs_prio((unsigned int)j) > pi) {
            top = false;
            break;
          }
        } else {
          const int col = sj & 255;
#pragma unroll
          for (int w = 0; w < 4; ++w)
            if ((col >> 6) == w) used[w] |= 1ull << (col & 63);
        }
      }
    }
    if (!top) {
      atomicAdd(remaining, 1u);
      continue;
    }
    int color = 256;
#pragma unroll
    for (int w = 3; w >= 0; --w)
      if (~used[w]) color = w * 64 + __ffsll((long long)~used[w]) - 1;
    if (color >= BK_SGS_MAXC) {
      atomicMax(overflow, 1);
      color = BK_SGS_MAXC;
    }
    state[i] = color | (round << 8);
  }
}

// colors (uint8) and radix-sort keys from the final state; ncol = the number of colors
__global__ void bk_sgs_finish_kernel(const int* __restrict__ state, long long n, unsigned char* __restrict__ colors,
                                     int* __restrict__ keys, int* __restrict__ ncol) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int c = state[i] & 255;
    colors[i] = (unsigned char)c;
    keys[i] = c;
    atomicMax(ncol, c + 1);
  }
}

template <typename T>
__global__ void bk_sgs_diag_check_kernel(const int* __restrict__ rp, const int* __restrict__ ci,
                                         const T* __restrict__ val, long long n, int* __restrict__ bad) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    T d = T(0);  // as bk_csr_diagonal: the sum of the row's col == row entries
    for (int k = rp[i]; k < rp[i + 1]; ++k)
      if (ci[k] == (int)i) d += val[k];
    if (d == T(0)) atomicMin(bad, (int)i);
  }
}

// ---- application --------------------------------------------------------------------------------------------
// One lane per row of the color's row list.  FIRST: the forward sweep of color 0 over ALL rows, which also clears z
// for the other colors (with z = 0 a color-0 row's sum is r_i - 0).
template <typename T, bool FIRST>
__global__ void __launch_bounds__(256) bk_sgs_sweep_kernel(const int* __restrict__ rp, const int* __restrict__ ci,
                                                           const T* __restrict__ val, const int* __restrict__ rows,
                                                           const unsigned char* __restrict__ colors, int count,
                                                           const T* __restrict__ r, T* z, const bk_dev_state* st,
                                                           int guard) {
  if (bk_guard_skip(st, guard)) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int i = FIRST ? t : rows[t];
  if (FIRST && colors[i] != 0) {
    z[i] = T(0);
    return;
  }
  T acc = T(0), d = T(0);
  for (int k = rp[i]; k < rp[i + 1]; ++k) {
    const int j = ci[k];
    const T a = val[k];
    if (j == i) {
      d += a;
    } else if (!FIRST) {
      acc = bk_add(acc, bk_mul(a, z[j]));
    }
  }
  z[i] = bk_sub(r[i], acc) / d;
}

template <typename T>
static int bk_sgs_run_t(const bk_sgs* S, const T* r, T* z, const bk_dev_state* st, int guard, cudaStream_t s) {
  const bk_csr* A = S->A;
  const T* val = (const T*)A->val;
  const int n = (int)A->n;
  bk_sgs_sweep_kernel<T, true><<<(n + 255) / 256, 256, 0, s>>>(A->rowptr, A->col, val, S->rows, S->colors, n, r, z,
                                                                st, guard);
  const int C = S->ncolors;
  for (int step = 1; step < 2 * C - 1; ++step) {
    const int c = step < C ? step : 2 * C - 2 - step;  // 1..C-1, then C-2..0
    const int cnt = S->offs[c + 1] - S->offs[c];
    bk_sgs_sweep_kernel<T, false><<<(cnt + 255) / 256, 256, 0, s>>>(A->rowptr, A->col, val, S->rows + S->offs[c],
                                                                     S->colors, cnt, r, z, st, guard);
  }
  BK_KERNEL_CHECK();
  return BK_OK;
}

int bk_sgs_run(bk_handle* h, const bk_sgs* S, const void* r, void* z, int guard, cudaStream_t s) {
  if (S->A->dtype == BK_F64) return bk_sgs_run_t<double>(S, (const double*)r, (double*)z, h->st, guard, s);
  return bk_sgs_run_t<float>(S, (const float*)r, (float*)z, h->st, guard, s);
}

void bk_sgs_free(bk_sgs* S) {
  if (!S) return;
  if (S->colors) bk_pool_free(S->colors);
  if (S->rows) bk_pool_free(S->rows);
  free(S->offs);
  free(S);
}

int bk_sgs_args_check(const char* who, bk_handle* h, const bk_csr* A, const bk_sgs* S) {
  if (!S) return bk_fail(BK_ERR_ARG, "%s: null preconditioner", who);
  if (S->A->h != h) return bk_fail(BK_ERR_ARG, "%s: preconditioner belongs to another handle", who);
  if (S->A->n != A->n || S->A->dtype != A->dtype)
    return bk_fail(BK_ERR_ARG, "%s: preconditioner of an order-%lld matrix (dtype %d) for an order-%lld system (dtype %d)",
                   who, (long long)S->A->n, S->A->dtype, (long long)A->n, A->dtype);
  return BK_OK;
}

extern "C" int bk_sgs_create(bk_handle* h, bk_csr* A, void* stream, bk_sgs** out) {
  if (!h || !A || !out) return bk_fail(BK_ERR_ARG, "bk_sgs_create: null argument");
  if (A->h != h) return bk_fail(BK_ERR_ARG, "bk_sgs_create: matrix belongs to another handle");
  if (A->n_cols != A->n) return bk_fail(BK_ERR_UNSUPPORTED, "bk_sgs_create: square single-GPU matrices only");
  if (!A->rowptr || !A->col) return bk_fail(BK_ERR_UNSUPPORTED, "bk_sgs_create: the matrix keeps no CSR arrays");
  if (A->sgs) {
    *out = A->sgs;
    return BK_OK;
  }
  BK_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const long long n = A->n;
  if (n == 0) return bk_fail(BK_ERR_ARG, "bk_sgs_create: empty matrix");
  bk_csr* At = nullptr;
  BK_TRY(bk_csr_transpose(h, A, stream, &At));

  bk_sgs* S = (bk_sgs*)calloc(1, sizeof(bk_sgs));
  if (!S) return bk_fail(BK_ERR_ALLOC, "bk_sgs_create: host allocation failed");
  S->A = A;
  const size_t nn = (size_t)(n > 0 ? n : 1);
  int *state = nullptr, *k0 = nullptr, *k1 = nullptr, *v0 = nullptr, *v1 = nullptr, *dev = nullptr;
  auto cleanup = [&]() {
    cudaStreamSynchronize(s);
    for (int* p : {state, k0, k1, v0, v1, dev})
      if (p) bk_pool_free(p);
  };
  auto fail = [&](int code, const char* msg) {
    cleanup();
    bk_sgs_free(S);
    return bk_fail(code, "bk_sgs_create: %s", msg);
  };
  bool ok = bk_pool_alloc((void**)&S->colors, nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&S->rows, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&state, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&k0, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&k1, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&v0, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&v1, sizeof(int) * nn, s) == cudaSuccess &&
            bk_pool_alloc((void**)&dev, sizeof(int) * (4 + BK_SGS_MAXC + 1), s) == cudaSuccess;
  if (!ok) {
    cudaGetLastError();
    return fail(BK_ERR_ALLOC, "device allocation failed");
  }
  // dev[0] smallest row without a nonzero diagonal, dev[1] rows left uncolored, dev[2] overflow, dev[3] colors
  const int g = bk_grid_rows(h->num_sms * 8, n, 256);
  int host[4] = {INT32_MAX, 0, 0, 0};
  if (cudaMemcpyAsync(dev, host, sizeof(host), cudaMemcpyHostToDevice, s) != cudaSuccess) {
    cudaGetLastError();
    return fail(BK_ERR_CUDA, "copy failed");
  }
  if (A->dtype == BK_F64)
    bk_sgs_diag_check_kernel<double><<<g, 256, 0, s>>>(A->rowptr, A->col, (const double*)A->val, n, dev);
  else
    bk_sgs_diag_check_kernel<float><<<g, 256, 0, s>>>(A->rowptr, A->col, (const float*)A->val, n, dev);
  if (cudaMemcpyAsync(host, dev, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    cudaGetLastError();
    return fail(BK_ERR_CUDA, "diagonal check failed");
  }
  if (host[0] != INT32_MAX) {
    cleanup();
    bk_sgs_free(S);
    return bk_fail(BK_ERR_ARG, "bk_sgs_create: row %d stores no nonzero diagonal entry", host[0]);
  }

  cudaMemsetAsync(state, 0xff, sizeof(int) * nn, s);
  int round = 0;
  for (;; ++round) {
    cudaMemsetAsync(dev + 1, 0, sizeof(int), s);
    bk_sgs_round_kernel<<<g, 256, 0, s>>>(A->rowptr, A->col, At->rowptr, At->col, n, round, state,
                                          (unsigned int*)(dev + 1), dev + 2);
    unsigned int left = 0;
    if (cudaMemcpyAsync(&left, dev + 1, sizeof(left), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
      cudaGetLastError();
      return fail(BK_ERR_CUDA, "coloring round failed");
    }
    if (left == 0) break;
  }
  S->rounds = round + 1;
  bk_sgs_finish_kernel<<<g, 256, 0, s>>>(state, n, S->colors, k0, dev + 3);
  bk_iota_i32(h, v0, n, s);
  int *ks = nullptr, *vs = nullptr;
  int rc = bk_sort_pairs_i32(h, k0, k1, v0, v1, n, 8, s, &ks, &vs);
  if (rc != BK_OK) {
    cleanup();
    bk_sgs_free(S);
    return rc;
  }
  cudaMemcpyAsync(S->rows, vs, sizeof(int) * (size_t)n, cudaMemcpyDeviceToDevice, s);
  bk_lower_bound_i32(h, ks, n, BK_SGS_MAXC, dev + 4, s);  // dev[4 + c] = first row of color c
  int offs[BK_SGS_MAXC + 1];
  if (cudaMemcpyAsync(host, dev, sizeof(host), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaMemcpyAsync(offs, dev + 4, sizeof(offs), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    cudaGetLastError();
    return fail(BK_ERR_CUDA, "row lists failed");
  }
  if (host[2]) {
    cleanup();
    bk_sgs_free(S);
    return bk_fail(BK_ERR_UNSUPPORTED, "bk_sgs_create: the coloring needs more than %d colors", BK_SGS_MAXC);
  }
  S->ncolors = host[3];
  S->offs = (int*)malloc(sizeof(int) * (size_t)(S->ncolors + 1));
  if (!S->offs) return fail(BK_ERR_ALLOC, "host allocation failed");
  memcpy(S->offs, offs, sizeof(int) * (size_t)(S->ncolors + 1));
  cleanup();
  A->sgs = S;
  *out = S;
  return BK_OK;
}

extern "C" int bk_sgs_get_info(const bk_sgs* S, int32_t* ncolors, int32_t* rounds) {
  if (!S || !ncolors || !rounds) return bk_fail(BK_ERR_ARG, "bk_sgs_get_info: null argument");
  *ncolors = S->ncolors;
  *rounds = S->rounds;
  return BK_OK;
}

extern "C" int bk_sgs_colors(const bk_sgs* S, void* out, void* stream) {
  if (!S || (!out && S->A->n > 0)) return bk_fail(BK_ERR_ARG, "bk_sgs_colors: null argument");
  BK_CUDA(cudaSetDevice(S->A->h->device));
  if (S->A->n == 0) return BK_OK;
  BK_CUDA(cudaMemcpyAsync(out, S->colors, (size_t)S->A->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return BK_OK;
}

extern "C" int bk_sgs_apply(bk_handle* h, const bk_sgs* S, const void* r, void* z, void* stream) {
  if (!h || !S) return bk_fail(BK_ERR_ARG, "bk_sgs_apply: null handle/preconditioner");
  if (S->A->h != h) return bk_fail(BK_ERR_ARG, "bk_sgs_apply: preconditioner belongs to another handle");
  const long long n = S->A->n;
  if (n > 0 && (!r || !z)) return bk_fail(BK_ERR_ARG, "bk_sgs_apply: null vector");
  const size_t vb = (size_t)n * bk_dtype_size(S->A->dtype);
  if ((const char*)r < (const char*)z + vb && (const char*)z < (const char*)r + vb)
    return bk_fail(BK_ERR_ARG, "bk_sgs_apply: r and z must not alias");
  BK_CUDA(cudaSetDevice(h->device));
  if (n == 0) return BK_OK;
  return bk_sgs_run(h, S, r, z, 0, (cudaStream_t)stream);
}
