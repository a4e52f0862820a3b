// bk_core.cu — handle, matrix registration, building-block entry points of libbk_krylov.
#include <stdarg.h>
#include <stdlib.h>

#include <nvtx3/nvToolsExt.h>

#include "bk_internal.cuh"
#include "bk_spmv.cuh"
#include "bk_vec.cuh"

thread_local char bk_err_buf[512] = {0};

// ---- per-call bracket: NVTX ranges (BK_NVTX=1 / option nvtx) and device time of the call (bk_result.device_ms) -----
// SURVEY section 5: the reference has no profiler hooks; these are ours.  nvtx3 is header-only and binds to the
// profiler's injection library lazily, so there is nothing to link and the calls are no-ops outside a profiler.
void bk_call_begin(bk_handle* h, cudaStream_t s, const char* name) {
  h->last_loop_mode = 0;
  if (h->nvtx) {
    nvtxRangePushA(name);
    nvtxRangePushA("setup");
  }
  cudaEventRecord(h->ev_t0, s);
}
void bk_call_mark(bk_handle* h, const char* phase) {
  if (h->nvtx) {
    nvtxRangePop();
    nvtxRangePushA(phase);
  }
}
void bk_call_stop(bk_handle* h, cudaStream_t s) { cudaEventRecord(h->ev_t1, s); }
void bk_call_finish(bk_handle* h, bk_result* res) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1) != cudaSuccess) {
    cudaGetLastError();
    ms = 0.f;
  }
  res->device_ms = (double)ms;
  res->loop_mode_used = h->last_loop_mode;
  if (h->nvtx) {
    nvtxRangePop();
    nvtxRangePop();
  }
}

int bk_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(bk_err_buf, sizeof(bk_err_buf), fmt, ap);
  va_end(ap);
  return code;
}

extern "C" int bk_version(void) { return BK_VERSION; }
extern "C" const char* bk_last_error(void) { return bk_err_buf; }

static int64_t bk_env_int(const char* name, int64_t dflt) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  return strtoll(v, nullptr, 10);
}

cudaError_t bk_pool_alloc(void** p, size_t bytes, cudaStream_t s) {
  cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 1, s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *p = nullptr;
  }
  return e;
}

void bk_pool_free(void* p) {
  // ordered on the legacy default stream: callers have synchronised the streams that used the memory
  // (solver entry points end with a stream sync; bk_csr_destroy synchronises the device first)
  if (p) cudaFreeAsync(p, 0);
}

extern "C" int bk_create(int device, bk_handle** out) {
  if (!out) return bk_fail(BK_ERR_ARG, "bk_create: out is null");
  *out = nullptr;
  int count = 0;
  BK_CUDA(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count)
    return bk_fail(BK_ERR_ARG, "bk_create: device %d out of range (%d CUDA devices)", device, count);
  BK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BK_CUDA(cudaGetDeviceProperties(&prop, device));
  {  // keep freed pool memory cached instead of returning it to the driver at every synchronisation
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long thr = ~0ULL;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
  }
  bk_handle* h = (bk_handle*)calloc(1, sizeof(bk_handle));
  if (!h) return bk_fail(BK_ERR_ALLOC, "bk_create: host allocation failed");
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->l2_bytes = prop.l2CacheSize;
  h->mem_bytes = (int64_t)prop.totalGlobalMem;
  h->grid_mult_vec = (int)bk_env_int("BK_GRID_MULT_VEC", 3);
  h->grid_mult_spmv = (int)bk_env_int("BK_GRID_MULT_SPMV", 4);
  h->tma_ctas = (int)bk_env_int("BK_TMA_CTAS", 4);
  h->pair_ctas = (int)bk_env_int("BK_PAIR_CTAS", 4);
  h->mask_ctas = (int)bk_env_int("BK_MASK_CTAS", 4);
  h->mask_cctas = (int)bk_env_int("BK_MASK_CCTAS", 4);
  h->mask2_prefetch = (int)bk_env_int("BK_MASK2_PREFETCH", 0);
  h->mask_group = (int)bk_env_int("BK_MASK_GROUP", 8);
  h->mask_prefetch = (int)bk_env_int("BK_MASK_PREFETCH", 1);
  h->mask_window = (int)bk_env_int("BK_MASK_WINDOW", 0);  // measured slower than LDG + L2 prefetch so far (115 vs 84 us)
  h->mask_wgroup = (int)bk_env_int("BK_MASK_WGROUP", 4);
  h->nvtx = (int)bk_env_int("BK_NVTX", 0);
  h->dist_fuse_push = (int)bk_env_int("BK_DIST_FUSE_PUSH", 1);
  h->dist_fold = (int)bk_env_int("BK_DIST_FOLD", 1);
  h->tma_stages = (int)bk_env_int("BK_TMA_STAGES", 0);
  h->use_tma = (int)bk_env_int("BK_SPMV_TMA", 1);
  h->dist_p2p = (int)bk_env_int("BK_DIST_P2P", 1);
  h->use_compress = (int)bk_env_int("BK_SPMV_COMPRESS", 3);
  h->use_split = (int)bk_env_int("BK_SPMV_SPLIT", 1);
  h->persistent = (int)bk_env_int("BK_PERSISTENT", 1);
  h->persistent_max_n = (int)bk_env_int("BK_PERSISTENT_MAX_N", 200000);
  h->persistent_cluster = (int)bk_env_int("BK_PERSISTENT_CLUSTER", 1);
  h->prefetch_x = (int)bk_env_int("BK_SPMV_PREFETCH_X", 0);  // measured: 5 % slower on P3D-256, kept as an experiment
  h->loop_mode = (int)bk_env_int("BK_LOOP_MODE", BK_LOOP_AUTO);
  h->chunk = (int)bk_env_int("BK_CHUNK", 0);
  h->fuse_xpay = (int)bk_env_int("BK_FUSE_XPAY", -1);  // -1 auto, 0 off, 1 on
  h->snake = (int)bk_env_int("BK_SNAKE", 1);
  h->l2_hints = (int)bk_env_int("BK_L2_HINTS", 0);
  h->cg_lag_x = (int)bk_env_int("BK_CG_LAG_X", 1);
  h->mask_const = (int)bk_env_int("BK_MASK_CONST", 1);
  h->next_uid = 1;
  cudaError_t e;
  e = cudaMalloc(&h->partials, sizeof(double) * BK_NSLOT * BK_SLOT_ROWS * BK_MAXB);
  if (e == cudaSuccess) e = cudaMalloc(&h->counters, sizeof(unsigned int) * 16);
  if (e == cudaSuccess) e = cudaMemset(h->counters, 0, sizeof(unsigned int) * 16);
  if (e == cudaSuccess) e = cudaMalloc(&h->st, sizeof(bk_dev_state));
  if (e == cudaSuccess) e = cudaMemset(h->st, 0, sizeof(bk_dev_state));
  if (e == cudaSuccess) e = cudaMallocHost(&h->st_host, sizeof(bk_dev_state) * 4);
  for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&h->ev[i], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev_t0);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev_t1);
  if (e == cudaSuccess) e = cudaMalloc((void**)&h->cksum, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->io_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    bk_destroy(h);
    return bk_fail(BK_ERR_CUDA, "bk_create: %s", cudaGetErrorString(e));
  }
  *out = h;
  return BK_OK;
}

void bk_graphs_invalidate(bk_handle* h) {
  for (int i = 0; i < 8; ++i) {
    if (h->graphs[i].valid && h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
    h->graphs[i].valid = 0;
    h->graphs[i].exec = nullptr;
  }
}

extern "C" int bk_destroy(bk_handle* h) {
  if (!h) return BK_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  bk_graphs_invalidate(h);
  // h->dist_comm (NCCL) is deliberately not destroyed here: handles die at interpreter exit, when peers may already
  // be gone, and ncclCommDestroy may then block; the driver reclaims it with the process
  if (h->partials) cudaFree(h->partials);
  if (h->counters) cudaFree(h->counters);
  if (h->st) cudaFree(h->st);
  if (h->st_host) cudaFreeHost(h->st_host);
  if (h->ws) cudaFree(h->ws);
  if (h->stage) cudaFree(h->stage);
  if (h->gm_small) cudaFree(h->gm_small);
  if (h->gm_partials) cudaFree(h->gm_partials);
  for (int i = 0; i < 4; ++i)
    if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->ev_t0) cudaEventDestroy(h->ev_t0);
  if (h->ev_t1) cudaEventDestroy(h->ev_t1);
  if (h->cksum) cudaFree(h->cksum);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->io_stream) cudaStreamDestroy(h->io_stream);
  free(h);
  return BK_OK;
}

int bk_ws_reserve(bk_handle* h, size_t bytes) {
  if (bytes <= h->ws_bytes) return BK_OK;
  bk_graphs_invalidate(h);
  if (h->ws) {
    BK_CUDA(cudaDeviceSynchronize());
    BK_CUDA(cudaFree(h->ws));
    h->ws = nullptr;
    h->ws_bytes = 0;
  }
  const size_t want = (bytes + 255) & ~(size_t)255;
  cudaError_t e = cudaMalloc(&h->ws, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return bk_fail(BK_ERR_ALLOC, "workspace of %zu bytes: %s", want, cudaGetErrorString(e));
  }
  h->ws_bytes = want;
  return BK_OK;
}

static int* bk_opt_field(bk_handle* h, const char* key) {
  if (!key) return nullptr;
  if (!strcmp(key, "grid_mult_vec")) return &h->grid_mult_vec;
  if (!strcmp(key, "grid_mult_spmv")) return &h->grid_mult_spmv;
  if (!strcmp(key, "grid_mult")) return &h->grid_mult_spmv;
  if (!strcmp(key, "tma_ctas")) return &h->tma_ctas;
  if (!strcmp(key, "pair_ctas")) return &h->pair_ctas;
  if (!strcmp(key, "mask_ctas")) return &h->mask_ctas;
  if (!strcmp(key, "mask_cctas")) return &h->mask_cctas;
  if (!strcmp(key, "mask2_prefetch")) return &h->mask2_prefetch;
  if (!strcmp(key, "mask_group")) return &h->mask_group;
  if (!strcmp(key, "mask_prefetch")) return &h->mask_prefetch;
  if (!strcmp(key, "mask_window")) return &h->mask_window;
  if (!strcmp(key, "mask_wgroup")) return &h->mask_wgroup;
  if (!strcmp(key, "nvtx")) return &h->nvtx;
  if (!strcmp(key, "dist_fuse_push")) return &h->dist_fuse_push;
  if (!strcmp(key, "dist_fold")) return &h->dist_fold;
  if (!strcmp(key, "tma_stages")) return &h->tma_stages;
  if (!strcmp(key, "use_tma")) return &h->use_tma;
  if (!strcmp(key, "dist_p2p")) return &h->dist_p2p;
  if (!strcmp(key, "use_compress")) return &h->use_compress;
  if (!strcmp(key, "use_split")) return &h->use_split;
  if (!strcmp(key, "persistent")) return &h->persistent;
  if (!strcmp(key, "persistent_max_n")) return &h->persistent_max_n;
  if (!strcmp(key, "persistent_cluster")) return &h->persistent_cluster;
  if (!strcmp(key, "prefetch_x")) return &h->prefetch_x;
  if (!strcmp(key, "loop_mode")) return &h->loop_mode;
  if (!strcmp(key, "chunk")) return &h->chunk;
  if (!strcmp(key, "fuse_xpay")) return &h->fuse_xpay;
  if (!strcmp(key, "snake")) return &h->snake;
  if (!strcmp(key, "l2_hints")) return &h->l2_hints;
  if (!strcmp(key, "cg_lag_x")) return &h->cg_lag_x;
  if (!strcmp(key, "mask_const")) return &h->mask_const;
  return nullptr;
}

extern "C" int bk_set_option(bk_handle* h, const char* key, int64_t value) {
  if (!h) return bk_fail(BK_ERR_ARG, "bk_set_option: null handle");
  int* f = bk_opt_field(h, key);
  if (!f) return bk_fail(BK_ERR_ARG, "bk_set_option: unknown key '%s'", key ? key : "(null)");
  if ((!strcmp(key, "grid_mult_vec") || !strcmp(key, "grid_mult_spmv") || !strcmp(key, "grid_mult")) &&
      (value < 1 || value * h->num_sms > BK_MAXB))
    return bk_fail(BK_ERR_ARG, "bk_set_option: %s=%lld out of range", key, (long long)value);
  if (!strcmp(key, "grid_mult")) h->grid_mult_vec = (int)value;
  *f = (int)value;
  bk_graphs_invalidate(h);
  return BK_OK;
}

extern "C" int64_t bk_get_option(bk_handle* h, const char* key) {
  if (!h) return -1;
  int* f = bk_opt_field(h, key);
  return f ? *f : -1;
}

extern "C" int bk_device_info(bk_handle* h, int32_t* num_sms, int64_t* l2_bytes, int64_t* mem_bytes) {
  if (!h) return bk_fail(BK_ERR_ARG, "bk_device_info: null handle");
  if (num_sms) *num_sms = h->num_sms;
  if (l2_bytes) *l2_bytes = h->l2_bytes;
  if (mem_bytes) *mem_bytes = h->mem_bytes;
  return BK_OK;
}

// ------------------------------------------------------------------------------------------
// matrix registration
// ------------------------------------------------------------------------------------------
__global__ void bk_cvt_i64_i32_kernel(const long long* __restrict__ in, int* __restrict__ out, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (int)in[i];
}

void bk_convert_i64_i32(bk_handle* h, const void* in, void* out, long long n, cudaStream_t s) {
  if (n > 0) bk_cvt_i64_i32_kernel<<<h->num_sms * 8, 256, 0, s>>>((const long long*)in, (int*)out, n);
}

// max row length + validity (monotone rowptr, columns in range) in one pass over rowptr/col
__global__ void bk_csr_stats_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, long long n,
                                    long long n_cols, long long nnz,
                                    int* __restrict__ out /* [0] max len, [1] bad flag */) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  int mx = 0;
  int bad = 0;
  for (long long i = tid; i < n; i += stride) {
    const int a = rowptr[i], b = rowptr[i + 1];
    if (b < a) bad = 1;
    mx = max(mx, b - a);
  }
  for (long long i = tid; i < nnz; i += stride) {
    const int c = col[i];
    if (c < 0 || c >= n_cols) bad = 1;
  }
  for (int o = 16; o > 0; o >>= 1) {
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&out[0], mx);
    if (bad) atomicOr(&out[1], 1);
  }
}

static void bk_csr_plan(bk_handle* h, bk_csr* A) {
  const double mean = A->n > 0 ? (double)A->nnz / (double)A->n : 0.0;
  A->mean_row_nnz = mean;
  const double skew_limit = 64.0 * (mean > 8.0 ? mean : 8.0);
  int kernel = (mean <= 32.0 && (double)A->max_row_nnz <= skew_limit) ? 0 : 1;
  const int64_t forced = bk_env_int("BK_SPMV_KERNEL", -1);
  if (forced == 0 || forced == 1) kernel = (int)forced;
  A->kernel = kernel;
  A->cap = (mean <= 8.0) ? 256 : 1024;
  A->lanes_per_row = (mean <= 64.0) ? 8 : (mean <= 128.0 ? 16 : 32);
  (void)h;
}

// ---- long-row splitting for skewed row-length distributions --------------------------------------------------
// count[r] = number of virtual rows of real row r (at least 1, so empty rows keep a slot)
__global__ void bk_vrow_count_kernel(const int* __restrict__ rowptr, long long n, unsigned int* __restrict__ cnt) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += stride) {
    if (r == n) {
      cnt[r] = 0;
    } else {
      const int len = rowptr[r + 1] - rowptr[r];
      cnt[r] = len <= BK_SPLIT_LEN ? 1u : (unsigned int)((len + BK_SPLIT_LEN - 1) / BK_SPLIT_LEN);
    }
  }
}
// vrowptr: virtual row v of real row r covers entries [rowptr[r] + i*L, min(rowptr[r] + (i+1)*L, rowptr[r+1]))
__global__ void bk_vrow_fill_kernel(const int* __restrict__ rowptr, const int* __restrict__ vstart, long long n,
                                    int* __restrict__ vrowptr) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
    const int s = rowptr[r], e = rowptr[r + 1];
    const int v0 = vstart[r], v1 = vstart[r + 1];
    for (int v = v0; v < v1; ++v) vrowptr[v] = s + (v - v0) * BK_SPLIT_LEN;
    if (r == n - 1) vrowptr[v1] = e;
  }
}

static int bk_csr_plan_split(bk_handle* h, bk_csr* A, cudaStream_t s) {
  // only for short-mean matrices with a few very long rows (the row-stream kernels would serialise on them and
  // the warp-per-row kernel wastes 31 lanes on every short row)
  const double mean = A->mean_row_nnz;
  if (A->is_view || !h->use_split || A->n == 0 || mean > 32.0) return BK_OK;
  if ((double)A->max_row_nnz <= 64.0 * (mean > 8.0 ? mean : 8.0)) return BK_OK;
  const long long n = A->n;
  unsigned int* cnt = nullptr;
  if (bk_pool_alloc((void**)&cnt, sizeof(unsigned int) * (size_t)(n + 1), s) != cudaSuccess)
    return bk_fail(BK_ERR_ALLOC, "row splitting: allocation failed");
  const int g = h->num_sms * 8;
  bk_vrow_count_kernel<<<g, 256, 0, s>>>(A->rowptr, n, cnt);
  int rc = bk_exclusive_scan_u32(cnt, n + 1, s);
  if (rc != BK_OK) {
    bk_pool_free(cnt);
    return rc;
  }
  unsigned int nv_u = 0;
  cudaMemcpyAsync(&nv_u, cnt + n, sizeof(unsigned int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    bk_pool_free(cnt);
    return bk_fail(BK_ERR_CUDA, "row splitting: %s", cudaGetErrorString(e));
  }
  const long long nv = (long long)nv_u;
  A->vstart = (int*)cnt;  // exclusive scan of the counts == first virtual row of every real row (n+1 entries)
  bk_csr* S = (bk_csr*)calloc(1, sizeof(bk_csr));
  if (!S) return bk_fail(BK_ERR_ALLOC, "row splitting: host allocation failed");
  S->h = h;
  S->n = nv;
  S->nnz = A->nnz;
  S->dtype = A->dtype;
  S->col = A->col;
  S->val = A->val;
  S->is_view = 1;
  S->uid = h->next_uid++;
  A->split = S;
  if (bk_pool_alloc(&S->own_rowptr, sizeof(int) * (size_t)(nv + 1), s) != cudaSuccess ||
      bk_pool_alloc(&A->yv, bk_dtype_size(A->dtype) * (size_t)(nv > 0 ? nv : 1), s) != cudaSuccess)
    return bk_fail(BK_ERR_ALLOC, "row splitting: allocation failed");
  S->rowptr = (const int*)S->own_rowptr;
  bk_vrow_fill_kernel<<<g, 256, 0, s>>>(A->rowptr, A->vstart, n, (int*)S->own_rowptr);
  A->kernel = 4;
  return bk_csr_finish_plan(h, S, s);  // statistics + kernel choice (row-stream / TMA) for the virtual rows
}

// widest 16-byte aligned val/col span of any 256-row block: max over blocks of ((e+3)&~3) - (s&~3)
__global__ void bk_block_span_kernel(const int* __restrict__ rowptr, long long n, long long nblk, int rpb, int al,
                                     int* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  int mx = 0;
  for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += stride) {
    const long long r0 = b * rpb;
    const long long r1 = (r0 + rpb < n) ? r0 + rpb : n;
    const int s = rowptr[r0], e = rowptr[r1];
    mx = max(mx, ((e + al - 1) & ~(al - 1)) - (s & ~(al - 1)));
  }
  for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, mx);
}

// ---- 8-bit dictionary coding of the column stream (kernel 3) ---------------------------------------------------
// For every 256-row block collect the distinct (column - row) offsets; if no block has more than 32 of them (all
// stencil / structured-grid matrices), each column index is replaced by a 1-byte code into its block's dictionary.
#define BK_DICT_EMPTY ((int)0x80000000)
__global__ void __launch_bounds__(256)
bk_build_dict_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, long long n, long long nblk,
                     int* __restrict__ dict, unsigned char* __restrict__ codes, int* __restrict__ fail) {
  __shared__ int tab[32];
  for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    if (threadIdx.x < 32) tab[threadIdx.x] = BK_DICT_EMPTY;
    __syncthreads();
    const long long r = blk * 256 + threadIdx.x;
    if (r < n) {
      for (int k = rowptr[r]; k < rowptr[r + 1]; ++k) {
        const int off = col[k] - (int)r;
        int code = -1;
        for (int i = 0; i < 32 && code < 0; ++i) {
          int old = ((volatile int*)tab)[i];
          if (old == BK_DICT_EMPTY) old = atomicCAS(&tab[i], BK_DICT_EMPTY, off);
          if (old == BK_DICT_EMPTY || old == off) code = i;
        }
        if (code < 0) {
          *fail = 1;
          code = 0;
        }
        codes[k] = (unsigned char)code;
      }
    }
    __syncthreads();
    if (threadIdx.x < 32) dict[blk * 32 + threadIdx.x] = (tab[threadIdx.x] == BK_DICT_EMPTY) ? 0 : tab[threadIdx.x];
    __syncthreads();
  }
}

static int bk_csr_plan_compress(bk_handle* h, bk_csr* A, cudaStream_t s) {
  if (A->kernel != 2 || !h->use_compress) return BK_OK;
  const long long nblk = (A->n + 255) / 256;
  const size_t vs = bk_dtype_size(A->dtype);
  int* dstat = (int*)(h->counters + 8);
  int host[2] = {0, 0};
  if (bk_pool_alloc((void**)&A->codes, (size_t)A->nnz + 64, s) != cudaSuccess ||
      bk_pool_alloc((void**)&A->dict, sizeof(int) * 32 * (size_t)nblk, s) != cudaSuccess) {
    cudaGetLastError();
    if (A->codes) bk_pool_free(A->codes);
    if (A->dict) bk_pool_free(A->dict);
    A->codes = nullptr;
    A->dict = nullptr;
    return BK_OK;  // not enough memory for the coded copy: stay on int32 columns
  }
  cudaMemsetAsync(dstat, 0, 2 * sizeof(int), s);
  int grid = (int)(nblk < (long long)h->num_sms * 8 ? nblk : (long long)h->num_sms * 8);
  bk_build_dict_kernel<<<grid, 256, 0, s>>>(A->rowptr, A->col, A->n, nblk, A->dict, A->codes, dstat + 1);
  bk_block_span_kernel<<<h->num_sms * 4, 256, 0, s>>>(A->rowptr, A->n, nblk, 256, 16, dstat);
  cudaMemcpyAsync(host, dstat, 2 * sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (index coding): %s", cudaGetErrorString(e));
  const int cap = (host[0] + 31) & ~31;
  const size_t stage = (size_t)cap * (vs + 1) + 128;
  if (host[1] != 0 || cap <= 0 || 2 * stage > 110 * 1024) {  // a block with > 32 distinct offsets, or too wide
    bk_pool_free(A->codes);
    bk_pool_free(A->dict);
    A->codes = nullptr;
    A->dict = nullptr;
    return BK_OK;
  }
  const int tail = (int)(A->nnz & 15);
  if (tail) {
    if (bk_pool_alloc(&A->tail_val16, 16 * vs, s) != cudaSuccess || bk_pool_alloc((void**)&A->tail_code16, 16, s) != cudaSuccess) {
      cudaGetLastError();
      return bk_fail(BK_ERR_ALLOC, "csr registration: tail buffer allocation failed");
    }
    const int64_t base = A->nnz & ~(int64_t)15;
    cudaMemsetAsync(A->tail_val16, 0, 16 * vs, s);
    cudaMemsetAsync(A->tail_code16, 0, 16, s);
    cudaMemcpyAsync(A->tail_val16, (const char*)A->val + base * vs, tail * vs, cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(A->tail_code16, A->codes + base, tail, cudaMemcpyDeviceToDevice, s);
    e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (coded tail): %s", cudaGetErrorString(e));
  }
  A->cmp_cap = cap;
  A->kernel = 3;
  A->bytes_stream = A->nnz * (int64_t)(vs + 1) + nblk * 128 + (A->n + 1) * 4;
  return BK_OK;
}

// ---- 8-bit coding of (column - row, value) PAIRS, SELL-32-4 layout (kernel 5, bk_spmv_pair.cuh) ---------------
// bytes of every 256-row block's span: 128-byte header + per 32-row chunk (longest row rounded up to 4) x 32 lanes
__global__ void bk_pair_block_bytes_kernel(const int* __restrict__ rowptr, long long n, long long nblk,
                                           unsigned int* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long blk = warp0; blk < nblk; blk += nwarps) {
    unsigned int units = BK_PAIR_HDR_BYTES / 128;
    for (int pass = 0; pass < 8; ++pass) {
      const long long r = blk * 256 + pass * 32 + lane;
      int len = (r < n) ? rowptr[r + 1] - rowptr[r] : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
      units += (unsigned int)((len + 3) >> 2);
    }
    if (lane == 0) out[blk] = units * 128u;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[nblk] = 0u;
}

// One warp per 256-row block.  Lane i keeps dictionary entry i in registers; the warp walks its 8 chunks of 32 rows,
// entry position by entry position: the (offset, value-bits) pairs of the 32 lanes are grouped (leader broadcast +
// ballot), each group is looked up in / appended to the dictionary by one ballot, and every lane stores the code of
// its entry at its SELL position.  A block with more than 31 distinct pairs sets `fail` (slot 31 is the zero entry).
template <typename T>
__global__ void __launch_bounds__(256)
bk_build_pair_dict_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const T* __restrict__ val,
                          long long n, long long nblk, const int* __restrict__ bptr,
                          bk_pair_entry* __restrict__ dict, unsigned char* __restrict__ codes, int* __restrict__ fail) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * 8;
  for (long long blk = warp0; blk < nblk; blk += nwarps) {
    int t_off = 0;
    unsigned long long t_val = 0ull;
    int count = 0;
    bool bad = false;
    unsigned char* span = codes + bptr[blk];
    unsigned int unit = BK_PAIR_HDR_BYTES / 128;  // running chunk start, in 128-byte units from the span start
    for (int pass = 0; pass < 8; ++pass) {
      const long long r = blk * 256 + pass * 32 + lane;
      int s = 0, e = 0;
      if (r < n) {
        s = rowptr[r];
        e = rowptr[r + 1];
      }
      int maxlen = e - s;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
      const unsigned int words = (unsigned int)((maxlen + 3) >> 2);
      if (lane == 0) reinterpret_cast<unsigned int*>(span)[pass] = ((unit + words) << 16) | unit;
      unsigned char* out = span + (size_t)unit * 128 + lane * 4;
      unit += words;
      for (int k = 0; k < maxlen && !bad; ++k) {
        const bool active = k < e - s;
        int off = 0;
        unsigned long long vb = 0ull;
        if (active) {
          off = col[s + k] - (int)r;
          if (sizeof(T) == 8) vb = (unsigned long long)__double_as_longlong((double)val[s + k]);
          else vb = (unsigned long long)__float_as_uint((float)val[s + k]);
        }
        unsigned int remaining = __ballot_sync(0xffffffffu, active);
        int code = 0;
        while (remaining) {
          const int leader = __ffs(remaining) - 1;
          const int lo = __shfl_sync(0xffffffffu, off, leader);
          const unsigned long long lv = __shfl_sync(0xffffffffu, vb, leader);
          const bool same = active && off == lo && vb == lv;
          const unsigned int grp = __ballot_sync(0xffffffffu, same);
          const unsigned int hit = __ballot_sync(0xffffffffu, lane < count && t_off == lo && t_val == lv);
          int idx;
          if (hit) {
            idx = __ffs(hit) - 1;
          } else {
            idx = count;
            if (count >= BK_PAIR_ZERO) {
              bad = true;
              idx = 0;
            } else {
              if (lane == count) {
                t_off = lo;
                t_val = lv;
              }
              ++count;
            }
          }
          if (same) code = idx;
          remaining &= ~grp;
        }
        if (active) out[(k >> 2) * 128 + (k & 3)] = (unsigned char)code;
      }
    }
    if (bad && lane == 0) *fail = 1;
    bk_pair_entry ent;
    ent.val = (lane < count) ? t_val : 0ull;
    ent.off = (lane < count) ? t_off : 0;
    ent.pad = 0;
    dict[blk * 32 + lane] = ent;
  }
}

// Try the pair-coded stream (kernel 5); on success one SpMV reads neither val, col nor rowptr.
static int bk_csr_plan_pairs(bk_handle* h, bk_csr* A, cudaStream_t s) {
  if (A->kernel != 2 || h->use_compress < 2) return BK_OK;
  // virtual-row views (kernel 4) number their rows beyond the length of x: the padding entries' x[row] would be out
  // of bounds there
  if (A->is_view) return BK_OK;
  const long long nblk = (A->n + 255) / 256;
  int* dstat = (int*)(h->counters + 8);
  auto drop = [&]() {
    if (A->pcodes) bk_pool_free(A->pcodes);
    if (A->pdict) bk_pool_free(A->pdict);
    if (A->pbptr) bk_pool_free(A->pbptr);
    A->pcodes = nullptr;
    A->pdict = nullptr;
    A->pbptr = nullptr;
  };
  if (bk_pool_alloc((void**)&A->pbptr, sizeof(int) * (size_t)(nblk + 1), s) != cudaSuccess) {
    cudaGetLastError();
    return BK_OK;
  }
  bk_pair_block_bytes_kernel<<<h->num_sms * 8, 256, 0, s>>>(A->rowptr, A->n, nblk, (unsigned int*)A->pbptr);
  int rc = bk_exclusive_scan_u32((unsigned int*)A->pbptr, nblk + 1, s);
  if (rc != BK_OK) {
    drop();
    return rc;
  }
  unsigned int total = 0;
  cudaMemcpyAsync(&total, A->pbptr + nblk, sizeof(unsigned int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (pair coding): %s", cudaGetErrorString(e));
  // padding must stay modest (rows of similar length inside each chunk) and offsets must fit an int
  if ((double)total > 1.5 * (double)A->nnz + 1152.0 * (double)nblk || total >= 0x7fffff00u || total == 0) {
    drop();
    return BK_OK;
  }
  if (bk_pool_alloc((void**)&A->pcodes, (size_t)total + 128, s) != cudaSuccess ||
      bk_pool_alloc(&A->pdict, sizeof(bk_pair_entry) * 32 * (size_t)nblk, s) != cudaSuccess) {
    cudaGetLastError();
    drop();
    return BK_OK;  // not enough memory for the coded copy
  }
  int host[2] = {0, 0};
  cudaMemsetAsync(dstat, 0, 2 * sizeof(int), s);
  cudaMemsetAsync(A->pcodes, BK_PAIR_ZERO, (size_t)total + 128, s);
  long long want = (nblk + 7) / 8;
  int grid = (int)(want < (long long)h->num_sms * 8 ? want : (long long)h->num_sms * 8);
  if (grid < 1) grid = 1;
  if (A->dtype == BK_F64)
    bk_build_pair_dict_kernel<double><<<grid, 256, 0, s>>>(A->rowptr, A->col, (const double*)A->val, A->n, nblk,
                                                          A->pbptr, (bk_pair_entry*)A->pdict, A->pcodes, dstat + 1);
  else
    bk_build_pair_dict_kernel<float><<<grid, 256, 0, s>>>(A->rowptr, A->col, (const float*)A->val, A->n, nblk,
                                                         A->pbptr, (bk_pair_entry*)A->pdict, A->pcodes, dstat + 1);
  bk_block_span_kernel<<<h->num_sms * 4, 256, 0, s>>>(A->pbptr, nblk, nblk, 1, 128, dstat);
  cudaMemcpyAsync(host, dstat, 2 * sizeof(int), cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (pair coding): %s", cudaGetErrorString(e));
  const int cap = (host[0] + 127) & ~127;
  const size_t stage = (size_t)cap + BK_PAIR_DICT_BYTES;
  if (host[1] != 0 || cap <= 0 || 2 * stage > 110 * 1024) {  // a block with > 31 distinct pairs, or too wide
    drop();
    return BK_OK;
  }
  A->pair_cap = cap;
  A->kernel = 5;
  A->bytes_stream = (int64_t)total + nblk * (int64_t)BK_PAIR_DICT_BYTES + (nblk + 1) * 4;
  return BK_OK;
}

// ---- row bitmasks over per-chunk patterns of (column - row, value) pairs (kernel 6, bk_spmv_mask.cuh) -------------
// One warp per 32-row chunk: (1) collect the chunk's distinct pairs (lane i keeps pair i; leader broadcast + ballot as
// in the pair-dictionary builder above); (2) rank them by (global offset, value bits, ...) -> the sorted PATTERN;
// (3) every lane ORs the ranks of its row's entries into its mask and checks that they ascend, i.e. that the pattern
// order is the CSR order of every row (the SpMV then reproduces the CSR FMA chain bit for bit).
// Row-partitioned matrices (n_cols > n): columns >= n index the ghost vector; `ghost_gid` gives their global ids and
// `row_begin` the global id of row 0, so that pairs are ordered by GLOBAL offset like the rows of the global matrix.
struct bk_mask_key {
  long long goff;          // global column - global row (sort key)
  unsigned long long vb;   // value bits
  int off;                 // load offset: index into x (or the ghost vector) minus the local row
  int gh;                  // 1: ghost entry
};
__device__ __forceinline__ bool bk_mask_less(const bk_mask_key& a, const bk_mask_key& b) {
  if (a.goff != b.goff) return a.goff < b.goff;
  if (a.vb != b.vb) return a.vb < b.vb;
  if (a.gh != b.gh) return a.gh < b.gh;
  return a.off < b.off;
}
__device__ __forceinline__ bool bk_mask_same(const bk_mask_key& a, const bk_mask_key& b) {
  return a.goff == b.goff && a.vb == b.vb && a.gh == b.gh && a.off == b.off;
}
__device__ __forceinline__ bk_mask_key bk_mask_shfl(const bk_mask_key& k, int src) {
  bk_mask_key r;
  r.goff = __shfl_sync(0xffffffffu, k.goff, src);
  r.vb = __shfl_sync(0xffffffffu, k.vb, src);
  r.off = __shfl_sync(0xffffffffu, k.off, src);
  r.gh = __shfl_sync(0xffffffffu, k.gh, src);
  return r;
}

template <typename T>
__global__ void __launch_bounds__(256)
bk_mask_build_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const T* __restrict__ val,
                     long long n, long long nchunks, const long long* __restrict__ ghost_gid, long long row_begin,
                     bk_pair_entry* __restrict__ cpat, unsigned char* __restrict__ masks, int* __restrict__ pids,
                     int* __restrict__ fail) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * 8;
  for (long long ch = warp0; ch < nchunks; ch += nwarps) {
    if (*(volatile int*)fail) return;  // another chunk already disqualified the matrix
    const long long r = ch * 32 + lane;
    int s = 0, e = 0;
    if (r < n) {
      s = rowptr[r];
      e = rowptr[r + 1];
    }
    const int len = e - s;
    int maxlen = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
    bool bad = maxlen > BK_MASK_L;
    bk_mask_key tab;  // lane i < count holds pattern entry i (unsorted)
    tab.goff = 0;
    tab.vb = 0ull;
    tab.off = 0;
    tab.gh = 0;
    int count = 0;
    int codes[BK_MASK_L];
    int any_ghost = 0;
#pragma unroll
    for (int k = 0; k < BK_MASK_L; ++k) {
      codes[k] = 0;
      if (k < maxlen && !bad) {  // warp-uniform
        const bool active = k < len;
        bk_mask_key me;
        me.goff = 0;
        me.vb = 0ull;
        me.off = 0;
        me.gh = 0;
        if (active) {
          const int c = col[s + k];
          if ((long long)c >= n) {  // ghost column of a row-partitioned matrix
            me.gh = 1;
            me.off = (int)((long long)c - n - r);
            me.goff = ghost_gid[c - n] - (row_begin + r);
          } else {
            me.off = (int)((long long)c - r);
            me.goff = (long long)c - r;
          }
          if (sizeof(T) == 8) me.vb = (unsigned long long)__double_as_longlong((double)val[s + k]);
          else me.vb = (unsigned long long)__float_as_uint((float)val[s + k]);
        }
        any_ghost |= me.gh;
        unsigned int remaining = __ballot_sync(0xffffffffu, active);
        while (remaining) {
          const int leader = __ffs(remaining) - 1;
          const bk_mask_key lk = bk_mask_shfl(me, leader);
          const bool same = active && bk_mask_same(me, lk);
          const unsigned int grp = __ballot_sync(0xffffffffu, same);
          const unsigned int hit = __ballot_sync(0xffffffffu, lane < count && bk_mask_same(tab, lk));
          int idx;
          if (hit) {
            idx = __ffs(hit) - 1;
          } else if (count >= BK_MASK_L) {
            bad = true;
            idx = 0;
          } else {
            idx = count;
            if (lane == count) tab = lk;
            ++count;
          }
          if (same) codes[k] = idx;
          remaining &= ~grp;
        }
      }
    }
    // rank of every table entry in the sorted pattern
    int rank = 0;
    for (int j = 0; j < count; ++j) {
      const bk_mask_key kj = bk_mask_shfl(tab, j);
      if (lane < count && bk_mask_less(kj, tab)) ++rank;
    }
    unsigned int mask = 0u;
    int prev = -1;
    bool disorder = false;
#pragma unroll
    for (int k = 0; k < BK_MASK_L; ++k) {
      const int rk = __shfl_sync(0xffffffffu, rank, codes[k]);
      if (k < len) {
        if (rk <= prev) disorder = true;  // columns not ascending / repeated inside the row
        prev = rk;
        mask |= 1u << rk;
      }
    }
    if (__any_sync(0xffffffffu, disorder)) bad = true;
    any_ghost = __any_sync(0xffffffffu, any_ghost != 0) ? 1 : 0;
    if (bad) {
      if (lane == 0) *fail = 1;
      return;
    }
    masks[ch * 32 + lane] = (unsigned char)((r < n) ? mask : 0u);
    bk_pair_entry ent;
    ent.val = 0ull;
    ent.off = 0;
    ent.pad = 0;
    const int full = (1 << count) - 1;  // mask of a row that has every entry; kept in entry 0 (bk_mask_load_pattern)
    if (lane < count) {
      ent.val = tab.vb;
      ent.off = tab.off;
      ent.pad = (tab.gh ? BK_MASK_GHOST : 0) | (rank == 0 ? (full << BK_MASK_FULL_SHIFT) : 0);
      cpat[ch * BK_MASK_L + rank] = ent;
    } else if (lane < BK_MASK_L) {
      cpat[ch * BK_MASK_L + lane] = ent;  // lanes count..7 fill the unused tail (ranks cover 0..count-1)
    }
    if (lane == 0) pids[ch] = any_ghost ? BK_MASK_PID_GHOST : 0;
  }
}

__device__ __forceinline__ unsigned long long bk_mix64(unsigned long long x) {
  x ^= x >> 30;
  x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27;
  x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}

// De-duplicate the chunk patterns into an open-addressing table keyed by a 64-bit hash of the 128 pattern bytes; the
// chunk that claims a slot stores its pattern there.  bk_mask_verify_kernel (next launch) compares every chunk's pattern
// with the stored one, so a hash collision disqualifies the matrix instead of corrupting it.
__global__ void bk_mask_insert_kernel(const bk_pair_entry* __restrict__ cpat, long long nchunks,
                                      unsigned long long* __restrict__ keys, bk_pair_entry* __restrict__ ptab,
                                      int* __restrict__ pids, int* __restrict__ stat /* [0] fail [1] patterns */) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x; ch < nchunks; ch += stride) {
    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(cpat + ch * BK_MASK_L);
    ulonglong2 q[BK_MASK_L];
    unsigned long long hsh = 0x9e3779b97f4a7c15ull;
#pragma unroll
    for (int e = 0; e < BK_MASK_L; ++e) {
      q[e] = src[e];
      hsh = bk_mix64(hsh ^ q[e].x) + 0x632be59bd9b4e019ull;
      hsh = bk_mix64(hsh ^ q[e].y);
    }
    if (hsh == 0ull) hsh = 1ull;
    int slot = (int)(hsh & (BK_MASK_HT - 1));
    bool found = false;
    for (int probe = 0; probe < BK_MASK_HT; ++probe) {
      const unsigned long long old = atomicCAS(&keys[slot], 0ull, hsh);
      if (old == 0ull) {
        atomicAdd(&stat[1], 1);
        ulonglong2* dst = reinterpret_cast<ulonglong2*>(ptab + (size_t)slot * BK_MASK_L);
#pragma unroll
        for (int e = 0; e < BK_MASK_L; ++e) dst[e] = q[e];
        found = true;
        break;
      }
      if (old == hsh) {
        found = true;
        break;
      }
      slot = (slot + 1) & (BK_MASK_HT - 1);
    }
    if (!found) stat[0] = 2;
    pids[ch] |= slot;
  }
}

__global__ void bk_mask_verify_kernel(const bk_pair_entry* __restrict__ cpat, long long nchunks,
                                      const bk_pair_entry* __restrict__ ptab, const int* __restrict__ pids,
                                      int* __restrict__ stat) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x; ch < nchunks; ch += stride) {
    const ulonglong2* a = reinterpret_cast<const ulonglong2*>(cpat + ch * BK_MASK_L);
    const ulonglong2* b =
        reinterpret_cast<const ulonglong2*>(ptab + (size_t)(pids[ch] & (BK_MASK_PID_GHOST - 1)) * BK_MASK_L);
    bool same = true;
#pragma unroll
    for (int e = 0; e < BK_MASK_L; ++e) {
      const ulonglong2 x = a[e], y = b[e];
      same = same && x.x == y.x && x.y == y.y;
    }
    if (!same) stat[0] = 3;
  }
}

// flags[ch] = 1 for chunks with ghost entries -> (after an exclusive scan) their compact list
__global__ void bk_mask_flag_kernel(const int* __restrict__ pids, long long nchunks, unsigned int* __restrict__ flags) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x; ch <= nchunks; ch += stride)
    flags[ch] = (ch < nchunks && (pids[ch] & BK_MASK_PID_GHOST)) ? 1u : 0u;
}
__global__ void bk_mask_compact_kernel(const int* __restrict__ pids, long long nchunks,
                                       const unsigned int* __restrict__ pos, int* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x; ch < nchunks; ch += stride)
    if (pids[ch] & BK_MASK_PID_GHOST) out[pos[ch]] = (int)ch;
}

// Try the row-bitmask plan (kernel 6).  ghost_gid / row_begin: see bk_mask_build_kernel (nullptr / 0 on one GPU).
// kernel 7: every row's presence bits in UNION numbering, and one summary per 64-row step (two 32-row chunks): pattern
// id, "some row lacks an entry of its pattern", "two patterns / matrix end within reach of the gathers".
struct bk_mask_umap {
  unsigned char pos[BK_MASK_CP][BK_MASK_L];  // union position of entry k of pattern p
  unsigned int fullu[BK_MASK_CP];            // union bits of a complete row of pattern p
};
static __global__ void bk_mask_usum_kernel(const unsigned char* __restrict__ masks, const int* __restrict__ pids,
                                           const unsigned char* __restrict__ slot2dense, const bk_mask_umap um,
                                           const long long n, const long long nsteps, const long long minoff,
                                           const long long maxoff, const int kc, unsigned char* __restrict__ umasks,
                                           unsigned short* __restrict__ usum, int* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long st = warp; st < nsteps; st += nwarps) {
    const long long r0 = st * 64;
    // pairs are loaded with one element of slack on both sides: everything must stay inside [0, n rounded down to a pair)
    bool mixed = r0 + 64 > n || r0 + minoff - 1 < 0 || r0 + 63 + maxoff + 1 >= (n & ~1LL);
    bool dirty = false;      // some row lacks an entry of its pattern, other than the two edge cases below
    bool lo_miss = false;    // the step's first row lacks (only) the -1 neighbour: union position kc - 1
    bool hi_miss = false;    // the step's last row lacks (only) the +1 neighbour: union position kc + 1
    int pid0 = 0;
    for (int u = 0; u < 2; ++u) {
      const long long c = st * 2 + u;  // (masks / pids are padded to whole groups)
      const int praw = pids[c];
      if (praw & BK_MASK_PID_GHOST) mixed = true;  // (row partition) ghost entries: the chunk waits for the halo
      int pid = (int)slot2dense[praw & (BK_MASK_HT - 1)];
      if (pid >= BK_MASK_CP) pid = 0;
      if (u == 0) pid0 = pid;
      if (pid != pid0) mixed = true;
      const unsigned int m = masks[c * 32 + lane];
      unsigned int mu = 0u;
#pragma unroll
      for (int k = 0; k < BK_MASK_L; ++k) mu |= ((m >> k) & 1u) << um.pos[pid][k];
      umasks[c * 32 + lane] = (unsigned char)mu;
      unsigned int miss = um.fullu[pid] & ~mu;
      if (kc >= 1 && u == 0 && lane == 0 && miss == (1u << (kc - 1))) {
        lo_miss = true;
        miss = 0u;
      }
      if (kc >= 1 && u == 1 && lane == 31 && miss == (1u << (kc + 1))) {
        hi_miss = true;
        miss = 0u;
      }
      dirty = dirty || __any_sync(0xffffffffu, miss != 0u);
    }
    lo_miss = __any_sync(0xffffffffu, lo_miss);
    hi_miss = __any_sync(0xffffffffu, hi_miss);
    if (lane == 0) {
      // step st = (group g, step j, warp w) in row order; stored as [g][w][j]: a warp reads its four summaries at once
      const long long g = st >> 5;
      const int j = (int)((st >> 3) & 3), w = (int)(st & 7);
      // (a step that reads masks anyway gets its edge operands zeroed by them: the edge flags are for mask-free steps)
      usum[(g * 8 + w) * 4 + j] =
          (unsigned short)(pid0 | (dirty ? BK_MASK_US_DIRTY : 0) | (mixed ? BK_MASK_US_MIXED : 0) |
                           ((lo_miss && !dirty) ? BK_MASK_US_LO : 0) | ((hi_miss && !dirty) ? BK_MASK_US_HI : 0));
      if (mixed) atomicAdd(&counts[1], 1);
      else if (dirty) atomicAdd(&counts[0], 1);
    }
  }
}

int bk_csr_plan_mask(bk_handle* h, bk_csr* A, const long long* ghost_gid, long long row_begin, cudaStream_t s) {
  if (h->use_compress < 3 || A->is_view || A->n == 0 || A->nnz == 0 || A->max_row_nnz > BK_MASK_L) return BK_OK;
  const long long nchunks = (A->n + 31) / 32;
  const long long nblk8 = ((A->n + 255) / 256 + 32) * 8;  // chunks of whole 256-row blocks + 32 blocks of padding: the
                                                          // kernel walks whole groups of up to 32 blocks without a tail test
  bk_pair_entry* cpat = nullptr;
  unsigned long long* keys = nullptr;
  int* dstat = (int*)(h->counters + 8);
  auto drop = [&]() {
    if (A->mmasks) bk_pool_free(A->mmasks);
    if (A->mpids) bk_pool_free(A->mpids);
    if (A->mptab) bk_pool_free(A->mptab);
    if (A->mdeferred) bk_pool_free(A->mdeferred);
    if (A->musum) bk_pool_free(A->musum);
    if (A->mumasks) bk_pool_free(A->mumasks);
    A->musum = nullptr;
    A->mumasks = nullptr;
    A->mu_len = 0;
    A->mmasks = nullptr;
    A->mpids = nullptr;
    A->mptab = nullptr;
    A->mdeferred = nullptr;
    A->n_mdeferred = 0;
  };
  auto done = [&](int rc) {
    if (cpat) bk_pool_free(cpat);
    if (keys) bk_pool_free(keys);
    return rc;
  };
  if (bk_pool_alloc((void**)&cpat, sizeof(bk_pair_entry) * BK_MASK_L * (size_t)nchunks, s) != cudaSuccess ||
      bk_pool_alloc((void**)&keys, sizeof(unsigned long long) * BK_MASK_HT, s) != cudaSuccess ||
      bk_pool_alloc((void**)&A->mmasks, (size_t)nblk8 * 32, s) != cudaSuccess ||
      bk_pool_alloc((void**)&A->mpids, sizeof(int) * (size_t)nblk8, s) != cudaSuccess ||
      bk_pool_alloc(&A->mptab, sizeof(bk_pair_entry) * BK_MASK_L * BK_MASK_HT, s) != cudaSuccess) {
    cudaGetLastError();
    drop();
    return done(BK_OK);  // not enough memory for the coded copy: other plans follow
  }
  int host[2] = {0, 0};
  cudaMemsetAsync(dstat, 0, 2 * sizeof(int), s);
  cudaMemsetAsync(keys, 0, sizeof(unsigned long long) * BK_MASK_HT, s);
  cudaMemsetAsync(A->mptab, 0, sizeof(bk_pair_entry) * BK_MASK_L * BK_MASK_HT, s);
  cudaMemsetAsync(A->mmasks, 0, (size_t)nblk8 * 32, s);
  cudaMemsetAsync(A->mpids, 0, sizeof(int) * (size_t)nblk8, s);
  long long want = (nchunks + 7) / 8;
  int grid = (int)(want < (long long)h->num_sms * 8 ? want : (long long)h->num_sms * 8);
  if (grid < 1) grid = 1;
  if (A->dtype == BK_F64)
    bk_mask_build_kernel<double><<<grid, 256, 0, s>>>(A->rowptr, A->col, (const double*)A->val, A->n, nchunks, ghost_gid,
                                                     row_begin, cpat, A->mmasks, A->mpids, dstat);
  else
    bk_mask_build_kernel<float><<<grid, 256, 0, s>>>(A->rowptr, A->col, (const float*)A->val, A->n, nchunks, ghost_gid,
                                                    row_begin, cpat, A->mmasks, A->mpids, dstat);
  cudaMemcpyAsync(host, dstat, sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    drop();
    return done(bk_fail(BK_ERR_CUDA, "csr registration (row bitmasks): %s", cudaGetErrorString(e)));
  }
  if (host[0] != 0) {  // some chunk has > 8 distinct pairs, or rows with unsorted / repeated columns
    drop();
    return done(BK_OK);
  }
  want = (nchunks + 255) / 256;
  grid = (int)(want < (long long)h->num_sms * 8 ? want : (long long)h->num_sms * 8);
  if (grid < 1) grid = 1;
  bk_mask_insert_kernel<<<grid, 256, 0, s>>>(cpat, nchunks, keys, (bk_pair_entry*)A->mptab, A->mpids, dstat);
  bk_mask_verify_kernel<<<grid, 256, 0, s>>>(cpat, nchunks, (const bk_pair_entry*)A->mptab, A->mpids, dstat);
  cudaMemcpyAsync(host, dstat, 2 * sizeof(int), cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    drop();
    return done(bk_fail(BK_ERR_CUDA, "csr registration (pattern table): %s", cudaGetErrorString(e)));
  }
  if (host[0] != 0 || host[1] > BK_MASK_HT / 2) {  // table overflow / hash collision: not a pattern matrix
    drop();
    return done(BK_OK);
  }
  A->mask_patterns = host[1];
  {  // window plan of kernel 6W: near half-width W and up to two far offsets, from the (small) pattern table
    const size_t ne = (size_t)BK_MASK_HT * BK_MASK_L;
    bk_pair_entry* tab = (bk_pair_entry*)malloc(sizeof(bk_pair_entry) * ne);
    unsigned long long* hk = (unsigned long long*)malloc(sizeof(unsigned long long) * BK_MASK_HT);
    A->mw_win = 0;
    A->mw_nfar = 0;
    if (tab && hk &&
        cudaMemcpyAsync(tab, A->mptab, sizeof(bk_pair_entry) * ne, cudaMemcpyDeviceToHost, s) == cudaSuccess &&
        cudaMemcpyAsync(hk, keys, sizeof(unsigned long long) * BK_MASK_HT, cudaMemcpyDeviceToHost, s) == cudaSuccess &&
        cudaStreamSynchronize(s) == cudaSuccess) {
      const int ea = (int)(16 / bk_dtype_size(A->dtype));
      int W = 0;
      int far[64];
      int nfar_all = 0;
      for (int slot = 0; slot < BK_MASK_HT; ++slot) {
        if (!hk[slot]) continue;
        const bk_pair_entry* pe = tab + (size_t)slot * BK_MASK_L;
        const int full = (pe[0].pad >> BK_MASK_FULL_SHIFT) & 0x1ff;
        for (int e = 0; e < BK_MASK_L; ++e) {
          if (!(full & (1 << e)) || (pe[e].pad & BK_MASK_GHOST)) continue;
          const int off = pe[e].off, ao = off < 0 ? -off : off;
          if (ao <= 1040) {
            if (ao > W) W = ao;
          } else {
            bool seen = false;
            for (int k = 0; k < nfar_all; ++k) seen = seen || far[k] == off;
            if (!seen && nfar_all < 64) far[nfar_all++] = off;
          }
        }
      }
      A->mw_win = ((W + 7) / 8) * 8;
      if (A->mw_win < 8) A->mw_win = 8;
      for (int k = 0; k < nfar_all && A->mw_nfar < 2; ++k)
        if (far[k] % ea == 0) A->mw_far[A->mw_nfar++] = far[k];
      // kernel 7 (fp64): up to BK_MASK_CP patterns, all sub-patterns of one set of <= 8 offsets, no ghost entries -> the
      // union's byte offsets and the per-pattern values as a kernel parameter block, masks in union numbering, one
      // summary per 64-row step
      if (A->dtype == BK_F64) {
        unsigned char* s2d = (unsigned char*)calloc(BK_MASK_HT, 1);
        unsigned char* d_s2d = nullptr;
        bk_mask_utab* ctb = (bk_mask_utab*)A->mctab;
        static_assert(sizeof(bk_mask_utab) <= sizeof(A->mctab), "parameter block does not fit bk_csr::mctab");
        memset(A->mctab, 0, sizeof(A->mctab));
        bk_mask_umap um;
        memset(&um, 0, sizeof(um));
        long long uni[BK_MASK_L];
        int nu = 0;
        bool ok = s2d != nullptr;
        for (int slot = 0; ok && slot < BK_MASK_HT; ++slot) {  // the union of the offsets, ascending
          if (!hk[slot]) continue;
          const bk_pair_entry* pe = tab + (size_t)slot * BK_MASK_L;
          const unsigned int full = (unsigned int)(pe[0].pad >> BK_MASK_FULL_SHIFT) & 0x1ffu;
          bool ghosty = false;  // (row partition) patterns with ghost entries belong to chunks of the second phase
          for (int e = 0; e < BK_MASK_L; ++e) ghosty = ghosty || ((full & (1u << e)) && (pe[e].pad & BK_MASK_GHOST));
          if (ghosty) continue;
          for (int e = 0; e < BK_MASK_L && ok; ++e) {
            if (!(full & (1u << e))) continue;
            const long long off = pe[e].off;
            int at = 0;
            while (at < nu && uni[at] < off) ++at;
            if (at < nu && uni[at] == off) continue;
            if (nu >= BK_MASK_L) {
              ok = false;
              break;
            }
            for (int q = nu; q > at; --q) uni[q] = uni[q - 1];
            uni[at] = off;
            ++nu;
          }
        }
        int np = 0;
        unsigned int oddmask = 0u;
        for (int q = 0; ok && q < nu; ++q) {
          if (uni[q] & 1) {
            oddmask |= 1u << q;
            ctb->offb[q] = 8 * (uni[q] - 1);
          } else {
            ctb->offb[q] = 8 * uni[q];
          }
        }
        for (int slot = 0; ok && slot < BK_MASK_HT; ++slot) {
          if (!hk[slot]) continue;
          const bk_pair_entry* pe = tab + (size_t)slot * BK_MASK_L;
          const unsigned int full = (unsigned int)(pe[0].pad >> BK_MASK_FULL_SHIFT) & 0x1ffu;
          bool ghosty = false;
          for (int e = 0; e < BK_MASK_L; ++e) ghosty = ghosty || ((full & (1u << e)) && (pe[e].pad & BK_MASK_GHOST));
          if (ghosty) continue;  // (s2d stays 0: steps with such chunks are marked mixed below and never use it)
          if (np >= BK_MASK_CP) {
            ok = false;
            break;
          }
          for (int e = 0; e < BK_MASK_L; ++e) {
            if (!(full & (1u << e))) continue;
            int at = 0;
            while (at < nu && uni[at] != (long long)pe[e].off) ++at;
            // ONE value per offset and pattern: a chunk whose rows carry different coefficients on the same diagonal
            // (variable-coefficient operators, e.g. the LDC pressure matrix) has two pairs with one offset -> kernel 6
            if (um.fullu[np] & (1u << at)) ok = false;
            memcpy(&ctb->val[np][at], &pe[e].val, 8);
            um.pos[np][e] = (unsigned char)at;
            um.fullu[np] |= 1u << at;
          }
          s2d[slot] = (unsigned char)np;
          ++np;
        }
        const long long ngroups8 = ((A->n + 255) / 256 + 7) / 8;
        const long long nsteps = ngroups8 * 32;
        int* dcount = (int*)(h->counters + 8);
        if (ok && nu >= 1 && bk_pool_alloc((void**)&d_s2d, BK_MASK_HT, s) == cudaSuccess &&
            bk_pool_alloc((void**)&A->musum, sizeof(unsigned short) * (size_t)nsteps, s) == cudaSuccess &&
            bk_pool_alloc((void**)&A->mumasks, (size_t)nblk8 * 32, s) == cudaSuccess) {
          cudaMemcpyAsync(d_s2d, s2d, BK_MASK_HT, cudaMemcpyHostToDevice, s);
          cudaMemsetAsync(A->mumasks, 0, (size_t)nblk8 * 32, s);
          cudaMemsetAsync(dcount, 0, 2 * sizeof(int), s);
          long long wantw = (nsteps * 32 + 255) / 256;
          int gg = (int)(wantw < (long long)h->num_sms * 8 ? wantw : (long long)h->num_sms * 8);
          if (gg < 1) gg = 1;
          // union position of offset 0 when its neighbours are -1 and +1 (the structures kernel 7 runs), else -1
          const int kc = (nu >= 3 && uni[nu / 2] == 0 && uni[nu / 2 - 1] == -1 && uni[nu / 2 + 1] == 1) ? nu / 2 : -1;
          bk_mask_usum_kernel<<<gg, 256, 0, s>>>(A->mmasks, A->mpids, d_s2d, um, A->n, nsteps, uni[0], uni[nu - 1], kc,
                                                 A->mumasks, A->musum, dcount);
          int cnt[2] = {0, 0};
          cudaMemcpyAsync(cnt, dcount, 2 * sizeof(int), cudaMemcpyDeviceToHost, s);
          if (cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
            ok = false;
          } else {
            A->mu_len = nu;
            A->mu_odd = (int)oddmask;
            A->mu_center = (nu >= 3 && uni[nu / 2] == 0 && uni[nu / 2 - 1] == -1 && uni[nu / 2 + 1] == 1) ? 1 : 0;
            // matrix-side bytes of kernel 7: a 2-byte summary per 64 rows, mask bytes of the steps that read them
            // (kernel 6's share for the mixed steps), the parameter block
            A->mu_bytes = nsteps * 2 + (int64_t)cnt[0] * 64 + (int64_t)cnt[1] * (64 + 8) + (int64_t)sizeof(bk_mask_utab);
          }
        } else {
          ok = false;
          cudaGetLastError();
        }
        if (!ok) {
          if (A->musum) bk_pool_free(A->musum);
          if (A->mumasks) bk_pool_free(A->mumasks);
          A->musum = nullptr;
          A->mumasks = nullptr;
          A->mu_len = 0;
        }
        if (d_s2d) bk_pool_free(d_s2d);
        free(s2d);
      }
    } else {
      cudaGetLastError();
    }
    free(tab);
    free(hk);
  }
  if (A->n_cols > A->n) {  // row partition: compact list of the chunks that gather from the ghost vector
    unsigned int* flags = nullptr;
    if (bk_pool_alloc((void**)&flags, sizeof(unsigned int) * (size_t)(nchunks + 1), s) != cudaSuccess) {
      cudaGetLastError();
      drop();
      return done(BK_OK);
    }
    bk_mask_flag_kernel<<<grid, 256, 0, s>>>(A->mpids, nchunks, flags);
    int rc = bk_exclusive_scan_u32(flags, nchunks + 1, s);
    unsigned int total = 0;
    if (rc == BK_OK) {
      cudaMemcpyAsync(&total, flags + nchunks, sizeof(unsigned int), cudaMemcpyDeviceToHost, s);
      if (cudaStreamSynchronize(s) != cudaSuccess) rc = bk_fail(BK_ERR_CUDA, "csr registration (deferred chunks)");
    }
    if (rc == BK_OK && total > 0) {
      if (bk_pool_alloc((void**)&A->mdeferred, sizeof(int) * (size_t)total, s) != cudaSuccess) {
        cudaGetLastError();
        rc = bk_fail(BK_ERR_ALLOC, "csr registration (deferred chunks): allocation failed");
      } else {
        bk_mask_compact_kernel<<<grid, 256, 0, s>>>(A->mpids, nchunks, flags, A->mdeferred);
        if (cudaStreamSynchronize(s) != cudaSuccess) rc = bk_fail(BK_ERR_CUDA, "csr registration (deferred chunks)");
      }
    }
    bk_pool_free(flags);
    if (rc != BK_OK) {
      drop();
      return done(rc);
    }
    A->n_mdeferred = (int)total;
  }
  A->kernel = 6;
  A->bytes_stream = nchunks * 32 + nchunks * 4 + (int64_t)A->mask_patterns * BK_MASK_L * (int64_t)sizeof(bk_pair_entry);
  return done(BK_OK);
}

// Decide whether the TMA row-stream kernel (bk_spmv_tma.cuh) can serve this matrix, size its pipeline and
// build the 4-entry tail buffers.  Falls back silently to kernel 0 when a requirement is not met.
static int bk_csr_plan_tma(bk_handle* h, bk_csr* A, cudaStream_t s) {
  if (A->kernel != 0 || !h->use_tma || A->n == 0 || A->nnz == 0) return BK_OK;
  if (!bk_aligned16(A->val) || !bk_aligned16(A->col)) return BK_OK;
  const long long nblk = (A->n + 255) / 256;
  int* dstat = (int*)(h->counters + 8);
  int span = 0;
  cudaMemsetAsync(dstat, 0, sizeof(int), s);
  bk_block_span_kernel<<<h->num_sms * 4, 256, 0, s>>>(A->rowptr, A->n, nblk, 256, 4, dstat);
  cudaMemcpyAsync(&span, dstat, sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (TMA plan): %s", cudaGetErrorString(e));
  const int cap = (span + 31) & ~31;
  const size_t entry = bk_dtype_size(A->dtype) + 4;
  const size_t budget = 110 * 1024;  // per CTA with two CTAs per SM (the launch picks CTAs/SM and depth)
  int stages = (int)(budget / ((size_t)cap * entry));
  if (stages > 8) stages = 8;
  if (cap <= 0 || stages < 2) return BK_OK;  // blocks too wide for shared memory: keep kernel 0
  const int tail = (int)(A->nnz & 3);
  if (tail) {
    const size_t vs = bk_dtype_size(A->dtype);
    if (bk_pool_alloc(&A->tail_val, 4 * vs, s) != cudaSuccess || bk_pool_alloc((void**)&A->tail_col, 16, s) != cudaSuccess) {
      cudaGetLastError();
      return bk_fail(BK_ERR_ALLOC, "csr registration: tail buffer allocation failed");
    }
    const int64_t base = A->nnz & ~(int64_t)3;
    cudaMemsetAsync(A->tail_val, 0, 4 * vs, s);
    cudaMemsetAsync(A->tail_col, 0, 16, s);
    cudaMemcpyAsync(A->tail_val, (const char*)A->val + base * vs, tail * vs, cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(A->tail_col, A->col + base, tail * sizeof(int), cudaMemcpyDeviceToDevice, s);
    e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration (tail): %s", cudaGetErrorString(e));
  }
  A->tma_cap = cap;
  A->tma_stages = stages;
  A->kernel = 2;
  BK_TRY(bk_csr_plan_pairs(h, A, s));
  return bk_csr_plan_compress(h, A, s);
}

// statistics + validation + kernel plan (one sync at registration time; never on the per-iteration path)
int bk_csr_finish_plan(bk_handle* h, bk_csr* A, cudaStream_t s) {
  const int64_t n = A->n, nnz = A->nnz;
  if (A->n_cols < n) A->n_cols = n;
  int* dstat = (int*)(h->counters + 8);
  int hstat[2] = {0, 0};
  int ends[2] = {0, 0};
  cudaMemsetAsync(dstat, 0, 2 * sizeof(int), s);
  if (n > 0) bk_csr_stats_kernel<<<h->num_sms * 8, 256, 0, s>>>(A->rowptr, A->col, n, A->n_cols, nnz, dstat);
  cudaMemcpyAsync(hstat, dstat, 2 * sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(&ends[0], A->rowptr, sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(&ends[1], A->rowptr + n, sizeof(int), cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return bk_fail(BK_ERR_CUDA, "csr registration: %s", cudaGetErrorString(e));
  if (ends[0] != 0 || ends[1] != (int)nnz || hstat[1] != 0)
    return bk_fail(BK_ERR_ARG, "malformed CSR (rowptr[0]=%d, rowptr[n]=%d, nnz=%lld, bad=%d)", ends[0], ends[1],
                   (long long)nnz, hstat[1]);
  A->max_row_nnz = hstat[0];
  bk_csr_plan(h, A);
  A->bytes_stream = nnz * (int64_t)(bk_dtype_size(A->dtype) + 4) + (n + 1) * 4;
  BK_TRY(bk_csr_plan_split(h, A, s));
  if (A->split) {  // the virtual-row view carries the kernel plan
    A->bytes_stream = A->split->bytes_stream + (n + 1) * 4 + 2 * A->split->n * (int64_t)bk_dtype_size(A->dtype);
    return BK_OK;
  }
  if (A->n_cols != A->n) {  // extended [local | ghost] matrix of a row partition: the row-bitmask plan or nothing
    if (A->kernel == 0) BK_TRY(bk_csr_plan_mask(h, A, A->reg_ghost_gid, A->reg_row_begin, s));
    return BK_OK;
  }
  if (A->kernel == 0) BK_TRY(bk_csr_plan_mask(h, A, nullptr, 0, s));
  if (A->kernel == 6) return BK_OK;
  return bk_csr_plan_tma(h, A, s);
}

extern "C" int bk_csr_create(bk_handle* h, int64_t n, int64_t nnz, const void* rowptr, const void* col,
                             int idx_bits, const void* val, int dtype, int copy, void* stream, bk_csr** out) {
  if (!h || !out) return bk_fail(BK_ERR_ARG, "bk_csr_create: null handle/out");
  *out = nullptr;
  if (n < 0 || nnz < 0) return bk_fail(BK_ERR_ARG, "bk_csr_create: negative size");
  if (n >= 2147483647LL || nnz >= 2147483647LL)
    return bk_fail(BK_ERR_UNSUPPORTED, "bk_csr_create: n and nnz must be < 2^31 (int32 indices), got n=%lld nnz=%lld",
                   (long long)n, (long long)nnz);
  if (idx_bits != 32 && idx_bits != 64) return bk_fail(BK_ERR_ARG, "bk_csr_create: idx_bits must be 32 or 64");
  if (dtype != BK_F64 && dtype != BK_F32) return bk_fail(BK_ERR_ARG, "bk_csr_create: dtype must be BK_F64 or BK_F32");
  if (!rowptr || (nnz > 0 && (!col || !val))) return bk_fail(BK_ERR_ARG, "bk_csr_create: null array");
  BK_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  bk_csr* A = (bk_csr*)calloc(1, sizeof(bk_csr));
  if (!A) return bk_fail(BK_ERR_ALLOC, "bk_csr_create: host allocation failed");
  A->h = h;
  A->n = n;
  A->nnz = nnz;
  A->dtype = dtype;
  A->uid = h->next_uid++;
  const size_t vs = bk_dtype_size(dtype);
  auto fail = [&](int code) {
    bk_csr_destroy(A);
    return code;
  };
  if (idx_bits == 64) {
    if (bk_pool_alloc(&A->own_rowptr, sizeof(int) * (size_t)(n + 1), s) != cudaSuccess ||
        bk_pool_alloc(&A->own_col, sizeof(int) * (size_t)(nnz > 0 ? nnz : 1), s) != cudaSuccess) {
      cudaGetLastError();
      return fail(bk_fail(BK_ERR_ALLOC, "bk_csr_create: int32 index copy allocation failed"));
    }
    bk_cvt_i64_i32_kernel<<<h->num_sms * 8, 256, 0, s>>>((const long long*)rowptr, (int*)A->own_rowptr, n + 1);
    if (nnz > 0) bk_cvt_i64_i32_kernel<<<h->num_sms * 8, 256, 0, s>>>((const long long*)col, (int*)A->own_col, nnz);
    A->rowptr = (const int*)A->own_rowptr;
    A->col = (const int*)A->own_col;
  } else if (copy) {
    if (bk_pool_alloc(&A->own_rowptr, sizeof(int) * (size_t)(n + 1), s) != cudaSuccess ||
        bk_pool_alloc(&A->own_col, sizeof(int) * (size_t)(nnz > 0 ? nnz : 1), s) != cudaSuccess) {
      cudaGetLastError();
      return fail(bk_fail(BK_ERR_ALLOC, "bk_csr_create: index copy allocation failed"));
    }
    cudaMemcpyAsync(A->own_rowptr, rowptr, sizeof(int) * (size_t)(n + 1), cudaMemcpyDeviceToDevice, s);
    if (nnz > 0) cudaMemcpyAsync(A->own_col, col, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s);
    A->rowptr = (const int*)A->own_rowptr;
    A->col = (const int*)A->own_col;
  } else {
    A->rowptr = (const int*)rowptr;
    A->col = (const int*)col;
  }
  if (copy) {
    if (bk_pool_alloc(&A->own_val, vs * (size_t)(nnz > 0 ? nnz : 1), s) != cudaSuccess) {
      cudaGetLastError();
      return fail(bk_fail(BK_ERR_ALLOC, "bk_csr_create: value copy allocation failed"));
    }
    if (nnz > 0) cudaMemcpyAsync(A->own_val, val, vs * (size_t)nnz, cudaMemcpyDeviceToDevice, s);
    A->val = A->own_val;
  } else {
    A->val = val;
  }
  {
    int prc = bk_csr_finish_plan(h, A, s);
    if (prc != BK_OK) return fail(prc);
  }
  *out = A;
  return BK_OK;
}

extern "C" int bk_csr_destroy(bk_csr* A) {
  if (!A) return BK_OK;
  if (A->h) {
    cudaSetDevice(A->h->device);
    bk_graphs_invalidate(A->h);
    cudaDeviceSynchronize();  // nothing may still be reading the arrays: the frees below are stream-ordered
  }
  if (A->transpose) bk_csr_destroy(A->transpose);
  if (A->sgs) bk_sgs_free(A->sgs);
  if (A->split) bk_csr_destroy(A->split);
  if (A->vstart) bk_pool_free(A->vstart);
  if (A->yv) bk_pool_free(A->yv);
  if (A->own_rowptr) bk_pool_free(A->own_rowptr);
  if (A->own_col) bk_pool_free(A->own_col);
  if (A->own_val) bk_pool_free(A->own_val);
  if (A->tail_val) bk_pool_free(A->tail_val);
  if (A->tail_col) bk_pool_free(A->tail_col);
  if (A->codes) bk_pool_free(A->codes);
  if (A->dict) bk_pool_free(A->dict);
  if (A->tail_val16) bk_pool_free(A->tail_val16);
  if (A->tail_code16) bk_pool_free(A->tail_code16);
  if (A->pcodes) bk_pool_free(A->pcodes);
  if (A->pdict) bk_pool_free(A->pdict);
  if (A->pbptr) bk_pool_free(A->pbptr);
  if (A->mmasks) bk_pool_free(A->mmasks);
  if (A->mpids) bk_pool_free(A->mpids);
  if (A->mptab) bk_pool_free(A->mptab);
  if (A->mdeferred) bk_pool_free(A->mdeferred);
  if (A->musum) bk_pool_free(A->musum);
  if (A->mumasks) bk_pool_free(A->mumasks);
  free(A);
  return BK_OK;
}

extern "C" int bk_csr_get_info(const bk_csr* A, bk_csr_info* out) {
  if (!A || !out) return bk_fail(BK_ERR_ARG, "bk_csr_get_info: null argument");
  out->n = A->n;
  out->nnz = A->nnz;
  out->dtype = A->dtype;
  out->kernel = A->kernel;
  out->lanes_per_row = A->lanes_per_row;
  out->max_row_nnz = A->max_row_nnz;
  out->mean_row_nnz = A->mean_row_nnz;
  out->bytes_matrix = A->nnz * (int64_t)(bk_dtype_size(A->dtype) + 4) + (A->n + 1) * 4;
  out->bytes_stream = A->bytes_stream;
  if (A->kernel == 6 && bk_mask2_usable(A->h, A)) {  // the stencil fast path serves this matrix (operands permitting)
    out->kernel = 7;
    out->bytes_stream = A->mu_bytes;
  }
  return BK_OK;
}

extern "C" int bk_csr_arrays(const bk_csr* A, const void** rowptr, const void** col, const void** val) {
  if (!A) return bk_fail(BK_ERR_ARG, "bk_csr_arrays: null matrix");
  if (rowptr) *rowptr = A->rowptr;
  if (col) *col = A->col;
  if (val) *val = A->val;
  return BK_OK;
}

// ------------------------------------------------------------------------------------------
// building blocks
// ------------------------------------------------------------------------------------------
struct bk_epi_store {
  double* out;
  __device__ __forceinline__ void operator()(const double* s) const { out[0] = s[0]; }
};

extern "C" int bk_spmv(bk_handle* h, const bk_csr* A, const void* x, void* y, void* stream) {
  if (!h || !A || !x || !y) return bk_fail(BK_ERR_ARG, "bk_spmv: null argument");
  if (x == y) return bk_fail(BK_ERR_ARG, "bk_spmv: x and y must not alias");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) return BK_OK;
  bk_spmv_args a = bk_spmv_base(A, h->st);
  a.x = x;
  a.y = y;
  return bk_launch_spmv<0, 0, 0>(h, A, a, bk_slot(h, 0), bk_epi_none(), (cudaStream_t)stream);
}

extern "C" int bk_spmv_dot(bk_handle* h, const bk_csr* A, const void* x, void* y, const void* w, double* dot_out,
                           void* stream) {
  if (!h || !A || !x || !y || !w || !dot_out) return bk_fail(BK_ERR_ARG, "bk_spmv_dot: null argument");
  if (x == y) return bk_fail(BK_ERR_ARG, "bk_spmv_dot: x and y must not alias");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0) {
    BK_CUDA(cudaMemsetAsync(dot_out, 0, sizeof(double), (cudaStream_t)stream));
    return BK_OK;
  }
  bk_spmv_args a = bk_spmv_base(A, h->st);
  a.x = x;
  a.y = y;
  a.w = w;
  bk_epi_store epi;
  epi.out = dot_out;
  return bk_launch_spmv<0, 1, 0>(h, A, a, bk_slot(h, 0), epi, (cudaStream_t)stream);
}

template <typename T>
static int bk_dot_t(bk_handle* h, int64_t n, const void* x, const void* y, double* out, int sqrt_out, cudaStream_t s) {
  bk_op_dot<T> op;
  op.x = (const T*)x;
  op.y = (const T*)y;
  op.out = out;
  op.sqrt_out = sqrt_out;
  return bk_launch_ew<T>(h, op, n, bk_aligned16(x) && bk_aligned16(y), bk_slot(h, 0), s);
}

extern "C" int bk_dot(bk_handle* h, int64_t n, int dtype, const void* x, const void* y, double* out, void* stream) {
  if (!h || !out || (n > 0 && (!x || !y))) return bk_fail(BK_ERR_ARG, "bk_dot: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (dtype == BK_F64) return bk_dot_t<double>(h, n, x, y, out, 0, (cudaStream_t)stream);
  if (dtype == BK_F32) return bk_dot_t<float>(h, n, x, y, out, 0, (cudaStream_t)stream);
  return bk_fail(BK_ERR_ARG, "bk_dot: bad dtype %d", dtype);
}

extern "C" int bk_nrm2(bk_handle* h, int64_t n, int dtype, const void* x, double* out, void* stream) {
  if (!h || !out || (n > 0 && !x)) return bk_fail(BK_ERR_ARG, "bk_nrm2: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (dtype == BK_F64) return bk_dot_t<double>(h, n, x, x, out, 1, (cudaStream_t)stream);
  if (dtype == BK_F32) return bk_dot_t<float>(h, n, x, x, out, 1, (cudaStream_t)stream);
  return bk_fail(BK_ERR_ARG, "bk_nrm2: bad dtype %d", dtype);
}

template <typename T>
static int bk_axpby_t(bk_handle* h, int64_t n, double a, const void* x, double b, const void* y, void* z,
                      cudaStream_t s) {
  bk_op_axpby<T> op;
  op.x = (const T*)x;
  op.y = (const T*)y;
  op.z = (T*)z;
  op.ca = (T)a;
  op.cb = (T)b;
  return bk_launch_ew<T>(h, op, n, bk_aligned16(x) && bk_aligned16(y) && bk_aligned16(z), bk_slot(h, 0), s);
}

extern "C" int bk_axpby(bk_handle* h, int64_t n, int dtype, double a, const void* x, double b, const void* y, void* z,
                        void* stream) {
  if (!h || (n > 0 && (!x || !y || !z))) return bk_fail(BK_ERR_ARG, "bk_axpby: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (n == 0) return BK_OK;
  if (dtype == BK_F64) return bk_axpby_t<double>(h, n, a, x, b, y, z, (cudaStream_t)stream);
  if (dtype == BK_F32) return bk_axpby_t<float>(h, n, a, x, b, y, z, (cudaStream_t)stream);
  return bk_fail(BK_ERR_ARG, "bk_axpby: bad dtype %d", dtype);
}

template <typename T>
static int bk_axpby_dev_t(bk_handle* h, int64_t n, double sa, const double* pa, const void* x, double sb,
                          const double* pb, const void* y, void* z, cudaStream_t s) {
  bk_op_axpby_dev<T> op;
  op.x = (const T*)x;
  op.y = (const T*)y;
  op.z = (T*)z;
  op.pa = pa;
  op.pb = pb;
  op.sa = sa;
  op.sb = sb;
  return bk_launch_ew<T>(h, op, n, bk_aligned16(x) && bk_aligned16(y) && bk_aligned16(z), bk_slot(h, 0), s);
}

extern "C" int bk_axpby_dev(bk_handle* h, int64_t n, int dtype, double sa, const double* a_dev, const void* x,
                            double sb, const double* b_dev, const void* y, void* z, void* stream) {
  if (!h || (n > 0 && (!x || !y || !z))) return bk_fail(BK_ERR_ARG, "bk_axpby_dev: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (n == 0) return BK_OK;
  if (dtype == BK_F64) return bk_axpby_dev_t<double>(h, n, sa, a_dev, x, sb, b_dev, y, z, (cudaStream_t)stream);
  if (dtype == BK_F32) return bk_axpby_dev_t<float>(h, n, sa, a_dev, x, sb, b_dev, y, z, (cudaStream_t)stream);
  return bk_fail(BK_ERR_ARG, "bk_axpby_dev: bad dtype %d", dtype);
}

template <typename T>
static int bk_div_t(bk_handle* h, int64_t n, const void* x, double d, void* z, cudaStream_t s) {
  bk_op_div<T> op;
  op.x = (const T*)x;
  op.z = (T*)z;
  op.d = (T)d;
  return bk_launch_ew<T>(h, op, n, bk_aligned16(x) && bk_aligned16(z), bk_slot(h, 0), s);
}

extern "C" int bk_div_scalar(bk_handle* h, int64_t n, int dtype, const void* x, double d, void* z, void* stream) {
  if (!h || (n > 0 && (!x || !z))) return bk_fail(BK_ERR_ARG, "bk_div_scalar: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (n == 0) return BK_OK;
  if (dtype == BK_F64) return bk_div_t<double>(h, n, x, d, z, (cudaStream_t)stream);
  if (dtype == BK_F32) return bk_div_t<float>(h, n, x, d, z, (cudaStream_t)stream);
  return bk_fail(BK_ERR_ARG, "bk_div_scalar: bad dtype %d", dtype);
}

// ---- block-Jacobi application (SURVEY 8f-1): z = blockdiag(inv) r, inv = [nblocks][bs][bs] row-major ---------------
template <typename T>
__global__ void bk_block_apply_kernel(const T* __restrict__ inv, const T* __restrict__ r, T* __restrict__ z,
                                      long long n, int bs) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += stride) {
    const long long blk = row / bs;
    const int lr = (int)(row - blk * bs);
    const T* __restrict__ m = inv + ((size_t)blk * bs + lr) * bs;
    const long long c0 = blk * bs;
    T sum = T(0);
    for (int c = 0; c < bs; ++c) {
      const long long col = c0 + c;
      if (col < n) sum = fma(m[c], r[col], sum);
    }
    z[row] = sum;
  }
}

extern "C" int bk_block_apply(bk_handle* h, int64_t n, int bs, int dtype, const void* inv, const void* r, void* z,
                              void* stream) {
  if (!h || (n > 0 && (!inv || !r || !z))) return bk_fail(BK_ERR_ARG, "bk_block_apply: null argument");
  if (bs < 1 || bs > 64) return bk_fail(BK_ERR_ARG, "bk_block_apply: block size must be in [1, 64]");
  if (r == z) return bk_fail(BK_ERR_ARG, "bk_block_apply: r and z must not alias");
  BK_CUDA(cudaSetDevice(h->device));
  if (n == 0) return BK_OK;
  const int g = bk_grid_rows(h->num_sms * 8, n, 256);
  if (dtype == BK_F64)
    bk_block_apply_kernel<double><<<g, 256, 0, (cudaStream_t)stream>>>((const double*)inv, (const double*)r, (double*)z, n, bs);
  else if (dtype == BK_F32)
    bk_block_apply_kernel<float><<<g, 256, 0, (cudaStream_t)stream>>>((const float*)inv, (const float*)r, (float*)z, n, bs);
  else
    return bk_fail(BK_ERR_ARG, "bk_block_apply: bad dtype %d", dtype);
  BK_KERNEL_CHECK();
  return BK_OK;
}

// ---- complex128 building blocks (SURVEY 8f-4; reference :86-127, :1220): vectors are interleaved (re, im) fp64 -------
extern "C" int bk_cdot(bk_handle* h, int64_t n_complex, const void* x, const void* y, double* out2, void* stream) {
  if (!h || !out2 || (n_complex > 0 && (!x || !y))) return bk_fail(BK_ERR_ARG, "bk_cdot: null argument");
  if (!bk_aligned16(x) || !bk_aligned16(y)) return bk_fail(BK_ERR_ARG, "bk_cdot: complex vectors must be 16-byte aligned");
  BK_CUDA(cudaSetDevice(h->device));
  bk_op_cdot op;
  op.x = (const double*)x;
  op.y = (const double*)y;
  op.out = out2;
  return bk_launch_ew<double>(h, op, 2 * n_complex, true, bk_slot(h, 0), (cudaStream_t)stream);
}

extern "C" int bk_caxpby(bk_handle* h, int64_t n_complex, double ar, double ai, const void* x, double br, double bi,
                         const void* y, void* z, void* stream) {
  if (!h || (n_complex > 0 && (!x || !y || !z))) return bk_fail(BK_ERR_ARG, "bk_caxpby: null argument");
  if (!bk_aligned16(x) || !bk_aligned16(y) || !bk_aligned16(z))
    return bk_fail(BK_ERR_ARG, "bk_caxpby: complex vectors must be 16-byte aligned");
  BK_CUDA(cudaSetDevice(h->device));
  if (n_complex == 0) return BK_OK;
  bk_op_caxpby op;
  op.x = (const double*)x;
  op.y = (const double*)y;
  op.z = (double*)z;
  op.ar = ar;
  op.ai = ai;
  op.br = br;
  op.bi = bi;
  return bk_launch_ew<double>(h, op, 2 * n_complex, true, bk_slot(h, 0), (cudaStream_t)stream);
}

// ---- gradient with respect to the stored entries of A (SURVEY §8f-3) -----------------------------------------
// For A x = b and a loss L(x):  dL/dA_ij = -(A^-T dL/dx)_i x_j = -g_i x_j, evaluated on the sparsity pattern only
// (an SDDMM-shaped kernel).  The reference returns no gradient for A (torch_sparse_linalg.py:1248); its Modules B/C
// compute this product with Python row loops (module_b/torch_amgx.py:444-462).  One warp per row.
template <typename T>
__global__ void bk_grad_pattern_kernel(const int* __restrict__ rowptr, const int* __restrict__ col,
                                       const T* __restrict__ g, const T* __restrict__ x, T* __restrict__ out,
                                       long long n) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const T gi = -g[r];
    for (int k = rowptr[r] + lane; k < rowptr[r + 1]; k += 32) out[k] = gi * x[col[k]];
  }
}

extern "C" int bk_csr_grad_pattern(bk_handle* h, const bk_csr* A, const void* g, const void* x, void* out_vals,
                                   void* stream) {
  if (!h || !A || (A->nnz > 0 && (!g || !x || !out_vals))) return bk_fail(BK_ERR_ARG, "bk_csr_grad_pattern: null argument");
  BK_CUDA(cudaSetDevice(h->device));
  if (A->n == 0 || A->nnz == 0) return BK_OK;
  int grid = (int)((A->n * 32 + 255) / 256);
  if (grid > h->num_sms * 8) grid = h->num_sms * 8;
  if (A->dtype == BK_F64)
    bk_grad_pattern_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(A->rowptr, A->col, (const double*)g,
                                                                            (const double*)x, (double*)out_vals, A->n);
  else
    bk_grad_pattern_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(A->rowptr, A->col, (const float*)g,
                                                                           (const float*)x, (float*)out_vals, A->n);
  BK_KERNEL_CHECK();
  return BK_OK;
}

// ---- checksum of a device array (cache validation of borrowed value arrays; see include/bk_krylov.h) ---------------
__global__ void bk_checksum_kernel(const unsigned int* __restrict__ p, long long nwords, unsigned long long* out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  unsigned long long acc = 0ull;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += stride)
    acc += bk_mix64(((unsigned long long)p[i] << 32) ^ (unsigned long long)i ^ 0x9e3779b97f4a7c15ull);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc != 0ull) atomicAdd(out, acc);  // integer sum: order-independent
}

extern "C" int bk_checksum(bk_handle* h, const void* data, int64_t nbytes, void* stream, uint64_t* out_host) {
  if (!h || !out_host || nbytes < 0 || (nbytes > 0 && !data)) return bk_fail(BK_ERR_ARG, "bk_checksum: bad argument");
  if (nbytes % 4 != 0 || (((uintptr_t)data) & 3u) != 0)
    return bk_fail(BK_ERR_ARG, "bk_checksum: data and size must be 4-byte aligned");
  BK_CUDA(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  BK_CUDA(cudaMemsetAsync(h->cksum, 0, sizeof(unsigned long long), s));
  const long long nwords = nbytes / 4;
  if (nwords > 0) {
    long long want = (nwords + 256 * 8 - 1) / (256 * 8);
    int grid = (int)(want < (long long)h->num_sms * 8 ? want : (long long)h->num_sms * 8);
    bk_checksum_kernel<<<grid, 256, 0, s>>>((const unsigned int*)data, nwords, h->cksum);
    BK_KERNEL_CHECK();
  }
  unsigned long long v = 0;
  BK_CUDA(cudaMemcpyAsync(&v, h->cksum, sizeof(v), cudaMemcpyDeviceToHost, s));
  BK_CUDA(cudaStreamSynchronize(s));
  *out_host = (uint64_t)(v ^ (unsigned long long)nbytes);
  return BK_OK;
}
