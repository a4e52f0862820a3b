"""The general CSR SpMV plans — kernel 0 (LDG row stream), 1 (sub-warp vector), 2 (TMA row stream), 3 (TMA row
stream over 8-bit column codes), 4 (virtual-row split + ordered reduction) and 5 (pair-coded SELL stream) — at their
selection and tiling boundaries.

Registration picks the plan from the matrix content alone, so `predict_csr_plan` restates the rules of `bk_csr_plan*`
(csrc/bk_core.cu) on the CPU and the GPU tests hold the library to it.  Seeded generators place matrices on each
boundary and one step past it: the tail buffers of kernels 2 / 3 at every residue of nnz, 32 vs 33 offsets per block,
the TMA stage width, the stream kernel's shared-memory window, the lanes-per-row steps of kernel 1, the skew limit and
the virtual-row cuts, misaligned borrowed arrays, tiny and 1.5 M-row matrices.  Every SpMV is compared row by row with
an extended-precision reference, bitwise across the launch variants of one plan, and through the solvers' residual
mode and fused p-update.  All inputs are seeded and finite.
"""
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch

from test_stencil_plans import (_csr_numpy, _longdouble, _transpose, check_rows, options, predict_plan, ref_spmv,
                                dot_roundings as mask_dot_roundings)

SPLIT_LEN = 256          # BK_SPLIT_LEN: virtual rows of kernel 4 hold at most this many entries
RPB = 256                # rows per block of kernels 0 / 2 / 3 / 5 and of the dictionaries
SMEM_BUDGET = 110 * 1024  # per-CTA stage budget used by bk_csr_plan_tma / _compress / _pairs
MAX_STAGES = 8
PAIR_HDR, PAIR_DICT, PAIR_ZERO = 128, 32 * 16, 31
NEITHER = "neither"


# --------------------------------------------------------------------------------------------------
# CPU model of plan selection (bk_csr_finish_plan and the bk_csr_plan* functions it calls)
# --------------------------------------------------------------------------------------------------
def _block_span(crow, n, al):
    """bk_block_span_kernel: widest al-aligned [s & ~(al-1), (e + al-1) & ~(al-1)) span of any 256-row block."""
    if n == 0:
        return 0
    r0 = np.arange(0, n, RPB)
    s = crow[r0]
    e = crow[np.minimum(r0 + RPB, n)]
    return int((((e + al - 1) & ~(al - 1)) - (s & ~(al - 1))).max())


def _distinct_per_block(rows, keys):
    """Largest number of distinct keys (an int64 array, or a tuple of them) over the 256-row blocks."""
    if rows.size == 0:
        return 0
    keys = keys if isinstance(keys, tuple) else (keys,)
    blk = rows // RPB
    order = np.lexsort(keys[::-1] + (blk,))
    cols = [blk[order]] + [k[order] for k in keys]
    new = np.ones(rows.size, dtype=bool)
    new[1:] = np.any([c[1:] != c[:-1] for c in cols], axis=0)
    return int(np.bincount(cols[0][new]).max())


def tma_stages(cap, vs):
    """bk_csr_plan_tma: stages of cap entries of (value + int32 column) within the per-CTA budget, at most 8."""
    return min(MAX_STAGES, SMEM_BUDGET // (cap * (vs + 4))) if cap > 0 else 0


def compress_fits(cap16, vs):
    """bk_csr_plan_compress: two stages of cap16 (value + 1-byte code) entries plus the 128-byte dictionary fit."""
    return cap16 > 0 and 2 * (cap16 * (vs + 1) + 128) <= SMEM_BUDGET


def pair_block_bytes(lens, n):
    """bk_pair_block_bytes_kernel: per 256-row block, the 128-byte header plus, per 32-row chunk, 128 bytes per 4
    entries of the chunk's longest row."""
    nblk = -(-n // RPB)
    L = np.zeros(nblk * RPB, dtype=np.int64)
    L[:n] = lens
    chunk_max = L.reshape(nblk, 8, 32).max(axis=2)
    return 128 * (PAIR_HDR // 128 + ((chunk_max + 3) >> 2).sum(axis=1))


def _row_stream_plan(crow, col, val, n, vs, is_view, use_tma, use_compress, aligned):
    """bk_csr_plan_tma -> bk_csr_plan_pairs -> bk_csr_plan_compress for a matrix already on kernel 0 (mask plan
    declined).  Returns (kernel, extra)."""
    nnz = col.size
    if not use_tma or n == 0 or nnz == 0 or not aligned:
        return 0, {}
    cap = (_block_span(crow, n, 4) + 31) & ~31
    stages = tma_stages(cap, vs)
    if stages < 2:
        return 0, {}
    extra = dict(tma_cap=cap, tma_stages=stages)
    lens = np.diff(crow)
    rows = np.repeat(np.arange(n, dtype=np.int64), lens)
    off = col - rows
    if use_compress >= 2 and not is_view:                     # bk_csr_plan_pairs
        blk_bytes = pair_block_bytes(lens, n)
        total = int(blk_bytes.sum())
        nblk = blk_bytes.size
        if 0 < total <= 1.5 * nnz + 1152.0 * nblk and total < 0x7fffff00:
            vb = (val.view(np.uint64) if vs == 8 else val.view(np.uint32)).astype(np.int64)
            pcap = (int(blk_bytes.max()) + 127) & ~127
            if _distinct_per_block(rows, (off, vb)) <= PAIR_ZERO and 2 * (pcap + PAIR_DICT) <= SMEM_BUDGET:
                return 5, dict(extra, pair_cap=pcap)
    if use_compress >= 1:                                     # bk_csr_plan_compress
        cap16 = (_block_span(crow, n, 16) + 31) & ~31
        if _distinct_per_block(rows, off) <= 32 and compress_fits(cap16, vs):
            return 3, dict(extra, cmp_cap=cap16)
    return 2, extra


def virtual_rows(crow):
    """bk_vrow_count_kernel / bk_vrow_fill_kernel: every row longer than 256 entries cut into rows of 256 (the last
    shorter); every other row, empty ones included, keeps one virtual row.  Returns (vrowptr, vstart)."""
    lens = np.diff(crow)
    cnt = np.where(lens <= SPLIT_LEN, 1, -(-lens // SPLIT_LEN))
    vstart = np.zeros(lens.size + 1, dtype=np.int64)
    vstart[1:] = np.cumsum(cnt)
    real = np.repeat(np.arange(lens.size), cnt)
    k = np.arange(int(vstart[-1])) - vstart[:-1][real]
    vrowptr = np.append(crow[:-1][real] + k * SPLIT_LEN, crow[-1])
    return vrowptr, vstart


def predict_csr_plan(A, dtype=torch.float64, use_tma=1, use_compress=3, use_split=1, aligned=True):
    """The plan that registering the CPU CSR matrix `A` as `dtype` under these handle options selects (bk_csr_finish_plan):

    * bk_csr_plan: mean = nnz / n (double), skew_limit = 64 max(mean, 8); kernel 0 if mean <= 32 and max_row <=
      skew_limit, else 1; stream window cap 256 if mean <= 8 else 1024; lanes per row 8 / 16 / 32 for mean <= 64 / <=
      128 / above.
    * bk_csr_plan_split: kernel 4 if use_split, mean <= 32 and max_row > skew_limit; the virtual-row view (rows cut at
      256 entries) is planned by bk_csr_finish_plan again, as a view (no mask, no pair plan).
    * bk_csr_plan_mask (use_compress >= 3, max_row <= 8): test_stencil_plans.predict_plan (kernel 6 / 7).
    * bk_csr_plan_tma: use_tma, n > 0, nnz > 0, val and col 16-byte aligned; cap = roundup32(widest 4-aligned block
      span), stages = min(8, 112640 // (cap (sizeof T + 4))); kernel 2 if stages >= 2.
    * bk_csr_plan_pairs (use_compress >= 2, not a view): <= 31 distinct (col - row, value bits) per block, pair-stream
      bytes <= 1.5 nnz + 1152 nblk, two stages of roundup128(widest block) + 512 bytes fit: kernel 5.
    * bk_csr_plan_compress (use_compress >= 1, still kernel 2): <= 32 distinct col - row per block and two stages of
      roundup32(widest 16-aligned span) (sizeof T + 1) + 128 bytes fit: kernel 3.

    `aligned`: val and (int32) col as borrowed are 16-byte aligned.  Returns a dict with kernel, lanes_per_row,
    max_row_nnz, mean_row_nnz and the stage sizes of kernels 2 / 3 / 5 (for kernel 4: of the view, under "view")."""
    crow, col, val = _csr_numpy(A, dtype)
    n = A.shape[0]
    nnz = col.size
    vs = 8 if dtype == torch.float64 else 4
    lens = np.diff(crow)
    max_row = int(lens.max()) if n else 0
    mean = nnz / n if n else 0.0
    skew_limit = 64.0 * max(mean, 8.0)
    out = dict(kernel=0 if (mean <= 32.0 and max_row <= skew_limit) else 1,
               lanes_per_row=8 if mean <= 64.0 else (16 if mean <= 128.0 else 32),
               max_row_nnz=max_row, mean_row_nnz=mean, cap=256 if mean <= 8.0 else 1024)
    if use_split and n > 0 and mean <= 32.0 and max_row > skew_limit:
        vrowptr, _ = virtual_rows(crow)
        nv = vrowptr.size - 1
        vmean = nnz / nv
        vkernel = 0 if (vmean <= 32.0 and int(np.diff(vrowptr).max()) <= 64.0 * max(vmean, 8.0)) else 1
        extra = {}
        if vkernel == 0:
            vkernel, extra = _row_stream_plan(vrowptr, col, val, nv, vs, True, use_tma, use_compress, aligned)
        out.update(kernel=4, view=dict(extra, kernel=vkernel, n=nv, cap=256 if vmean <= 8.0 else 1024))
        return out
    if out["kernel"] == 1:
        return out
    if use_compress >= 3 and max_row <= 8:
        k = predict_plan(A, dtype)[0]
        if k != NEITHER:
            out["kernel"] = k
            return out
    k, extra = _row_stream_plan(crow, col, val, n, vs, False, use_tma, use_compress, aligned)
    out.update(extra, kernel=k)
    return out


# --------------------------------------------------------------------------------------------------
# Generators (all seeded, CPU, fp64 values, int64 indices)
# --------------------------------------------------------------------------------------------------
def _csr(lens, col, val, n):
    crow = np.zeros(len(lens) + 1, dtype=np.int64)
    crow[1:] = np.cumsum(lens)
    return torch.sparse_csr_tensor(torch.from_numpy(crow), torch.from_numpy(np.asarray(col, dtype=np.int64)),
                                   torch.from_numpy(np.asarray(val, dtype=np.float64)), size=(n, n))


def _exact_total(lens, lo, hi, total, rng):
    """Move row lengths within [lo, hi] by one at random rows until they add up to `total`."""
    lens = lens.copy()
    while (d := total - int(lens.sum())) != 0:
        can = np.nonzero(lens < hi if d > 0 else lens > lo)[0]
        pick = rng.choice(can, size=min(abs(d), can.size), replace=False)
        lens[pick] += 1 if d > 0 else -1
    return lens


def _trim(lens, mod, r):
    """Drop entries from the end of the matrix (the last row first) until nnz % mod == r."""
    lens = lens.copy()
    k = (int(lens.sum()) - r) % mod
    i = lens.size - 1
    while k:
        t = min(k, int(lens[i]))
        lens[i] -= t
        k -= t
        i -= 1
    return lens


def random_matrix(lens, seed, n=None):
    """Rows of the given lengths with distinct ascending columns (a random start plus random positive gaps, wrapped
    into [0, n)) and standard normal values."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, dtype=np.int64)
    n = lens.size if n is None else n
    nnz = int(lens.sum())
    rows = np.repeat(np.arange(lens.size), lens)
    gapmax = np.maximum(1, (n - 1) // np.maximum(lens, 1))[rows]
    gaps = 1 + np.floor(rng.random(nnz) * gapmax).astype(np.int64)
    cs = np.cumsum(gaps)
    before = np.concatenate([[0], cs])[np.concatenate([[0], np.cumsum(lens)])[:-1]]
    col = (rng.integers(0, n, size=lens.size)[rows] + cs - np.repeat(before, lens)) % n
    col = col[np.lexsort((col, rows))]
    return _csr(lens, col, rng.standard_normal(nnz), n)


def banded_matrix(n, row_offsets, seed):
    """Rows whose entries sit at the given (column - row) offsets (a list of sorted arrays, one per row), entries
    outside [0, n) dropped, standard normal values."""
    rng = np.random.default_rng(seed)
    rows = np.concatenate([np.full(len(o), r) for r, o in enumerate(row_offsets)])
    col = rows + np.concatenate(row_offsets)
    keep = (col >= 0) & (col < n)
    rows, col = rows[keep], col[keep]
    return _csr(np.bincount(rows, minlength=n), col, rng.standard_normal(col.size), n)


def tails(r, n=4099, seed=0):
    """Random short rows (0..12 entries, empty ones included), the last rows trimmed so that nnz % 4 == r."""
    rng = np.random.default_rng(100 + seed)
    return random_matrix(_trim(rng.integers(0, 13, n), 4, r), 200 + seed)


_DICT = np.array([-1500, -700, -301, -256, -255, -129, -64, -33, -32, -31, -17, -9, -5, -3, -2, -1,
                  0, 1, 2, 4, 7, 16, 31, 32, 63, 100, 128, 200, 257, 511, 900, 2000])


def dict_offsets(n, seed, extra_block=None):
    """Per row 4..12 of the 32 offsets in _DICT (row r takes _DICT[(r + 3k) % 32], k < length), so every 256-row block
    uses all 32; `extra_block`: one row of that block also takes offset 3, a 33rd."""
    rng = np.random.default_rng(300 + seed)
    L = rng.integers(4, 13, n)
    offs = [np.sort(_DICT[(r + 3 * np.arange(L[r])) % 32]) for r in range(n)]
    if extra_block is not None:
        r = extra_block * RPB + 77
        offs[r] = np.sort(np.append(offs[r], 3))
    return offs


def dict_tail(r, n=4099):
    """32 offsets in every block, random values, the last rows trimmed so that nnz % 16 == r."""
    A = banded_matrix(n, dict_offsets(n, 0), 400)
    crow, col, val = _csr_numpy(A, torch.float64)
    lens = _trim(np.diff(crow), 16, r)
    keep = np.concatenate([np.arange(crow[i], crow[i] + lens[i]) for i in range(n)])
    return _csr(lens, col[keep], val[keep], n)


def tma_width(span_entries, s_mod4=0, n=4096, seed=0):
    """Short rows (0..6 entries) plus block 3 (rows 768..1023) holding `span_entries` entries in rows of 18..28,
    starting at an entry index = s_mod4 (mod 4): its 4-aligned span is span_entries rounded out to multiples of 4."""
    rng = np.random.default_rng(500 + seed)
    lens = rng.integers(0, 7, n)
    q, rem = divmod(span_entries, RPB)
    lens[768:1024] = q
    lens[768:768 + rem] += 1
    lens[767] += (s_mod4 - int(lens[:768].sum())) % 4
    return random_matrix(lens, 600 + seed)


def exact_mean(n, mean_num, extra, lo, hi, seed, long_row=None):
    """Rows of lo..hi entries (plus one row of `long_row`) adding up to exactly mean_num * n + extra entries."""
    rng = np.random.default_rng(700 + seed)
    lens = rng.integers(lo, hi + 1, n)
    fixed = 0
    if long_row is not None:
        lens[n // 3] = long_row
        fixed = long_row
    rest = np.delete(np.arange(n), n // 3) if long_row is not None else np.arange(n)
    lens[rest] = _exact_total(lens[rest], lo, hi, mean_num * n + extra - fixed, rng)
    return random_matrix(lens, 800 + seed)


def skew(longest, n=8192, seed=0, extra_long=(256, 257)):
    """Rows of 0..8 entries (mean ~ 4.5, so the skew limit is 512) plus rows of `extra_long` entries and one row of
    `longest` entries, spread apart."""
    rng = np.random.default_rng(900 + seed)
    lens = rng.integers(0, 9, n)
    for i, L in enumerate(extra_long):
        lens[700 + 1013 * i] = L
    lens[n // 2 + 5] = longest
    return random_matrix(lens, 1000 + seed)


def skew_edges(n=8192, seed=0):
    """Long rows (2000 entries; mean ~ 24, so the limit is 1536) at row 0, at row n - 1, followed by 40 empty rows,
    and on 1 % of the rows."""
    rng = np.random.default_rng(1100 + seed)
    lens = rng.integers(0, 9, n)
    lens[rng.choice(n, n // 100, replace=False)] = 2000
    lens[[0, n - 1, 3000]] = 2000
    lens[3001:3041] = 0
    return random_matrix(lens, 1200 + seed)


def tiny(n, seed=0):
    rng = np.random.default_rng(1300 + n + seed)
    return random_matrix(rng.integers(0, min(n, 12) + 1, n) if n > 1 else np.array([1]), 1400 + n + seed)


def pairs(n_values, n=4099, seed=0):
    """A 9-point band (offsets -4..4, boundary rows shorter): offsets -4..3 carry one value each, offset +4 carries
    `n_values` values inside every 256-row block, so each block holds 8 + n_values distinct (offset, value) pairs."""
    base = np.array([3.0, -1.25, 0.5, -2.0, 10.0, -0.75, 1.5, -3.5])
    rows = np.repeat(np.arange(n), 9)
    off = np.tile(np.arange(-4, 5), n)
    col = rows + off
    keep = (col >= 0) & (col < n)
    rows, off, col = rows[keep], off[keep], col[keep]
    val = np.where(off < 4, base[np.minimum(off + 4, 7)], 1.0 + ((rows % RPB) * n_values // RPB) / 8.0)
    return _csr(np.bincount(rows, minlength=n), col, val, n)


def ring_large(n=1_500_000, seed=0):
    """1.5 M random rows of 0..12 entries (mean 6), nnz % 4 == 3: every kernel 2 CTA wraps its stage ring."""
    rng = np.random.default_rng(1500 + seed)
    return random_matrix(_trim(rng.integers(0, 13, n), 4, 3), 1600 + seed)


def ring_large_dict(n=1_500_000, seed=0):
    """1.5 M rows; every 256-row block draws 32 of 40 offsets, a row keeps each of 16 slots (slot j: one of the block's
    offsets 2j, 2j + 1) with probability 0.4; random values; nnz % 16 == 13."""
    rng = np.random.default_rng(1700 + seed)
    pool = np.sort(rng.choice(np.arange(-3000, 3001), 40, replace=False))
    nblk = -(-n // RPB)
    sets = np.sort(pool[np.argsort(rng.random((nblk, 40)), axis=1)[:, :32]], axis=1)   # (nblk, 32) sorted
    r = np.arange(n)
    slot_off = sets[r // RPB][:, 0::2] + 0
    pick = rng.random((n, 16)) < 0.5
    slot_off = np.where(pick, sets[r // RPB][:, 1::2], slot_off)
    keep = rng.random((n, 16)) < 0.4
    col = r[:, None] + slot_off
    keep &= (col >= 0) & (col < n)
    lens = _trim(keep.sum(1), 16, 13)
    keep &= np.cumsum(keep, 1) <= lens[:, None]          # slots are in ascending column order already
    return _csr(lens, col[keep], rng.standard_normal(int(lens.sum())), n)


def _family_list():
    F = []  # (id, generator, registration options, fp64 kernel, fp32 kernel)
    for r in range(4):
        F.append((f"tails_{r}", (lambda r=r: tails(r, seed=r)), {}, 2, 2))
    for r in range(16):
        F.append((f"dict32_tail{r}", (lambda r=r: dict_tail(r)), {}, 3, 3))
    F.append(("dict33", lambda: banded_matrix(4099, dict_offsets(4099, 0, extra_block=7), 401), {}, 2, 2))
    F += [("tma_w4672", lambda: tma_width(4672), {}, 2, 2),
          ("tma_w4673", lambda: tma_width(4673), {}, 0, 2),
          ("tma_w4670_s3", lambda: tma_width(4670, s_mod4=3), {}, 0, 2),
          ("tma_w7040", lambda: tma_width(7040, seed=1), {}, 0, 2),
          ("tma_w7041", lambda: tma_width(7041, seed=1), {}, 0, 0),
          ("mean8", lambda: exact_mean(4099, 8, 0, 0, 16, 0, long_row=512), dict(use_tma=0), 0, 0),
          ("mean8p", lambda: exact_mean(4099, 8, 1, 0, 16, 1, long_row=512), dict(use_tma=0), 0, 0),
          ("mean32", lambda: exact_mean(1001, 32, 0, 16, 48, 2), {}, 0, 0),
          ("mean32p", lambda: exact_mean(1001, 32, 1, 16, 48, 3), {}, 1, 1),
          ("mean64", lambda: exact_mean(1001, 64, 0, 33, 95, 4), {}, 1, 1),
          ("mean64p", lambda: exact_mean(1001, 64, 1, 33, 95, 5), {}, 1, 1),
          ("mean128", lambda: exact_mean(1001, 128, 0, 67, 189, 6), {}, 1, 1),
          ("mean128p", lambda: exact_mean(1001, 128, 1, 67, 189, 7), {}, 1, 1),
          ("skew_512", lambda: skew(512), {}, 2, 2),
          ("skew_513", lambda: skew(513, extra_long=(256, 257, 768, 769)), {}, 4, 4),
          ("skew_513_nosplit", lambda: skew(513, extra_long=(256, 257, 768, 769)), dict(use_split=0), 1, 1),
          ("skew_edges", lambda: skew_edges(), {}, 4, 4),
          ("pairs_31", lambda: pairs(23), {}, 5, 5),
          ("pairs_32", lambda: pairs(24), {}, 3, 3)]
    for n, k64, k32 in [(1, 6, 6), (2, 6, 6), (31, 2, 2), (255, 2, 2), (256, 2, 2), (257, 2, 2)]:
        F.append((f"tiny_{n}", (lambda n=n: tiny(n)), {}, k64, k32))
    return F


FAMILIES = _family_list()
LARGE = [("ring_large", lambda: ring_large(), {}, 2, 2),
         ("ring_large_dict", lambda: ring_large_dict(), {}, 3, 3)]
ALL = FAMILIES + LARGE
_BY_ID = {f[0]: f for f in ALL}
TRANSPOSED = [f[0] for f in FAMILIES if f[0].startswith(("tiny", "skew", "mean"))]

_MATS = {}


def _matrix(name):
    if name not in _MATS:
        _MATS[name] = _BY_ID[name][1]()
    return _MATS[name]


def _kernel_want(name, dtype):
    return _BY_ID[name][3] if dtype == torch.float64 else _BY_ID[name][4]


# --------------------------------------------------------------------------------------------------
# Rounding-error bounds of the fused reductions
# --------------------------------------------------------------------------------------------------
def rows_per_visit(plan):
    """Rows one CTA finishes per visit of the kernel that computes y and the dots: 8 warps x 32 / LPR rows for kernel
    1, 256 for the others (kernel 4: 256 threads of bk_vrow_reduce_kernel, one row each)."""
    return 8 * (32 // plan["lanes_per_row"]) if plan["kernel"] == 1 else RPB


def csr_dot_roundings(n, plan, num_sms):
    """Upper bound K on the roundings a product w_i y_i (or y_i y_i) passes through in the fused dot of kernels 0-5:
    1 for the product; the thread's sequential sum over its visits — every kernel launches at least min(blocks, SMs)
    CTAs and walks its blocks grid-stride, a thread taking one row per visit, so V <= ceil(blocks / min(blocks,
    SMs)); bk_block_reduce over up to 9 warps (the TMA / pair kernels add their producer warp): 5 shuffle levels + 4;
    the last CTA's strided pass over at most 2048 partials (<= 8 per thread) and the block tree again (9).  Kernels 6
    / 7 reduce by their own grid (test_stencil_plans.dot_roundings)."""
    if plan["kernel"] in (6, 7):
        return mask_dot_roundings(n, num_sms)
    blocks = max(1, -(-n // rows_per_visit(plan)))
    V = -(-blocks // min(blocks, num_sms))
    return 1 + V + 9 + 8 + 9


def _gamma(K, u):
    return K * u / (1 - K * u)


def check_dot_k(d, yhat, w, K):
    """|d^ - sum w_i y^_i| <= gamma_K sum |w_i y^_i| (the products and the sum are formed in double)."""
    ld = _longdouble()
    p = w.astype(ld) * yhat.astype(ld)
    bound = _gamma(K, 2.0 ** -53) * float(np.sum(np.abs(p)))
    assert abs(float(ld(d) - np.sum(p))) <= bound, (float(d), float(np.sum(p)), bound, K)


def residual_bound(A, x0, b, dtype, K):
    """(rr, bound) for the fused residual r = b - A x0 and rr = r.r: row i of r^ is within
    e_i = gamma_{L_i + 1}(|b_i| + (|A||x0|)_i) of r_i (the row sum's L_i roundings, then the subtraction), and the
    double-precision dot adds gamma_K sum r^_i^2 <= gamma_K sum (|r_i| + e_i)^2, so
    |rr^ - r.r| <= sum (2 |r_i| e_i + e_i^2) + gamma_K sum (|r_i| + e_i)^2."""
    ld = _longdouble()
    y, ax, lens = ref_spmv(A, x0, dtype)
    r = b.astype(ld) - y
    u = ld(2.0) ** (-53 if dtype == torch.float64 else -24)
    m = (lens + 1).astype(ld) * u
    e = m / (1 - m) * (np.abs(b.astype(ld)) + ax)
    ar = np.abs(r)
    bound = np.sum(2 * ar * e + e * e) + ld(_gamma(K, 2.0 ** -53)) * np.sum((ar + e) ** 2)
    return np.sum(r * r), bound


# --------------------------------------------------------------------------------------------------
# CPU tests: the model, the generators, the reference
# --------------------------------------------------------------------------------------------------
def _hand(lens, n=None, seed=0):
    return random_matrix(np.asarray(lens), seed, n)


def test_model_kernel0_vs_kernel1_and_lanes():
    """bk_csr_plan on hand-built matrices at each boundary value and one entry past it."""
    n = 64
    for mean, kernel, lpr in [(32, 0, 8), (64, 1, 8), (128, 1, 16)]:
        at = predict_csr_plan(_hand(np.full(n, mean)), use_tma=0)
        past = predict_csr_plan(_hand(np.r_[np.full(n - 1, mean), mean + 1]), use_tma=0)
        assert (at["kernel"], at["lanes_per_row"], at["mean_row_nnz"]) == (kernel, lpr, float(mean))
        assert past["kernel"] == 1 and past["lanes_per_row"] == {32: 8, 64: 16, 128: 32}[mean]
    # the stream window: 256 entries while mean <= 8
    assert predict_csr_plan(_hand(np.full(n, 8)), use_tma=0)["cap"] == 256
    assert predict_csr_plan(_hand(np.r_[np.full(n - 1, 8), 9]), use_tma=0)["cap"] == 1024


def test_model_skew_limit_and_split():
    lens = np.full(2048, 4)
    lens[5] = 512                                    # mean < 8: the limit is 64 * 8
    assert predict_csr_plan(_hand(lens))["kernel"] == 2
    lens[5] = 513
    p = predict_csr_plan(_hand(lens))
    assert p["kernel"] == 4 and p["max_row_nnz"] == 513
    assert predict_csr_plan(_hand(lens), use_split=0)["kernel"] == 1
    # mean above 8: the limit is 64 * mean, and the long row moves the mean: 1023 rows of 20 and one of 1364 sit exactly
    # on it (64 * 21824 / 1024 = 1364), one of 1365 is past it
    lens = np.full(1024, 20)
    lens[0] = 1364
    assert 64 * lens.sum() / lens.size == 1364 and predict_csr_plan(_hand(lens))["kernel"] == 0
    lens[0] = 1365
    assert predict_csr_plan(_hand(lens))["kernel"] == 4


def test_model_virtual_rows():
    """Rows are cut at 256 entries: 256 stays whole, 257 -> 256 + 1, 768 -> 3 x 256, 769 -> 3 x 256 + 1; empty rows
    keep a virtual row."""
    crow = np.concatenate([[0], np.cumsum([256, 257, 0, 768, 769, 3])])
    vrowptr, vstart = virtual_rows(crow)
    assert np.diff(vrowptr).tolist() == [256, 256, 1, 0, 256, 256, 256, 256, 256, 256, 1, 3]
    assert vstart.tolist() == [0, 1, 3, 4, 7, 11, 12]


def test_model_tma_width_and_alignment():
    for name, k64, k32 in [("tma_w4672", 2, 2), ("tma_w4673", 0, 2), ("tma_w4670_s3", 0, 2), ("tma_w7040", 0, 2),
                           ("tma_w7041", 0, 0)]:
        A = _matrix(name)
        assert predict_csr_plan(A)["kernel"] == k64 and predict_csr_plan(A, torch.float32)["kernel"] == k32, name
    assert tma_stages(4672, 8) == 2 and tma_stages(4704, 8) == 1
    assert tma_stages(7040, 4) == 2 and tma_stages(7072, 4) == 1
    assert predict_csr_plan(_matrix("tails_3"), aligned=False)["kernel"] == 0
    assert predict_csr_plan(_matrix("tails_3"), use_tma=0)["kernel"] == 0


def test_model_dictionary_and_pairs():
    assert predict_csr_plan(_matrix("dict32_tail0"), use_compress=1)["kernel"] == 3
    assert predict_csr_plan(_matrix("dict33"), use_compress=1)["kernel"] == 2
    assert predict_csr_plan(_matrix("dict32_tail0"), use_compress=0)["kernel"] == 2
    assert predict_csr_plan(_matrix("pairs_31"), use_compress=2)["kernel"] == 5
    assert predict_csr_plan(_matrix("pairs_31"), use_compress=1)["kernel"] == 3
    assert predict_csr_plan(_matrix("pairs_32"), use_compress=2)["kernel"] == 3
    # the pair plan's size rule: rows of 2 entries with one row of 8 (or 4) per 32-row chunk pad every chunk to 8 (4)
    # entries per lane: 2 x 2176 pair-stream bytes > 1.5 nnz + 2 x 1152 (kernel 3 instead), 2 x 1152 bytes fit
    for long_len, blk_bytes, kernel in [(8, 2176, 3), (4, 1152, 5)]:
        offs = [np.arange(long_len) if r % 32 == 0 else np.arange(2) for r in range(512)]
        A = banded_matrix(512, offs, 0)
        crow, col, _ = _csr_numpy(A, torch.float64)
        A = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(),
                                    torch.from_numpy(1.0 + col - np.repeat(np.arange(512), np.diff(crow))), size=A.shape)
        lens = np.diff(crow)
        assert pair_block_bytes(lens, 512).tolist() == [blk_bytes] * 2
        assert (2 * blk_bytes > 1.5 * lens.sum() + 2 * 1152) == (kernel == 3)
        assert predict_csr_plan(A, use_compress=2)["kernel"] == kernel


def test_model_kernel3_width_check_never_decides():
    """Kernel 3 is only tried on a kernel 2 plan, and kernel 2's width limit is the tighter one: the widest 4-aligned
    span kernel 2 accepts is cap 4672 (fp64) / 7040 (fp32); the 16-aligned span of the same blocks is at most 24
    entries wider, and two kernel 3 stages fit up to cap 6240 / 11232.  So bk_csr_plan_compress's width test cannot
    fail today."""
    for vs, k2_cap, k3_cap in [(8, 4672, 6240), (4, 7040, 11232)]:
        assert tma_stages(k2_cap, vs) >= 2 and tma_stages(k2_cap + 32, vs) < 2
        assert compress_fits(k3_cap, vs) and not compress_fits(k3_cap + 32, vs)
        assert ((k2_cap + 24 + 31) & ~31) <= k3_cap
    for s in range(64):                              # 16-aligned span - 4-aligned span <= 24 for every start / end
        for e in range(s, s + 64):
            assert (((e + 15) & ~15) - (s & ~15)) - (((e + 3) & ~3) - (s & ~3)) <= 24


@pytest.mark.parametrize("name", [f[0] for f in ALL])
def test_families_model_and_reference(name):
    """Every family: the model selects the kernel the family was built for, fp64 and fp32, and the per-row bound holds
    for torch-CPU's own SpMV."""
    A = _matrix(name)
    opts = _BY_ID[name][2]
    for dt in (torch.float64, torch.float32):
        assert predict_csr_plan(A, dt, **opts)["kernel"] == _kernel_want(name, dt), (name, dt)
    x = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(31))
    check_rows(torch.matmul(A, x).numpy(), A, x.numpy())
    A32 = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values().float(), size=A.shape)
    check_rows(torch.matmul(A32, x.float()).numpy(), A, x.float().numpy(), torch.float32)


def test_generators_hit_their_targets():
    lens = {name: np.diff(_matrix(name).crow_indices().numpy()) for name in _BY_ID if not name.startswith("ring")}
    for r in range(4):
        assert lens[f"tails_{r}"].sum() % 4 == r and (lens[f"tails_{r}"] == 0).any() and lens[f"tails_{r}"].max() > 8
    for r in range(16):
        assert lens[f"dict32_tail{r}"].sum() % 16 == r
    for name, target, s4 in [("tma_w4672", 4672, 0), ("tma_w4673", 4676, 0), ("tma_w4670_s3", 4676, 3),
                             ("tma_w7040", 7040, 0), ("tma_w7041", 7044, 0)]:
        crow = _matrix(name).crow_indices().numpy()
        assert crow[768] % 4 == s4 and _block_span(crow, crow.size - 1, 4) == target, name
    for name, m, extra, n in [("mean8", 8, 0, 4099), ("mean8p", 8, 1, 4099), ("mean32", 32, 0, 1001),
                              ("mean32p", 32, 1, 1001), ("mean64", 64, 0, 1001), ("mean64p", 64, 1, 1001),
                              ("mean128", 128, 0, 1001), ("mean128p", 128, 1, 1001)]:
        assert lens[name].size == n and lens[name].sum() == m * n + extra, name
        assert n % 32 and n % 16 and n % 8
    assert lens["mean8"].max() == 512 == lens["mean8p"].max()
    assert lens["skew_512"].max() == 512 and lens["skew_513"].max() == 769
    assert sorted(lens["skew_513"][lens["skew_513"] > 8].tolist()) == [256, 257, 513, 768, 769]
    e = lens["skew_edges"]
    assert e[0] == e[-1] == e[3000] == 2000 and (e[3001:3041] == 0).all() and (e == 2000).sum() >= 8192 // 100
    A = _matrix("dict33")
    crow, col, _ = _csr_numpy(A, torch.float64)
    rows = np.repeat(np.arange(A.shape[0]), np.diff(crow))
    per_block = [np.unique((col - rows)[rows // RPB == b]).size for b in range(17)]
    assert per_block[7] == 33 and max(per_block[:7] + per_block[8:]) == 32
    for name, want in [("pairs_31", 31), ("pairs_32", 32)]:
        crow, col, val = _csr_numpy(_matrix(name), torch.float64)
        rows = np.repeat(np.arange(crow.size - 1), np.diff(crow))
        assert _distinct_per_block(rows, (col - rows, val.view(np.int64))) == want


def test_large_generators():
    A = _matrix("ring_large")
    lens = np.diff(A.crow_indices().numpy())
    assert A.shape[0] == 1_500_000 and lens.sum() % 4 == 3 and abs(lens.mean() - 6) < 0.05
    # more than 8 blocks per CTA at the default 4 CTAs per SM (and at 2 CTAs per SM: twice that)
    assert -(-A.shape[0] // RPB) > 8 * 148 * 4
    B = _matrix("ring_large_dict")
    crow, col, _ = _csr_numpy(B, torch.float64)
    lens = np.diff(crow)
    rows = np.repeat(np.arange(B.shape[0]), lens)
    assert lens.sum() % 16 == 13 and lens.max() <= 16
    assert np.unique(col - rows).size == 40 and _distinct_per_block(rows, col - rows) == 32
    assert (np.diff(col)[np.diff(rows) == 0] > 0).all()
    assert _block_span(crow, B.shape[0], 4) <= 4672


def test_dot_bound_terms():
    p = dict(kernel=2, lanes_per_row=8)
    assert csr_dot_roundings(256, p, 148) == 1 + 1 + 26
    assert csr_dot_roundings(1_500_000, p, 148) == 1 + 40 + 26
    assert csr_dot_roundings(1001, dict(kernel=1, lanes_per_row=32), 148) == 1 + 1 + 26


# --------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------
@pytest.fixture
def h():
    from pytorch_sparse_solver import _native
    handle = _native.Handle.get(torch.device("cuda"))
    _native.clear_cache()
    yield handle
    _native.clear_cache()


def _register(A, dtype=torch.float64):
    from pytorch_sparse_solver import _native
    _native.clear_cache()
    return _native.register_matrix(A, dtype)


def _seeded(n, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, dtype=dtype, generator=g), torch.randn(n, dtype=dtype, generator=g)


def _misaligned(v):
    """The same values as a view at element offset 1 of a larger CUDA tensor (off 16-byte alignment)."""
    buf = torch.zeros(v.numel() + 1, dtype=v.dtype, device="cuda")
    buf[1:] = v.cuda()
    out = buf[1:]
    assert out.data_ptr() % 16 != 0
    return out


def _assert_info(m, plan, what):
    info = m.info()
    assert info["kernel"] == plan["kernel"], (what, info, plan)
    assert (info["lanes_per_row"], info["max_row_nnz"], info["mean_row_nnz"]) == \
        (plan["lanes_per_row"], plan["max_row_nnz"], plan["mean_row_nnz"]), (what, info, plan)


def _variants(kernel, view_kernel):
    """Launch options that must not change y of a plan: CTAs per SM and stage depth of the TMA kernels, the x prefetch
    of kernel 3, the grid of the others (row sums do not depend on it)."""
    k = view_kernel if kernel == 4 else kernel
    out = []
    if k in (2, 3):
        out += [dict(tma_ctas=c, tma_stages=s) for c, s in itertools.product((2, 3, 4), (2, 0))]
    if k == 3:
        out += [dict(prefetch_x=1), dict(prefetch_x=1, tma_ctas=2, tma_stages=2)]
    if k in (0, 1) or kernel == 4:
        out += [dict(grid_mult_spmv=g, grid_mult_vec=g) for g in (1, 4, 13)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", [f[0] for f in ALL])
def test_spmv_plan_selection_bits_and_rows(h, name, dtype):
    """Registration selects what the model predicts (kernel, lanes per row, max and mean row length; A^T for the tiny,
    skew and mean families); y is within the per-row bound of the long double reference, for an aligned x and for x
    off 16-byte alignment — whatever order a plan sums a row in, every term passes through at most L_i roundings; y is
    bit-identical across the launch variants of the plan and between spmv and spmv_dot; kernels 2, 3 and 5 (fma chains
    in CSR order) give the same bits wherever each applies; the fused dot is within gamma_K of sum w_i y_i."""
    A = _matrix(name)
    opts = _BY_ID[name][2]
    n = A.shape[0]
    x, w = _seeded(n, 41, dtype)
    xd, wd = x.cuda(), w.cuda()
    Ad = A.cuda()
    num_sms = h.device_info()["num_sms"]
    with options(h, **opts):
        m = _register(Ad, dtype)
    plan = predict_csr_plan(A, dtype, **opts)
    assert plan["kernel"] == _kernel_want(name, dtype)
    _assert_info(m, plan, name)
    y = m.spmv(xd)
    yd, d = m.spmv_dot(xd, wd)
    assert torch.equal(yd, y)
    ynp = y.cpu().numpy()
    check_rows(ynp, A, x.numpy(), dtype)
    check_dot_k(float(d), ynp, w.numpy(), csr_dot_roundings(n, plan, num_sms))
    assert torch.equal(m.spmv(_misaligned(xd)), y) and torch.equal(m.spmv_dot(_misaligned(xd), wd)[0], y)
    for var in _variants(plan["kernel"], plan.get("view", {}).get("kernel")):
        with options(h, **var):
            yv = m.spmv(xd)
            ydv, dv = m.spmv_dot(xd, wd)
        assert torch.equal(yv, y) and torch.equal(ydv, y), (name, var, int((yv != y).sum()))
        check_dot_k(float(dv), ynp, w.numpy(), csr_dot_roundings(n, plan, num_sms))
    if plan["kernel"] in (2, 3, 5):
        for uc in (0, 1, 2):
            with options(h, use_compress=uc, **opts):
                mc = _register(Ad, dtype)
            pc = predict_csr_plan(A, dtype, use_compress=uc, **opts)
            assert mc.info()["kernel"] == pc["kernel"] and pc["kernel"] in (2, 3, 5), (name, uc, pc["kernel"])
            assert torch.equal(mc.spmv(xd), y), (name, uc)
    if name in TRANSPOSED:
        At = _transpose(A)
        with options(h, **opts):
            m = _register(Ad, dtype)
            t = m.transpose()
        _assert_info(t, predict_csr_plan(At, dtype, **opts), name + "^T")
        check_rows(t.spmv(xd).cpu().numpy(), At, x.numpy(), dtype)


@pytest.mark.gpu
def test_misaligned_borrowed_arrays_fall_back_to_kernel0(h):
    """val (and an int32 col) borrowed at element offset 1: the library reads them where they are, so kernel 2's bulk
    copies cannot serve them and the plan falls back to kernel 0 with the same per-row bound."""
    from pytorch_sparse_solver import _native
    A = _matrix("tails_3")
    n = A.shape[0]
    for dtype, idx, mis_val, mis_col in [(torch.float64, torch.int64, True, False),
                                         (torch.float32, torch.int64, True, False),
                                         (torch.float64, torch.int32, False, True),
                                         (torch.float32, torch.int32, True, True),
                                         (torch.float64, torch.int32, False, False)]:
        crow = A.crow_indices().to(idx).cuda()
        col = A.col_indices().to(idx).cuda()
        val = A.values().to(dtype).cuda()
        col = _misaligned(col) if mis_col else col
        val = _misaligned(val) if mis_val else val
        m = _native.CsrMatrix(h, crow, col, val, n)
        rp, cp, vp = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        assert h.lib.bk_csr_arrays(m.ptr, ctypes.byref(rp), ctypes.byref(cp), ctypes.byref(vp)) == 0
        assert (vp.value % 16 != 0) == mis_val and (idx == torch.int64 or (cp.value % 16 != 0) == mis_col)
        plan = predict_csr_plan(A, dtype, aligned=not (mis_val or mis_col))
        assert plan["kernel"] == (0 if (mis_val or mis_col) else 2)
        _assert_info(m, plan, (dtype, idx, mis_val, mis_col))
        x = _seeded(n, 45, dtype)[0]
        check_rows(m.spmv(x.cuda()).cpu().numpy(), A, x.numpy(), dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tails_3", "dict32_tail13", "skew_513", "mean64p", "pairs_31", "tiny_257"])
def test_int32_and_int64_indices(h, name):
    A = _matrix(name)
    x = _seeded(A.shape[0], 47)[0].cuda()
    ys = []
    for idx in (torch.int64, torch.int32):
        Ad = torch.sparse_csr_tensor(A.crow_indices().to(idx).cuda(), A.col_indices().to(idx).cuda(),
                                     A.values().cuda(), size=A.shape)
        m = _register(Ad)
        assert m.info()["kernel"] == _kernel_want(name, torch.float64)
        ys.append(m.spmv(x))
    assert torch.equal(ys[0], ys[1])


# --------------------------------------------------------------------------------------------------
# GPU: residual mode (MODE 1, DOTS 2) through CG's r0 and final true residual
# --------------------------------------------------------------------------------------------------
RESIDUAL = ["tails_2", "dict32_tail5", "tma_w4673", "mean8p", "mean32p", "mean128p", "skew_513", "skew_513_nosplit",
            "skew_edges", "pairs_31", "tiny_31", "tiny_2", "ring_large"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", RESIDUAL)
def test_residual_mode(h, name, dtype):
    """CG with maxiter 0 and an x0 runs the plan's residual kernel twice on x0 — r0 = b - A x0 with r0.r0 (rr_last),
    then the final true residual (final_residual = sqrt of its r.r) — and no iteration in between (the init epilogue
    sets `done`), so both equal the same fused residual: rr_last is within the bound of `residual_bound` of the long
    double r.r and final_residual is its square root."""
    A = _matrix(name)
    opts = _BY_ID[name][2]
    n = A.shape[0]
    xt, x0 = _seeded(n, 51, dtype)
    xt, x0 = xt.double(), x0.to(dtype)
    noise = 1e-3 * _seeded(n, 52)[0]
    b = (torch.matmul(A, xt) + noise).to(dtype)
    with options(h, persistent=0, **opts):
        m = _register(A.cuda(), dtype)
        plan = predict_csr_plan(A, dtype, **opts)
        assert m.info()["kernel"] == plan["kernel"]
        x, res = m.cg(b.cuda(), x0.cuda(), 1e-30, 0.0, 0)
    assert res["iterations"] == 0 and torch.equal(x.cpu(), x0)
    rr, bound = residual_bound(A, x0.numpy(), b.numpy(), dtype, csr_dot_roundings(n, plan, h.device_info()["num_sms"]))
    assert abs(_longdouble()(res["rr_last"]) - rr) <= bound, (res["rr_last"], float(rr), float(bound))
    assert res["final_residual"] == math.sqrt(res["rr_last"])


# --------------------------------------------------------------------------------------------------
# GPU: the fused p-update (XMODE 1) of kernel 0 against the separate update kernels
# --------------------------------------------------------------------------------------------------
def spd_variant(A):
    """L + L^T + D from the strictly lower triangle L of A, with D_ii = 1 + sum_j |(L + L^T)_ij|: symmetric, strictly
    diagonally dominant, so SPD; about as many entries per row as A."""
    crow, col, val = _csr_numpy(A, torch.float64)
    n = A.shape[0]
    rows = np.repeat(np.arange(n), np.diff(crow))
    low = col < rows
    r = np.concatenate([rows[low], col[low], np.arange(n)])
    c = np.concatenate([col[low], rows[low], np.arange(n)])
    v = np.concatenate([val[low], val[low], np.zeros(n)])
    v[-n:] = 1.0 + np.bincount(r[:-n], weights=np.abs(v[:-n]), minlength=n)
    order = np.lexsort((c, r))
    return _csr(np.bincount(r, minlength=n), c[order], v[order], n)


# (not tiny_1 / tiny_2: CG solves those exactly in n steps, r becomes 0 and the loop stops before 6 iterations)
XPAY = ["tails_0", "tails_3", "mean8", "mean8p", "tiny_31", "tiny_255", "tiny_257"]


def test_spd_variants_are_spd_and_stay_on_kernel0():
    for name in XPAY:
        S = spd_variant(_matrix(name))
        D = S.to_dense()
        assert torch.equal(D, D.T) and float(torch.linalg.eigvalsh(D).min()) > 0, name
        assert predict_csr_plan(S, use_tma=0, use_compress=0)["kernel"] == 0
    caps = {predict_csr_plan(spd_variant(_matrix(nm)), use_tma=0, use_compress=0)["cap"] for nm in XPAY}
    assert caps == {256, 1024}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", XPAY)
def test_fused_p_update_bits(h, name, dtype):
    """CG on kernel 0 (multi-kernel loop): the fused p-update (the SpMV gathers r + beta p_old, bk_add(r, bk_mul(beta,
    p)), and stores the new p) gives the same x, bit for bit, as the separate x/p-update kernel with and without the
    lagged-x cut, after 6 and after 7 iterations: A p comes from the same stream kernel and bk_op_cg_update /
    bk_op_cg_r reduce r.r the same way."""
    S = spd_variant(_matrix(name))
    n = S.shape[0]
    b = _seeded(n, 55, dtype)[0].cuda()
    with options(h, use_tma=0, use_compress=0):
        m = _register(S.cuda(), dtype)
    assert m.info()["kernel"] == 0
    for iters in (6, 7):
        xs = {}
        for fuse, lag in [(1, 0), (0, 0), (0, 1)]:
            with options(h, persistent=0, fuse_xpay=fuse, cg_lag_x=lag):
                x, res = m.cg(b, None, 0.0, 0.0, iters)
            assert res["iterations"] == iters, (name, fuse, lag, res)
            xs[(fuse, lag)] = x
        ref = xs[(0, 0)]
        for key, x in xs.items():
            assert torch.equal(x, ref), (name, iters, key, int((x != ref).sum()), float((x - ref).abs().max()))
