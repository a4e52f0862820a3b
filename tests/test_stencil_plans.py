"""The stencil SpMV plans — kernel 6 (row bitmasks over 32-row chunk patterns) and kernel 7 (the stencil fast path:
two rows per lane, per-pattern values in the parameter block, one summary per 64-row step) — on IRREGULAR stencil
matrices: grids with inactive cells, rows missing entries next to 64-row step boundaries, bands of coefficients,
asymmetric 1-D bands, and matrices that must stay on kernel 6.

Registration picks the plan from the matrix content alone, so `predict_plan` restates its rules on the CPU and the GPU
tests hold the library to it.  Every SpMV is compared row by row: bit for bit against the plain CSR kernel (kernel 2)
and against an extended-precision reference with a rounding-error bound per row.  All inputs are seeded and finite.
"""
import contextlib
import itertools
import math

import numpy as np
import pytest
import torch

from conftest import rel_diff
from pytorch_sparse_solver import problems
from test_gpu_parity import _banded_coded_matrix

MASK_L = 8            # entries per row and distinct (offset, value) pairs per 32-row chunk (kernel 6)
MASK_PATTERNS = 2048  # distinct chunk patterns kernel 6 holds (half of its hash table)
MASK_CP = 12          # patterns kernel 7 holds in its parameter block
NEITHER = "neither"


# --------------------------------------------------------------------------------------------------
# CPU model of plan selection (bk_csr_plan_mask, bk_mask2_usable)
# --------------------------------------------------------------------------------------------------
def _csr_numpy(A, dtype):
    crow = A.crow_indices().numpy().astype(np.int64)
    col = A.col_indices().numpy().astype(np.int64)
    val = A.values().to(dtype).numpy()
    return crow, col, val


def predict_plan(A, dtype=torch.float64):
    """(kernel, n_patterns, offset_union) that registering the CPU CSR matrix `A` as `dtype` selects: kernel 7, 6 or
    NEITHER (another plan)."""
    crow, col, val = _csr_numpy(A, dtype)
    n = A.shape[0]
    lens = np.diff(crow)
    if n == 0 or col.size == 0 or lens.max() > MASK_L:
        return NEITHER, 0, ()
    rows = np.repeat(np.arange(n), lens)
    if np.any((np.diff(col) <= 0) & (rows[1:] == rows[:-1])):   # columns strictly ascending inside every row
        return NEITHER, 0, ()
    off = col - rows
    vb = (val.view(np.uint64) if val.dtype == np.float64 else val.view(np.uint32)).astype(np.uint64)
    # every chunk's distinct (offset, value bits) pairs, sorted: the chunk's pattern
    ch = rows >> 5
    order = np.lexsort((vb, off, ch))
    ch, off, vb = ch[order], off[order], vb[order]
    new = np.ones(ch.size, dtype=bool)
    new[1:] = (ch[1:] != ch[:-1]) | (off[1:] != off[:-1]) | (vb[1:] != vb[:-1])
    ch, off, vb = ch[new], off[new], vb[new]
    nch = (n + 31) // 32
    cnt = np.bincount(ch, minlength=nch)
    if cnt.max() > MASK_L:
        return NEITHER, 0, ()
    k = np.arange(ch.size) - (np.cumsum(cnt) - cnt)[ch]
    tab = np.zeros((nch, MASK_L, 3), dtype=np.int64)   # (present, offset, value bits) per pattern entry
    tab[ch, k, 0] = 1
    tab[ch, k, 1] = off
    tab[ch, k, 2] = vb.view(np.int64)
    npat = len(np.unique(tab.reshape(nch, -1), axis=0))
    if npat > MASK_PATTERNS:
        return NEITHER, 0, ()
    uni = tuple(int(o) for o in np.unique(off))
    if dtype != torch.float64 or len(uni) > MASK_L or npat > MASK_CP:
        return 6, npat, uni
    if np.any((ch[1:] == ch[:-1]) & (off[1:] == off[:-1])):    # one value per offset and pattern
        return 6, npat, uni
    nu = len(uni)
    odd = sum(1 << q for q, o in enumerate(uni) if o & 1)
    centre = nu >= 3 and uni[nu // 2 - 1: nu // 2 + 2] == (-1, 0, 1)
    shaped = (nu == 5 and odd == 0x0A) or (nu == 7 and odd == 0x14)
    return (7 if centre and shaped else 6), npat, uni


# --------------------------------------------------------------------------------------------------
# Generators (all seeded, CPU, fp64)
# --------------------------------------------------------------------------------------------------
def stencil_grid(shape, kind="poisson", holes=0.0, seed=0, hole_rows=(), drop=(), identity_rows=None, coef=None,
                 index_dtype=torch.int64):
    """5-point (2-D `shape`) or 7-point (3-D) stencil, row index in C order (the last axis is the grid line).

    kind: "poisson" (diagonal 2d, off-diagonals -1) or "convdiff" (first-order upwind, lower side -(1 + g_axis)).
    holes: fraction of inactive cells (plus the rows in `hole_rows`): an inactive row keeps only its diagonal and every
      coupling to it is dropped on both sides, so the Poisson matrix stays SPD.
    drop: (row, offset) entries removed from that row only.
    identity_rows: boolean row mask of Dirichlet rows: off-diagonals removed from the row only, diagonal 1.
    coef: per-row factor of the whole row (bands of coefficients)."""
    d = len(shape)
    N = math.prod(shape)
    strides = [math.prod(shape[a + 1:]) for a in range(d)]
    r = torch.arange(N)
    idx = [(r // strides[a]) % shape[a] for a in range(d)]
    gamma = (1.0, 0.5, 0.25)[:d] if kind == "convdiff" else (0.0,) * d
    offsets, values, masks = [], [], []
    for a in range(d):                                   # lower neighbours, far to near
        offsets.append(-strides[a])
        values.append(-(1.0 + gamma[a]))
        masks.append(idx[a] > 0)
    offsets.append(0)
    values.append(2.0 * d + sum(gamma))
    masks.append(torch.ones(N, dtype=torch.bool))
    for a in reversed(range(d)):                         # upper neighbours, near to far
        offsets.append(strides[a])
        values.append(-1.0)
        masks.append(idx[a] < shape[a] - 1)
    masks = torch.stack(masks, 1)
    active = torch.rand(N, dtype=torch.float64, generator=torch.Generator().manual_seed(seed)) >= holes
    active[list(hole_rows)] = False
    nb = (r[:, None] + torch.tensor(offsets)[None, :]).clamp(0, N - 1)
    centre = offsets.index(0)
    masks &= active[:, None] & active[nb]
    masks[:, centre] = True
    for row, o in drop:
        masks[row, offsets.index(o)] = False
    rowscale = torch.ones(N, dtype=torch.float64) if coef is None else coef.clone()
    if identity_rows is not None:
        masks[identity_rows] = False
        masks[identity_rows, centre] = True
        rowscale[identity_rows] = 1.0 / values[centre]
    A = problems._csr_from_masked_stencil(N, offsets, values, masks, torch.float64, index_dtype, "cpu")
    if coef is None and identity_rows is None:
        return A
    rows = torch.repeat_interleave(r, masks.sum(1))
    return torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values() * rowscale[rows], size=(N, N))


def planted_grid(kind):
    """2-D grid with 128-row lines (two 64-row steps each) and entries removed at step boundaries: the first row of a
    step lacking only -1 (odd steps start mid-line, so this is not a line start) / -1 plus another entry / +1 instead;
    the last row lacking only +1 / +1 plus another / -1 instead; a row inside a step; a whole 32-row chunk and a whole
    64-row step of holes; holes as the first and the last row of the matrix."""
    nx, ny = 40, 128
    drop = [(5 * 64, -1),                                # step 5: only -1 missing in its first row (+ line end)
            (8 * 64 + 63, 1),                            # step 8: only +1 missing in its last row (+ line start)
            (13 * 64, -1), (13 * 64, -ny),               # -1 and another entry
            (16 * 64 + 63, 1), (16 * 64 + 63, ny),
            (21 * 64, 1),                                # the first row lacks +1
            (24 * 64 + 63, -1),                          # the last row lacks -1
            (27 * 64 + 5, -1)]                           # inside the step
    holes = list(range(62 * 32, 63 * 32)) + list(range(35 * 64, 36 * 64)) + [0, nx * ny - 1]
    return stencil_grid((nx, ny), kind, hole_rows=holes, drop=drop)


def banded_grid(nbands, nx=40, ny=64):
    """2-D Poisson on 64-wide lines whose rows are scaled by one coefficient per band of lines; the bands alternate
    between O(1) and O(1e6).  k bands give k + 2 chunk patterns (interior of each band, first and last line)."""
    i = torch.arange(nx * ny) // ny
    band = (i * nbands) // nx
    coef = (1.0 + band.double()) * torch.where(band % 2 == 1, 1e6, 1.0).double()
    return stencil_grid((nx, ny), coef=coef)


def dirichlet_grid(nx=40, ny=64):
    """2-D Poisson whose boundary cells are identity rows (diagonal 1, interior rows keep their couplings): a chunk
    holds two values on offset 0."""
    r = torch.arange(nx * ny)
    i, j = r // ny, r % ny
    return stencil_grid((nx, ny), identity_rows=(i == 0) | (i == nx - 1) | (j == 0) | (j == ny - 1))


def band1d(n, offsets, drop, seed):
    """1-D band (not a grid): entries at offsets `offsets`, each kept with probability 1 - drop, one value per offset;
    row n // 3 is empty."""
    return _banded_coded_matrix(n, offsets, drop, seed)


_B5A, _B5B, _B7 = [-2, -1, 0, 1, 4096], [-64, -1, 0, 1, 2], [-4096, -62, -1, 0, 1, 2, 130]

# (id, generator, expected kernel of the fp64 registration)
FAMILIES = [
    ("holes2d_128x48_poisson", lambda: stencil_grid((48, 128), "poisson", holes=0.01, seed=1), 7),
    ("holes2d_110_convdiff", lambda: stencil_grid((110, 110), "convdiff", holes=0.20, seed=2), 7),
    ("holes3d_64line_poisson", lambda: stencil_grid((12, 16, 64), "poisson", holes=0.05, seed=3), 7),
    ("holes3d_30_convdiff", lambda: stencil_grid((30, 30, 30), "convdiff", holes=0.10, seed=4), 7),
    ("holes3d_30_poisson", lambda: stencil_grid((30, 30, 30), "poisson", holes=0.01, seed=5), 7),
    ("planted_poisson", lambda: planted_grid("poisson"), 7),
    ("planted_convdiff", lambda: planted_grid("convdiff"), 7),
    ("bands1", lambda: banded_grid(1), 7),
    ("bands10", lambda: banded_grid(10), 7),
    ("bands11", lambda: banded_grid(11), 6),             # 13 patterns
    ("band5a_6143", lambda: band1d(2048 * 3 - 1, _B5A, 0.01, 1), 7),
    ("band5a_6144", lambda: band1d(2048 * 3, _B5A, 0.2, 2), 7),
    ("band5a_6145", lambda: band1d(2048 * 3 + 1, _B5A, 0.01, 3), 7),
    ("band5a_6463", lambda: band1d(64 * 100 + 63, _B5A, 0.2, 4), 7),
    ("band5b_4095", lambda: band1d(2048 * 2 - 1, _B5B, 0.2, 5), 7),
    ("band5b_4096", lambda: band1d(2048 * 2, _B5B, 0.01, 6), 7),
    ("band5b_4097", lambda: band1d(2048 * 2 + 1, _B5B, 0.2, 7), 7),
    ("band5b_2111", lambda: band1d(64 * 32 + 63, _B5B, 0.01, 8), 7),
    ("band7_8191", lambda: band1d(2048 * 4 - 1, _B7, 0.01, 9), 7),
    ("band7_8192", lambda: band1d(2048 * 4, _B7, 0.2, 10), 7),
    ("band7_8193", lambda: band1d(2048 * 4 + 1, _B7, 0.01, 11), 7),
    ("band7_6271", lambda: band1d(64 * 97 + 63, _B7, 0.2, 12), 7),
    ("dirichlet_identity_rows", lambda: dirichlet_grid(), 6),   # two values on offset 0
    ("band_odd_far_offset", lambda: band1d(4096, [-2, -1, 0, 1, 63], 0.05, 13), 6),
]
# one of each large enough that every CTA visits a second 2048-row group
LARGE = [
    ("holes2d_2048x1280", lambda: stencil_grid((2048, 1280), "poisson", holes=0.05, seed=21), 7),
    ("holes3d_110", lambda: stencil_grid((110, 110, 110), "poisson", holes=0.05, seed=22), 7),
]
ALL = FAMILIES + LARGE

_MATS = {}


def _matrix(name):
    if name not in _MATS:
        _MATS[name] = dict((c[0], c[1]) for c in ALL)[name]()
    return _MATS[name]


def _transpose(A):
    return A.to_sparse_coo().t().coalesce().to_sparse_csr()


# --------------------------------------------------------------------------------------------------
# Extended-precision reference
# --------------------------------------------------------------------------------------------------
def _longdouble():
    assert np.finfo(np.longdouble).nmant >= 63, "the reference needs an 80-bit (or wider) long double"
    return np.longdouble


def ref_spmv(A, x, dtype=torch.float64):
    """(y, |A||x|, row lengths) in long double from the values `A` holds as `dtype` and the vector x (numpy)."""
    ld = _longdouble()
    crow, col, val = _csr_numpy(A, dtype)
    lens = np.diff(crow)
    prod = val.astype(ld) * x.astype(ld)[col]
    y = np.zeros(A.shape[0], dtype=ld)
    ax = np.zeros(A.shape[0], dtype=ld)
    nz = lens > 0
    if nz.any():
        y[nz] = np.add.reduceat(prod, crow[:-1][nz])
        ax[nz] = np.add.reduceat(np.abs(prod), crow[:-1][nz])
    return y, ax, lens


def check_rows(yhat, A, x, dtype=torch.float64):
    """Row by row: |y^_i - y_i| <= 1.01 L_i u (|A||x|)_i.  The row is one FMA chain over its L_i entries (entries a
    plan pads with value 0 leave the sum unchanged), so gamma_{L_i} u-bounded; the 1 % covers gamma_L vs L u and the
    long double reference's own rounding (2^-64)."""
    ld = _longdouble()
    y, ax, lens = ref_spmv(A, x, dtype)
    u = ld(2.0) ** (-53 if dtype == torch.float64 else -24)
    err = np.abs(yhat.astype(ld) - y)
    bound = ld(1.01) * lens.astype(ld) * u * ax
    bad = np.nonzero(err > bound)[0]
    assert bad.size == 0, f"{bad.size} rows out of bound, first {bad[:8].tolist()}: err {err[bad[:4]]}, bound {bound[bad[:4]]}"


def dot_roundings(n, num_sms):
    """Upper bound K on the roundings any product w_i y_i passes through in the fused dot of kernels 6 / 7:
    1 for the product; the lane's sequential chain — groups of 2048 rows are dealt round-robin to at least
    G = min(groups, 3 * SMs) CTAs (kernel 6 runs 3-5 CTAs per SM, kernel 7 4-6), so a CTA visits V <= ceil(groups / G)
    groups and a lane adds 8 rows per visit, plus one add per 64-row step that returns a partial from kernel 6's chunk
    code (<= 12 V); the block tree (5 shuffle levels + 3 over 8 warps); the last CTA's strided pass over at most 2048
    partials (<= 8 per thread) and the block tree again (8)."""
    groups = max(1, -(-n // 2048))
    G = min(groups, 3 * num_sms)
    V = -(-groups // G)
    return 1 + 12 * V + 8 + 8 + 8


def check_dot(d, yhat, w, num_sms):
    """|d^ - sum w_i y^_i| <= gamma_K sum |w_i y^_i| (a sum whose every term passes through at most K roundings)."""
    ld = _longdouble()
    p = w.astype(ld) * yhat.astype(ld)
    K = dot_roundings(yhat.size, num_sms)
    u = 2.0 ** -53
    bound = K * u / (1 - K * u) * float(np.sum(np.abs(p)))
    assert abs(float(ld(d) - np.sum(p))) <= bound, (float(d), float(np.sum(p)), bound)


# --------------------------------------------------------------------------------------------------
# CPU tests: the model, the generators, the reference
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gen,want", [
    (dict(matrix="poisson3d", n=16), (7, None)), (dict(matrix="poisson3d", n=30), (7, None)),
    (dict(matrix="poisson3d", n=64), (7, 9)), (dict(matrix="convdiff3d", n=48), (7, None)),
    (dict(matrix="poisson2d", nx=200, ny=64), (7, None)), (dict(matrix="poisson2d", nx=64, ny=63), (6, None)),
    (dict(matrix="poisson3d", n=15), (6, None)), (dict(matrix="ldc", nx=32), (6, None)),
    (dict(matrix="ldc", nx=100), (6, None))])
def test_model_on_generated_grids(gen, want):
    """The model agrees with the kernel expectations the GPU suite holds for the generated grids (K7_CASES), and finds
    the 9 patterns of P3D-64."""
    from conftest import build_matrix
    k, npat, uni = predict_plan(build_matrix(gen))
    assert k == want[0], (gen, k, npat, uni)
    if want[1] is not None:
        assert npat == want[1]
    assert predict_plan(build_matrix(gen), torch.float32)[0] == 6


@pytest.mark.parametrize("k,npat,kernel", [(1, 3, 7), (10, 12, 7), (11, 13, 6)])
def test_model_pattern_limit_on_bands(k, npat, kernel):
    """k bands of row coefficients on 64-wide lines: k + 2 patterns; 12 is the most kernel 7 holds."""
    assert predict_plan(banded_grid(k)) == (kernel, npat, (-64, -1, 0, 1, 64))


def test_model_rejections():
    A = stencil_grid((40, 64))
    assert predict_plan(A)[0] == 7
    # a chunk with more than 8 distinct pairs / columns out of order inside a row: no pattern plan at all
    crow, col, val = A.crow_indices(), A.col_indices(), A.values().clone()
    val[:20] = torch.arange(2.0, 22.0, dtype=torch.float64)
    assert predict_plan(torch.sparse_csr_tensor(crow, col, val, size=A.shape))[0] == NEITHER
    c2 = col.clone()
    c2[0], c2[1] = col[1], col[0]
    assert predict_plan(torch.sparse_csr_tensor(crow, c2, A.values(), size=A.shape))[0] == NEITHER
    # two values on one offset inside a pattern, an odd far offset: kernel 6
    assert predict_plan(dirichlet_grid())[0] == 6
    assert predict_plan(band1d(4096, [-2, -1, 0, 1, 63], 0.05, 13))[0] == 6
    assert predict_plan(band1d(4096, [-3, -1, 0, 1, 64], 0.05, 13))[0] == 6
    # no -1 / +1 around the centre, or 6 offsets: kernel 6
    assert predict_plan(band1d(4096, [-64, -2, 0, 2, 64], 0.05, 13))[0] == 6
    assert predict_plan(band1d(4096, [-64, -2, -1, 0, 1, 64], 0.05, 13))[0] == 6


@pytest.mark.parametrize("name,make,want", FAMILIES, ids=[c[0] for c in FAMILIES])
def test_families_model_and_reference(name, make, want):
    """Every family: the model's selection, and the reference agrees with a plain fp64 SpMV to its own bound."""
    A = _matrix(name)
    k, npat, uni = predict_plan(A)
    assert k == want, (name, k, npat, uni)
    assert predict_plan(A, torch.float32)[0] == 6
    x = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(31))
    check_rows(torch.matmul(A, x).numpy(), A, x.numpy())
    A32 = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values().float(), size=A.shape)
    check_rows(torch.matmul(A32, x.float()).numpy(), A, x.float().numpy(), torch.float32)


def test_planted_edges_are_where_they_were_put():
    """The planted family really has the rows the GPU tests rely on."""
    A = planted_grid("poisson")
    crow, col = A.crow_indices(), A.col_indices()

    def offs(r):
        return sorted((col[crow[r]:crow[r + 1]] - r).tolist())
    full = [-128, -1, 0, 1, 128]
    assert offs(5 * 64) == [-128, 0, 1, 128] and offs(5 * 64 + 1) == full
    assert offs(8 * 64 + 63) == [-128, -1, 0, 128]
    assert offs(13 * 64) == [0, 1, 128] and offs(21 * 64) == [-128, -1, 0, 128]
    assert all(offs(r) == [0] for r in list(range(62 * 32, 63 * 32)) + list(range(35 * 64, 36 * 64)) + [0, 5119])


@pytest.mark.parametrize("name,make,want", LARGE, ids=[c[0] for c in LARGE])
def test_large_model(name, make, want):
    A = _matrix(name)
    assert A.shape[0] > 148 * 4 * 2048, "a second group for every CTA"
    assert predict_plan(A)[0] == want


def test_dot_bound_terms():
    # one visit, no partial pass beyond one per thread: 1 + 12 + 24
    assert dot_roundings(2048, 148) == 37
    assert dot_roundings(148 * 3 * 2048 + 1, 148) == 1 + 24 + 24


# --------------------------------------------------------------------------------------------------
# GPU: selection, bits against kernel 2, rows against the reference
# --------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def options(h, **opts):
    saved = {k: h.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            h.set_option(k, v)
        yield
    finally:
        for k, v in saved.items():
            h.set_option(k, v)


@pytest.fixture
def h():
    from pytorch_sparse_solver import _native
    handle = _native.Handle.get(torch.device("cuda"))
    _native.clear_cache()
    yield handle
    _native.clear_cache()


def _register(A, dtype=torch.float64):
    """Fresh registration of the CUDA CSR tensor A and of its transpose (registered with the options in force)."""
    from pytorch_sparse_solver import _native
    _native.clear_cache()
    m = _native.register_matrix(A, dtype)
    return m, m.transpose()


def _seeded(n, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, dtype=dtype, generator=g), torch.randn(n, dtype=dtype, generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("name,make,want", ALL, ids=[c[0] for c in ALL])
def test_spmv_plan_selection_bits_and_rows(h, name, make, want):
    """Registration selects what the model predicts (A and A^T); y and the fused-dot y of kernels 7 and 6 (every
    CTAs-per-SM / prefetch variant of kernel 7) and of the pair-coded plan are bit-identical to kernel 2; y is within the
    per-row bound of the long double reference, the dot within gamma_K of sum w_i y_i; an x 8 bytes off 16-byte
    alignment (kernel 7 falls back to kernel 6 at launch) gives the same bits."""
    A = _matrix(name)
    At = _transpose(A)
    n = A.shape[0]
    x, w = _seeded(n, 41)
    xd, wd = x.cuda(), w.cuda()
    Ad = A.cuda()
    num_sms = h.device_info()["num_sms"]
    with options(h, use_compress=0):
        m2, t2 = _register(Ad)
        assert m2.info()["kernel"] == 2 and t2.info()["kernel"] == 2
        y2, _ = m2.spmv_dot(xd, wd)
        yt2 = t2.spmv(xd)
    with options(h, use_compress=2):          # kernel 5 where a 256-row block has <= 31 pairs (else 3 / 2)
        m5, t5 = _register(Ad)
        y5, _ = m5.spmv_dot(xd, wd)
        yt5 = t5.spmv(xd)
    assert torch.equal(y5, y2) and torch.equal(yt5, yt2)
    m, t = _register(Ad)
    assert m.info()["kernel"] == want == predict_plan(A)[0], (name, m.info()["kernel"])
    assert t.info()["kernel"] == predict_plan(At)[0], (name, t.info()["kernel"])
    with options(h, mask_const=0):
        assert m.info()["kernel"] == 6
        y6, d6 = m.spmv_dot(xd, wd)
        assert torch.equal(m.spmv(xd), y2) and torch.equal(y6, y2) and torch.equal(t.spmv(xd), yt2)
    check_dot(float(d6), y6.cpu().numpy(), w.numpy(), num_sms)
    for cctas, pf in itertools.product((4, 5, 6), (0, 1)) if want == 7 else [(4, 0)]:
        with options(h, mask_cctas=cctas, mask2_prefetch=pf):
            y = m.spmv(xd)
            yd, d = m.spmv_dot(xd, wd)
            yt = t.spmv(xd)
            ytd, dt = t.spmv_dot(xd, wd)
        assert torch.equal(y, y2), (name, cctas, pf, int((y != y2).sum()), float((y - y2).abs().max()))
        assert torch.equal(yd, y2) and torch.equal(yt, yt2) and torch.equal(ytd, yt2), (name, cctas, pf)
        check_dot(float(d), y2.cpu().numpy(), w.numpy(), num_sms)
        check_dot(float(dt), yt2.cpu().numpy(), w.numpy(), num_sms)
    xb = torch.zeros(n + 1, dtype=torch.float64, device="cuda")
    xb[1:] = xd
    assert xb[1:].data_ptr() % 16 == 8
    assert torch.equal(m.spmv(xb[1:]), y2) and torch.equal(m.spmv_dot(xb[1:], wd)[0], y2)
    check_rows(y2.cpu().numpy(), A, x.numpy())
    check_rows(yt2.cpu().numpy(), At, x.numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("name,make,want", FAMILIES, ids=[c[0] for c in FAMILIES])
def test_spmv_fp32_registration_stays_on_kernel6(h, name, make, want):
    """Kernel 7 is fp64 only: the fp32 registration of every family takes kernel 6, bit-identical to kernel 2 and
    within the fp32 per-row bound."""
    A = _matrix(name)
    x = _seeded(A.shape[0], 43, torch.float32)[0]
    Ad = A.cuda()
    with options(h, use_compress=0):
        m2, _ = _register(Ad, torch.float32)
        assert m2.info()["kernel"] == 2
        y2 = m2.spmv(x.cuda())
    m, _ = _register(Ad, torch.float32)
    assert m.info()["kernel"] == predict_plan(A, torch.float32)[0] == 6
    y = m.spmv(x.cuda())
    assert torch.equal(y, y2)
    check_rows(y.cpu().numpy(), A, x.numpy(), torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["planted_convdiff", "band7_8193"])
def test_spmv_int32_and_int64_indices(h, name):
    A = _matrix(name)
    x = _seeded(A.shape[0], 47)[0].cuda()
    ys = []
    for idx in (torch.int64, torch.int32):
        Ad = torch.sparse_csr_tensor(A.crow_indices().to(idx).cuda(), A.col_indices().to(idx).cuda(),
                                     A.values().cuda(), size=A.shape)
        m, _ = _register(Ad)
        assert m.info()["kernel"] == 7
        ys.append(m.spmv(x))
    assert torch.equal(ys[0], ys[1])


# --------------------------------------------------------------------------------------------------
# GPU: solver windows (kernel 7's residual mode and y.y epilogue are reached only through the solvers)
# --------------------------------------------------------------------------------------------------
def solver_system(kind):
    return stencil_grid((24, 24, 24), kind, holes=0.05, seed=51)


def test_solver_systems_take_kernel7():
    for kind in ("poisson", "convdiff"):
        assert predict_plan(solver_system(kind))[0] == 7


def _solve_native(m, method, b, x0, tol, maxiter):
    from pytorch_sparse_solver.module_a import krylov
    if method == "gmres":
        tol_eff, atol_eff = krylov._gmres_effective_tolerances(tol, 0.0, m.n, "cuda")
        x, res = m.gmres(b, x0, tol_eff, atol_eff, 20, maxiter, 0)
    else:
        x, res = getattr(m, method)(b, x0, tol, 0.0, maxiter)
    return x.cpu(), res


def _solve_oracle(A, method, b, x0, tol, maxiter):
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver.module_a import krylov
    if method == "gmres":
        return orc.gmres(A, b, x0, tol=tol, atol=0.0, restart=20, maxiter=maxiter, solve_method="batched",
                         device_type=krylov.GMRES_TOLERANCE_DEVICE or "cuda")
    return getattr(orc, method)(A, b, x0, tol=tol, atol=0.0, maxiter=maxiter)


def _check_solves(h, A, m, method, runs, extra_opts):
    b, _ = problems.manufactured_rhs(A, 0)
    for tol, maxiter, x0 in runs:
        x_ref, info_ref, st = _solve_oracle(A, method, b, x0, tol, maxiter)
        out = {}
        for const in (1, 0):
            with options(h, mask_const=const, **extra_opts):
                out[const] = _solve_native(m, method, b.cuda(), None if x0 is None else x0.cuda(), tol, maxiter)
        (x7, r7), (x6, r6) = out[1], out[0]
        what = (method, tol, maxiter, x0 is not None, extra_opts)
        assert r7["info"] == info_ref and abs(r7["iterations"] - st["iterations"]) <= 2, (what, r7, st)
        assert rel_diff(x7, x_ref) <= 1e-10, (what, rel_diff(x7, x_ref))
        if tol == 0.0:       # fixed window: the same iterates; only the dots' summation grid differs
            assert r7["iterations"] == r6["iterations"] and rel_diff(x7, x6) <= 1e-11, (what, rel_diff(x7, x6))
        else:
            assert abs(r7["iterations"] - r6["iterations"]) <= 1 and rel_diff(x7, x6) <= 1e-10, what


@pytest.mark.gpu
@pytest.mark.parametrize("method,kind,snake", [("cg", "poisson", 0), ("cg", "poisson", 1),
                                               ("bicgstab", "convdiff", 1), ("gmres", "convdiff", 1)])
def test_solver_windows_on_holes(h, method, kind, snake):
    """CG on holes-Poisson, BiCGStab and GMRES(20) on holes-convection-diffusion through the multi-kernel loop (the
    persistent solvers have their own CSR loop): windows of 1, 2, 7 iterations with and without x0 and a full solve at
    tol 1e-10, against the oracle and against the same solve on kernel 6."""
    A = solver_system(kind)
    m, _ = _register(A.cuda())
    assert m.info()["kernel"] == 7
    x0 = _seeded(A.shape[0], 53)[0]
    runs = [(0.0, k, v) for k in (1, 2, 7) for v in (None, x0)] + [(1e-10, None, None)]
    _check_solves(h, A, m, method, runs, dict(persistent=0, snake=snake))


@pytest.mark.gpu
def test_cg_on_large_holes_grid(h):
    """The 1.33 M-row holes grid (every CTA visits two groups) with the solver's own choice of loop."""
    A = _matrix("holes3d_110")
    m, _ = _register(A.cuda())
    assert m.info()["kernel"] == 7
    _check_solves(h, A, m, "cg", [(0.0, 7, _seeded(A.shape[0], 57)[0]), (1e-10, None, None)], {})
