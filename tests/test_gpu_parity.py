"""GPU parity tests: the CUDA path (through the Python API -> ctypes -> C ABI -> sm_100a kernels) against the
golden vectors of the unmodified reference and against the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): solution relative difference <= 1e-10 in fp64, <= 1e-4 in fp32,
iteration counts within +-2, same `info`.
"""
import json

import pytest
import torch

from conftest import GOLD, build_matrix, load_case, rel_diff

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-10
FP32_TOL = 1e-4


def _names(prefix):
    with open(GOLD / "manifest.json") as f:
        return sorted(k for k in json.load(f)["cases"] if k.startswith(prefix))


def _rhs_for(name, entry, data, A_cpu):
    if "b" in data:
        return data["b"]
    if "rand" in name:
        from pytorch_sparse_solver import problems
        return problems.manufactured_rhs(A_cpu, 0)[0]
    return torch.ones(entry["n"], dtype=torch.float64)


@pytest.fixture(scope="module")
def ma():
    from pytorch_sparse_solver import module_a
    from pytorch_sparse_solver.module_a import krylov
    krylov.GMRES_TOLERANCE_DEVICE = "cpu"  # goldens were produced by the reference on CPU tensors (:737-744)
    yield module_a
    krylov.GMRES_TOLERANCE_DEVICE = None


def _last():
    from pytorch_sparse_solver.module_a import krylov
    return krylov.last_result


# --------------------------------------------------------------------------------------------------
# SpMV and the building blocks
# --------------------------------------------------------------------------------------------------
def _random_csr(n, mean, seed, dtype=torch.float64, empty_rows=False, long_row=False):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0 if empty_rows else 1, 2 * mean + 1, (n,), generator=g)
    if long_row:
        lens[n // 3] = min(n, 3000)
        lens[n - 1] = min(n, 777)
    lens = torch.minimum(lens, torch.tensor(n))
    crow = torch.zeros(n + 1, dtype=torch.int64)
    crow[1:] = lens.cumsum(0)
    cols = torch.cat([torch.randperm(n, generator=g)[: int(k)].sort().values for k in lens]) if n else torch.zeros(0)
    vals = torch.randn(int(crow[-1]), dtype=dtype, generator=g)
    return torch.sparse_csr_tensor(crow, cols.long(), vals, size=(n, n))


SPMV_CASES = [
    ("p3d12", lambda: build_matrix(dict(matrix="poisson3d", n=12))),
    ("p2d_33x17", lambda: build_matrix(dict(matrix="poisson2d", nx=33, ny=17))),
    ("cd3d9", lambda: build_matrix(dict(matrix="convdiff3d", n=9))),
    ("rand_mean5_empty", lambda: _random_csr(1000, 5, 1, empty_rows=True)),
    ("rand_mean20", lambda: _random_csr(700, 20, 2)),
    ("rand_mean60", lambda: _random_csr(513, 60, 3)),
    ("rand_mean200", lambda: _random_csr(600, 200, 4)),
    ("rand_longrow", lambda: _random_csr(4000, 4, 5, long_row=True)),
    ("dense_100", lambda: torch.randn(100, 100, dtype=torch.float64, generator=torch.Generator().manual_seed(6)).to_sparse_csr()),
    ("one_by_one", lambda: torch.tensor([[3.0]], dtype=torch.float64).to_sparse_csr()),
    ("n31_tail", lambda: _random_csr(31, 3, 7)),
]


@pytest.mark.parametrize("name,make", SPMV_CASES, ids=[c[0] for c in SPMV_CASES])
@pytest.mark.parametrize("idx", [torch.int64, torch.int32])
def test_spmv_matches_cpu(name, make, idx):
    from pytorch_sparse_solver import _native
    A = make()
    n = A.shape[0]
    x = torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(11))
    ref = torch.matmul(A, x)
    Ad = torch.sparse_csr_tensor(A.crow_indices().to(idx).cuda(), A.col_indices().to(idx).cuda(), A.values().cuda(),
                                 size=A.shape)
    m = _native.register_matrix(Ad)
    y = m.spmv(x.cuda())
    scale = float(torch.matmul(torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values().abs(),
                                                       size=A.shape), x.abs()).max()) + 1e-300
    assert float((y.cpu() - ref).abs().max()) <= 1e-14 * scale * max(1, m.info()["max_row_nnz"]) ** 0.5
    # fused dot
    w = torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(12))
    y2, d = m.spmv_dot(x.cuda(), w.cuda())
    assert torch.equal(y2, y)
    dref = float(torch.dot(w, ref))
    assert abs(float(d) - dref) <= 1e-12 * float(w.abs() @ ref.abs() + 1e-300)


def test_spmv_kernel_selection():
    from pytorch_sparse_solver import _native
    m = _native.register_matrix(build_matrix(dict(matrix="poisson3d", n=12), device="cuda"))
    assert m.info()["kernel"] in (0, 2, 3, 5, 6, 7) and m.info()["max_row_nnz"] == 7
    m2 = _native.register_matrix(_random_csr(600, 200, 4).cuda())
    assert m2.info()["kernel"] == 1


@pytest.mark.parametrize("name,make", SPMV_CASES[:5] + SPMV_CASES[7:8], ids=[c[0] for c in SPMV_CASES[:5] + SPMV_CASES[7:8]])
def test_spmv_tma_and_ldg_row_stream_agree(name, make):
    """The TMA-staged row-stream kernel (kernel 2) against the LDG-staged one (kernel 0) on the same matrix."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    A = make().cuda()
    x = torch.randn(A.shape[0], dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    try:
        h.set_option("use_tma", 0)
        h.set_option("use_compress", 0)
        _native.clear_cache()
        m0 = _native.register_matrix(A)
        y0 = m0.spmv(x)
        k0 = m0.info()["kernel"]
        h.set_option("use_tma", 1)
        h.set_option("use_compress", 3)
        _native.clear_cache()
        m1 = _native.register_matrix(A)
        y1, d1 = m1.spmv_dot(x, x)
        k1 = m1.info()["kernel"]
    finally:
        h.set_option("use_tma", 1)
        h.set_option("use_compress", 3)
        _native.clear_cache()
    assert k0 in (0, 1, 4)
    if k0 == 0 and name != "rand_mean20":
        assert k1 in (2, 3, 5, 6, 7), "short-row matrices should take a staged / coded row-stream kernel"
    scale = float(y0.abs().max()) + 1e-300
    assert float((y0 - y1).abs().max()) <= 1e-13 * scale
    assert abs(float(d1) - float(torch.dot(x, y0))) <= 1e-11 * float(x.abs() @ y0.abs() + 1e-300)


@pytest.mark.parametrize("gen", [dict(matrix="poisson3d", n=13), dict(matrix="convdiff3d", n=10),
                                 dict(matrix="poisson2d", nx=40, ny=27), dict(matrix="ldc", nx=23)])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_spmv_dictionary_coded_columns_bitwise(gen, dtype):
    """Kernel 3 (8-bit dictionary-coded column stream) must equal kernel 2 (int32 columns) bit for bit."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    A = build_matrix(gen, device="cuda")
    x = torch.randn(A.shape[0], dtype=dtype, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    try:
        h.set_option("use_compress", 0)
        _native.clear_cache()
        m2 = _native.register_matrix(A, dtype)
        y2, d2 = m2.spmv_dot(x, x)
        assert m2.info()["kernel"] == 2
        h.set_option("use_compress", 1)
        _native.clear_cache()
        m3 = _native.register_matrix(A, dtype)
        y3, d3 = m3.spmv_dot(x, x)
        assert m3.info()["kernel"] == 3, "stencil matrices have <= 32 distinct offsets per block"
        t3 = m3.transpose()
        yt = t3.spmv(x)
        h.set_option("use_compress", 2)
        _native.clear_cache()
        m5 = _native.register_matrix(A, dtype)
        y5, d5 = m5.spmv_dot(x, x)
        assert m5.info()["kernel"] == 5, "constant-coefficient stencils have <= 31 (offset, value) pairs per block"
        yt5 = m5.transpose().spmv(x)
        h.set_option("use_compress", 3)
        h.set_option("mask_const", 0)            # kernel 6 itself (kernel 7 serves the same plan when the structure fits)
        _native.clear_cache()
        m6 = _native.register_matrix(A, dtype)
        y6, d6 = m6.spmv_dot(x, x)
        assert m6.info()["kernel"] == 6, "constant-coefficient stencils have <= 8 (offset, value) pairs per 32-row chunk"
        assert m6.info()["bytes_stream"] < m5.info()["bytes_stream"] < m3.info()["bytes_stream"] < m2.info()["bytes_stream"]
        h.set_option("mask_const", 1)
        y7, d7 = m6.spmv_dot(x, x)
        k7 = m6.info()["kernel"]
        # fp64 constant-coefficient 7-point / 5-point stencils with an even line length take the stencil fast path; the
        # LDC matrix (two coefficients on one diagonal inside a chunk), odd line lengths and fp32 stay on kernel 6
        want7 = dtype == torch.float64 and gen["matrix"] in ("poisson3d", "convdiff3d") and gen["n"] % 2 == 0
        assert k7 == (7 if want7 else 6), (gen, k7)
        assert torch.equal(y7, y6) and abs(float(d7) - float(d6)) <= 1e-13 * float(x.abs() @ y6.abs())
        assert m2.info()["bytes_stream"] == m2.info()["bytes_matrix"]
        yt6 = m6.transpose().spmv(x)
    finally:
        h.set_option("use_compress", 3)
        h.set_option("mask_const", 1)
        _native.clear_cache()
    assert torch.equal(y2, y3) and float(d2) == float(d3)
    assert torch.equal(y2, y5) and float(d2) == float(d5), "kernel 5 (pair codes, no value stream) must be bit-identical"
    assert torch.equal(y2, y6), "kernel 6 (row bitmasks over chunk patterns) must be bit-identical"
    assert abs(float(d2) - float(d6)) <= 1e-13 * float(x.abs() @ y2.abs())   # reduced over a different grid
    assert torch.equal(yt, yt6)
    ref = torch.matmul(A.cpu().to_dense().T.double(), x.cpu().double())
    assert rel_diff(yt, ref) <= (1e-13 if dtype == torch.float64 else 1e-5)
    assert torch.equal(yt, yt5)


K7_CASES = [
    ("p3d16", dict(matrix="poisson3d", n=16), 7),          # 4096 rows: two groups, every tile near a matrix end or a plane edge
    ("p3d30", dict(matrix="poisson3d", n=30), 7),          # 27000 rows: partial last group, lines of 30 (steps span lines)
    ("p3d64", dict(matrix="poisson3d", n=64), 7),
    ("cd3d48", dict(matrix="convdiff3d", n=48), 7),        # non-symmetric values
    ("p2d_200x64", dict(matrix="poisson2d", nx=200, ny=64), 7),   # 5-point, even line length
    ("p2d_300x300", dict(matrix="poisson2d", nx=300, ny=300), 7),
    ("p2d_64x63", dict(matrix="poisson2d", nx=64, ny=63), 6),     # odd line length: structure not instantiated
    ("p3d15", dict(matrix="poisson3d", n=15), 6),
    ("ldc100", dict(matrix="ldc", nx=100), 6),             # two coefficients on one diagonal inside a chunk
    ("ldc32", dict(matrix="ldc", nx=32), 6),
]


@pytest.mark.parametrize("name,gen,want", K7_CASES, ids=[c[0] for c in K7_CASES])
def test_spmv_stencil_fast_path_kernel7(name, gen, want):
    """Kernel 7 (two rows per lane, 128-bit gathers over the union of the pattern offsets, one summary per 64 rows) against
    kernel 6 on the same registration: y bit-identical in all four output modes (plain, fused dots, residual), every
    CTAs-per-SM variant; matrices whose structure is not instantiated — or that carry two coefficients on one diagonal
    inside a chunk (found the hard way: the LDC pressure matrix) — must stay on kernel 6."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    A = build_matrix(gen, device="cuda")
    n = A.shape[0]
    g = torch.Generator("cuda").manual_seed(21)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    w = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    ref = torch.matmul(A.cpu().to_dense(), x.cpu()) if n <= 30000 else torch.mv(A, x).cpu()
    try:
        _native.clear_cache()
        m = _native.register_matrix(A)
        h.set_option("mask_const", 0)
        assert m.info()["kernel"] == 6
        y6 = m.spmv(x).clone()
        _, d6 = m.spmv_dot(x, w)
        bs6 = m.info()["bytes_stream"]
        h.set_option("mask_const", 1)
        assert m.info()["kernel"] == want, (name, m.info()["kernel"])
        if want == 7 and n >= 200000:    # (small matrices: the steps near the matrix ends read kernel 6's stream as well)
            assert m.info()["bytes_stream"] < bs6
        for cctas in (4, 5, 6):
            h.set_option("mask_cctas", cctas)
            for pf in (0, 1):
                h.set_option("mask2_prefetch", pf)
                y7 = m.spmv(x)
                assert torch.equal(y7, y6), (name, cctas, pf, float((y7 - y6).abs().max()))
                y7d, d7 = m.spmv_dot(x, w)
                assert torch.equal(y7d, y6)
                assert abs(float(d7) - float(d6)) <= 1e-13 * float(w.abs() @ y6.abs() + 1e-300)
        assert rel_diff(y6.cpu(), ref) <= 1e-14
        # the solvers exercise the residual mode (b - A x, ||.||^2) and the y.y / w.y epilogues: a few iterations from
        # x0 != 0 give the same iterates either way (only the dots' summation order differs)
        b = torch.mv(A, x)
        outs = {}
        for const in (0, 1):
            h.set_option("mask_const", const)
            h.set_option("persistent", 0)
            xs, rs = m.bicgstab(b, w, 1e-30, 0.0, 5)
            xg, rg = m.gmres(b, w, 1e-30, 0.0, 8, 1, 0)
            xc, rc = m.cg(b, w, 1e-30, 0.0, 5)
            outs[const] = (xs.clone(), rs["iterations"], xg.clone(), rg["iterations"], xc.clone(), rs["final_residual"])
        assert outs[0][1] == outs[1][1] == 5 and outs[0][3] == outs[1][3]
        for k in (0, 2, 4):
            assert rel_diff(outs[0][k], outs[1][k]) <= 1e-11, (name, k, rel_diff(outs[0][k], outs[1][k]))
        assert abs(outs[0][5] - outs[1][5]) <= 1e-9 * outs[0][5]
    finally:
        h.set_option("mask_const", 1)
        h.set_option("mask_cctas", 4)
        h.set_option("mask2_prefetch", 0)
        h.set_option("persistent", 1)
        _native.clear_cache()


def test_spmv_pair_codes_fall_back_on_varying_values():
    """Stencil sparsity with all-different values: too many (offset, value) pairs -> column codes only (kernel 3)."""
    from pytorch_sparse_solver import _native
    A = build_matrix(dict(matrix="poisson3d", n=12), device="cuda")
    vals = torch.randn(A.values().numel(), dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(8))
    B = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), vals, size=A.shape)
    m = _native.register_matrix(B)
    assert m.info()["kernel"] == 3
    x = torch.randn(A.shape[0], dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(9))
    assert rel_diff(m.spmv(x), torch.matmul(B.cpu().to_dense(), x.cpu())) <= 1e-13


def test_spmv_dictionary_falls_back_on_unstructured():
    from pytorch_sparse_solver import _native
    m = _native.register_matrix(_random_csr(1000, 5, 1, empty_rows=True).cuda())
    assert m.info()["kernel"] == 2


def _arrowhead(n, dtype=torch.float64):
    """SPD arrowhead: dense first row/column + strong diagonal — mean row length ~3, one row of n entries."""
    i = torch.arange(1, n)
    rows = torch.cat([torch.arange(n), torch.zeros(n - 1, dtype=torch.long), i])
    cols = torch.cat([torch.arange(n), i, torch.zeros(n - 1, dtype=torch.long)])
    vals = torch.cat([torch.full((n,), 4.0, dtype=dtype), torch.full((2 * (n - 1),), -1.0 / n ** 0.5, dtype=dtype)])
    vals[0] = 6.0
    return torch.sparse_coo_tensor(torch.stack([rows, cols]), vals, (n, n)).coalesce().to_sparse_csr()


@pytest.mark.parametrize("n", [700, 5000, 70000])
def test_skewed_matrix_row_splitting(ma, n):
    """A few very long rows among short ones: kernel 4 (virtual rows + ordered reduction) vs CPU, and CG vs the oracle."""
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import _native
    A = _arrowhead(n)
    m = _native.register_matrix(A.cuda())
    assert m.info()["kernel"] == 4 and m.info()["max_row_nnz"] == n
    x = torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(4))
    ref = torch.matmul(A, x)
    y, d = m.spmv_dot(x.cuda(), x.cuda())
    assert rel_diff(y, ref) <= 1e-13
    assert abs(float(d) - float(x @ ref)) <= 1e-11 * float(x.abs() @ ref.abs())
    yt = m.transpose().spmv(x.cuda())                     # symmetric: A^T x == A x
    assert rel_diff(yt, ref) <= 1e-13
    b = torch.matmul(A, torch.ones(n, dtype=torch.float64))
    x_ref, info_ref, st = orc.cg(A, b, tol=1e-10)
    xs, info = ma.cg(A.cuda(), b.cuda(), tol=1e-10)
    assert info == info_ref == 0 and abs(_last()["iterations"] - st["iterations"]) <= 2
    assert rel_diff(xs, x_ref) <= FP64_TOL
    xb, info = ma.bicgstab(A.cuda(), b.cuda(), tol=1e-10)
    assert info == 0 and rel_diff(xb, x_ref) <= 1e-8
    xg, info = ma.gmres(A.cuda(), b.cuda(), tol=1e-10, restart=20)
    assert info == 0 and rel_diff(xg, x_ref) <= 1e-8


def test_spmv_fp32():
    from pytorch_sparse_solver import _native
    A = build_matrix(dict(matrix="convdiff3d", n=10))
    x = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    ref = torch.matmul(A, x)
    m = _native.register_matrix(A.cuda(), torch.float32)
    y = m.spmv(x.float().cuda())
    assert y.dtype == torch.float32
    assert rel_diff(y, ref) <= 1e-6


@pytest.mark.parametrize("n", [1, 2, 3, 255, 256, 1000, 65537, 1 << 20])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_dot_nrm2_axpby(n, dtype):
    from pytorch_sparse_solver import _native
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, dtype=torch.float64, generator=g)
    y = torch.randn(n, dtype=torch.float64, generator=g)
    xd, yd = x.to(dtype).cuda(), y.to(dtype).cuda()
    xr, yr = xd.cpu().double(), yd.cpu().double()
    tol = 1e-13 if dtype == torch.float64 else 1e-6
    assert abs(float(_native.dot(xd, yd)) - float(xr @ yr)) <= 1e-13 * float(xr.abs() @ yr.abs()) + 1e-300
    assert abs(float(_native.nrm2(xd)) - float(torch.linalg.norm(xr))) <= 1e-13 * float(torch.linalg.norm(xr))
    z = _native.axpby(1.5, xd, -0.25, yd)
    assert rel_diff(z, 1.5 * xr - 0.25 * yr) <= tol
    # misaligned views take the scalar path
    if n > 3:
        assert abs(float(_native.dot(xd[1:], yd[1:])) - float(xr[1:] @ yr[1:])) <= 1e-13 * float(xr.abs() @ yr.abs())


def test_reductions_are_bitwise_reproducible():
    from pytorch_sparse_solver import _native
    x = torch.randn(3_000_001, dtype=torch.float64, device="cuda")
    vals = {float(_native.dot(x, x)) for _ in range(5)}
    assert len(vals) == 1


# --------------------------------------------------------------------------------------------------
# solvers vs the reference goldens
# --------------------------------------------------------------------------------------------------
def _solve_case(ma, name, manifest, idx=torch.int64, **override):
    entry = manifest["cases"][name]
    data = load_case(name)
    A_cpu = build_matrix(entry["gen"])
    b = _rhs_for(name, entry, data, A_cpu)
    A = torch.sparse_csr_tensor(A_cpu.crow_indices().to(idx).cuda(), A_cpu.col_indices().to(idx).cuda(),
                                A_cpu.values().cuda(), size=A_cpu.shape)
    x0 = data["x0"].cuda() if "x0" in data else None
    kw = dict(entry["kwargs"])
    kw.update(override)
    if entry.get("jacobi") and "M" not in kw:
        kw["M"] = ma.JacobiPreconditioner(A)     # built-in M: stays on the native path (bk_cg_jacobi)
    x, info = getattr(ma, entry["kind"])(A, b.cuda(), x0, **kw)
    return entry, data, x, info


def _check_against_golden(entry, data, x, info, tol=FP64_TOL):
    res = _last()
    assert x.dtype == torch.float64 and x.is_cuda
    assert info == entry["info"]
    assert abs(int(res["iterations"]) - entry["iterations"]) <= 2, (res["iterations"], entry["iterations"])
    if "x" in data:
        assert rel_diff(x, data["x"]) <= tol
    else:
        idx = data["x_sample_idx"]
        assert rel_diff(x.cpu()[idx], data["x_sample"]) <= tol
        assert abs(float(torch.linalg.norm(x)) - entry["x_norm"]) <= tol * entry["x_norm"]


@pytest.mark.parametrize("name", _names("cg_"))
def test_cg_golden(ma, manifest, name):
    entry, data, x, info = _solve_case(ma, name, manifest)
    _check_against_golden(entry, data, x, info)
    if entry["kwargs"].get("tol", 1) == 0.0:  # fixed-iteration window: exact count
        assert _last()["iterations"] == entry["iterations"]


@pytest.mark.parametrize("name", _names("bicgstab_"))
def test_bicgstab_golden(ma, manifest, name):
    entry, data, x, info = _solve_case(ma, name, manifest)
    _check_against_golden(entry, data, x, info)


@pytest.mark.parametrize("name", _names("gmres_"))
def test_gmres_golden(ma, manifest, name):
    entry, data, x, info = _solve_case(ma, name, manifest)
    # LDC systems are singular (all-Neumann): compare after removing the constant null-space component too
    tol = FP64_TOL if "ldc" not in name else 5e-10
    _check_against_golden(entry, data, x, info, tol=tol)
    # restart cycles must agree exactly; matvec counts within the +-2 iteration band per cycle
    assert _last()["iterations"] == entry["iterations"]


@pytest.mark.parametrize("name", ["cg_p3d16_rand", "bicgstab_cd3d16_rand", "gmres_cd3d12_batched"])
def test_int32_indices_and_stream_mode(ma, manifest, name):
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    entry, data, x64, info = _solve_case(ma, name, manifest)
    try:
        h.set_option("loop_mode", 1)  # plain stream launches instead of the CUDA graph
        _native.clear_cache()
        entry, data, x32, info2 = _solve_case(ma, name, manifest, idx=torch.int32)
    finally:
        h.set_option("loop_mode", 0)
    assert info == info2
    assert torch.equal(x64, x32), "graph and stream loops must give bitwise identical results"


@pytest.mark.parametrize("name", ["cg_p3d16_rand", "bicgstab_cd3d16_rand", "gmres_ldc32_step1_batched"])
def test_solvers_bitwise_deterministic(ma, manifest, name):
    xs = [_solve_case(ma, name, manifest)[2] for _ in range(3)]
    assert torch.equal(xs[0], xs[1]) and torch.equal(xs[0], xs[2])


@pytest.mark.parametrize("opts", [dict(persistent=0), dict(persistent=0, use_compress=2), dict(persistent=0, mask_window=1), dict(persistent=0, mask_prefetch=0), dict(persistent=0, mask_window=1, mask_wgroup=2, mask_ctas=2, tma_stages=2), dict(persistent=0, mask_window=1, mask_wgroup=8, mask_ctas=3), dict(persistent=0, mask_group=1, mask_ctas=2), dict(persistent=0, mask_group=3, mask_ctas=6, snake=0), dict(persistent=0, fuse_xpay=1), dict(persistent=0, fuse_xpay=0), dict(persistent=0, snake=0), dict(persistent=0, fuse_xpay=1, snake=0), dict(persistent=0, chunk=2), dict(persistent=0, use_tma=0), dict(persistent=0, use_compress=0), dict(persistent=0, use_compress=1),
                                  dict(persistent=0, grid_mult_spmv=2, grid_mult_vec=2), dict(persistent=1)])
def test_cg_kernel_variants(ma, manifest, opts):
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    saved = {k: h.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            h.set_option(k, v)
        _native.clear_cache()
        for name in ("cg_p3d16_rand", "cg_p2d24x20_x0", "cg_p3d64_ones_digest", "cg_p3d16_fixed10"):
            entry, data, x, info = _solve_case(ma, name, manifest)
            _check_against_golden(entry, data, x, info)
    finally:
        for k, v in saved.items():
            h.set_option(k, v)
        _native.clear_cache()


def test_dense_and_coo_inputs(ma, manifest):
    """The reference's own tests feed dense matrices (test_module_a.py:93-124)."""
    entry = manifest["cases"]["cg_tridiag100"]
    data = load_case("cg_tridiag100")
    A = build_matrix(entry["gen"]).to_dense()
    for Ain in (A.cuda(), A.to_sparse_coo().cuda()):
        x, info = ma.cg(Ain, data["b"].cuda(), tol=1e-10, maxiter=1000)
        assert info == 0 and rel_diff(x, data["x"]) <= 1e-9  # ill-conditioned (kappa ~ 4e3): loose x gate


def test_fp32_native_path(ma, manifest):
    """fp32 A and b select the native fp32 kernels (the reference raises there); parity vs the fp64 golden <= 1e-4."""
    entry = manifest["cases"]["cg_p3d16_rand"]
    data = load_case("cg_p3d16_rand")
    A = build_matrix(entry["gen"])
    A32 = torch.sparse_csr_tensor(A.crow_indices().cuda(), A.col_indices().cuda(), A.values().float().cuda(),
                                  size=A.shape)
    x, info = ma.cg(A32, data["b"].float().cuda(), tol=1e-6)
    assert x.dtype == torch.float32
    assert rel_diff(x, data["x"]) <= FP32_TOL
    entry = manifest["cases"]["bicgstab_cd3d16_rand"]
    data = load_case("bicgstab_cd3d16_rand")
    A = build_matrix(entry["gen"])
    A32 = torch.sparse_csr_tensor(A.crow_indices().cuda(), A.col_indices().cuda(), A.values().float().cuda(),
                                  size=A.shape)
    x, info = ma.bicgstab(A32, data["b"].float().cuda(), tol=1e-6)
    assert rel_diff(x, data["x"]) <= FP32_TOL
    x, info = ma.gmres(A32, data["b"].float().cuda(), tol=1e-6, restart=30)
    assert rel_diff(x, data["x"]) <= FP32_TOL


def test_upcast_inputs(ma, manifest):
    """fp32 b / x0 with an fp64 matrix are upcast and x comes back fp64 (reference :979-980)."""
    entry = manifest["cases"]["cg_p2d32_ones"]
    data = load_case("cg_p2d32_ones")
    A = build_matrix(entry["gen"], device="cuda")
    x, info = ma.cg(A, torch.ones(entry["n"], dtype=torch.float32, device="cuda"), tol=1e-8)
    assert x.dtype == torch.float64 and info == 0
    assert rel_diff(x, data["x"]) <= FP64_TOL


def test_host_route_cpu_tensors(ma, manifest):
    """CPU tensors go through bk_solve_host (H2D, CUDA solve, D2H) and return a CPU tensor."""
    for name in ("cg_p3d16_rand", "bicgstab_cd3d16_rand", "gmres_cd3d12_incremental"):
        entry = manifest["cases"][name]
        data = load_case(name)
        A = build_matrix(entry["gen"])
        x, info = getattr(ma, entry["kind"])(A, data["b"], **entry["kwargs"])
        assert not x.is_cuda and info == entry["info"]
        assert rel_diff(x, data["x"]) <= FP64_TOL
        assert _last()["route"] == "host"


# --------------------------------------------------------------------------------------------------
# transpose + autograd
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,make", SPMV_CASES, ids=[c[0] for c in SPMV_CASES])
def test_transpose_matches_cpu(name, make):
    from pytorch_sparse_solver import _native
    A = make()
    m = _native.register_matrix(A.cuda())
    t = m.transpose()
    crow, col, val = t.arrays()
    At = A.to_dense().T.contiguous().to_sparse_csr() if A.shape[0] <= 1200 else None
    x = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(5))
    ref = torch.matmul(A.to_dense().T, x) if A.shape[0] <= 4096 else None
    y = t.spmv(x.cuda())
    assert rel_diff(y, ref) <= 1e-13
    # structure: sorted columns inside each row, same nnz, deterministic
    assert int(crow[-1]) == A.values().numel()
    crow2, col2, val2 = _native.register_matrix(A.clone().cuda()).transpose().arrays()
    assert torch.equal(col, col2) and torch.equal(val, val2) and torch.equal(crow, crow2)
    if At is not None and A.values().numel() == At.values().numel():
        assert torch.equal(crow.cpu().long(), At.crow_indices())
        assert torch.equal(col.cpu().long(), At.col_indices())
        assert torch.equal(val.cpu(), At.values())


@pytest.mark.parametrize("kind", ["cg", "bicgstab", "gmres"])
@pytest.mark.parametrize("layout", ["csr", "dense", "coo"])
def test_autograd_grad_b(ma, manifest, kind, layout):
    entry = manifest["autograd"][f"autograd_{kind}"]
    data = load_case(f"autograd_{kind}")
    A = build_matrix(entry["gen"])
    if layout == "dense":
        Ad = A.to_dense().cuda()
    elif layout == "coo":
        Ad = A.to_sparse_coo().cuda()
    else:
        Ad = A.cuda()
    b = data["b"].cuda().requires_grad_(True)
    x, info = getattr(ma, kind)(Ad, b, **entry["kwargs"])
    assert info == entry["info"]
    (x ** 2).sum().backward()
    assert b.grad is not None and torch.isfinite(b.grad).all()
    assert rel_diff(b.grad, data["grad_b"]) <= 1e-9
    assert rel_diff(x, data["x"]) <= FP64_TOL


@pytest.mark.parametrize("layout", ["csr", "coo", "dense"])
def test_optional_gradient_wrt_matrix(ma, manifest, layout):
    """Opt-in dL/dA (SURVEY 8f-3) against the analytic -A^-T (dL/dx) x^T on the pattern; default stays None (:1248)."""
    from pytorch_sparse_solver.module_a import krylov
    entry = manifest["autograd"]["autograd_bicgstab"]
    data = load_case("autograd_bicgstab")
    A_cpu = build_matrix(entry["gen"])
    Ad = A_cpu.to_dense()
    x_true = torch.linalg.solve(Ad, data["b"])
    gA_true = -torch.outer(torch.linalg.solve(Ad.T, 2 * x_true), x_true)
    A = {"csr": A_cpu.cuda(), "coo": A_cpu.to_sparse_coo().coalesce().cuda(), "dense": Ad.cuda()}[layout]
    A.requires_grad_(True)
    b = data["b"].cuda().requires_grad_(True)
    x, info = ma.bicgstab(A, b, tol=1e-12)
    (x ** 2).sum().backward()
    assert A.grad is None and b.grad is not None          # reference behaviour
    krylov.GRAD_WRT_A = True
    try:
        b.grad = None
        x, info = ma.bicgstab(A, b, tol=1e-12)
        (x ** 2).sum().backward()
    finally:
        krylov.GRAD_WRT_A = False
    assert A.grad is not None and A.grad.layout == A.layout
    got = A.grad.to_dense().cpu()
    mask = (Ad != 0) if layout != "dense" else torch.ones_like(Ad, dtype=torch.bool)
    assert rel_diff(got[mask], gA_true[mask]) <= 1e-8
    assert float(got[~mask].abs().max() if (~mask).any() else 0.0) == 0.0


@pytest.mark.parametrize("solve_method", ["batched", "incremental"])
def test_autograd_ldc_gmres_config4(ma, manifest, solve_method):
    """BASELINE configs[3]: GMRES(30) on the LDC pressure system (CSR input) with the implicit-diff backward."""
    entry = manifest["autograd"]["autograd_gmres_ldc32"]
    data = load_case("autograd_gmres_ldc32")
    A = build_matrix(entry["gen"], device="cuda")
    b = data["b"].cuda().requires_grad_(True)
    x, info = ma.gmres(A, b, solve_method=solve_method, **entry["kwargs"])
    assert info == entry["info"]
    (x ** 2).sum().backward()
    assert rel_diff(x, data["x"]) <= (5e-10 if solve_method == "batched" else 1e-7)
    assert rel_diff(b.grad, data["grad_b"]) <= (1e-8 if solve_method == "batched" else 1e-6)


@pytest.mark.parametrize("kind", ["cg", "bicgstab", "gmres"])
def test_legacy_differentiable(ma, manifest, kind):
    entry = manifest["autograd"][f"autograd_{kind}"]
    data = load_case(f"autograd_{kind}")
    A = build_matrix(entry["gen"], device="cuda")
    b = data["b"].cuda().requires_grad_(True)
    x = getattr(ma, f"{kind}_differentiable")(A, b, **entry["kwargs"])
    (x ** 2).sum().backward()
    assert rel_diff(b.grad, data["grad_b"]) <= 1e-9


# --------------------------------------------------------------------------------------------------
# router
# --------------------------------------------------------------------------------------------------
def test_sparse_solver_module_a(manifest):
    import pytorch_sparse_solver as pss
    entry = manifest["cases"]["cg_p2d32_ones"]
    data = load_case("cg_p2d32_ones")
    A = build_matrix(entry["gen"], device="cuda")
    b = torch.ones(entry["n"], dtype=torch.float64, device="cuda")
    solver = pss.SparseSolver()
    x, result = solver.solve(A, b, method="cg", backend="module_a", tol=1e-8)
    assert result.converged and result.backend == "module_a" and result.method == "cg"
    assert result.residual < 1e-7 and result.iterations == entry["iterations"]
    assert rel_diff(x, data["x"]) <= FP64_TOL
    x2, r2 = pss.solve(A, b, method="bicgstab", tol=1e-8)
    assert r2.converged and rel_diff(x2, data["x"]) <= 1e-7
    x3, r3 = pss.gmres(A, b, tol=1e-8, restart=30)
    assert r3.converged
    with pytest.raises(ValueError):
        solver.solve(A, b, backend="module_b")
    with pytest.raises(ValueError):
        solver.solve(A, b, method="nope", backend="module_a")


# --------------------------------------------------------------------------------------------------
# full-size configs of BASELINE.json (digests measured with the reference at survey time)
# --------------------------------------------------------------------------------------------------
def test_cg_poisson3d_256_full_size(ma, manifest):
    """Config 2: CG fp64, 7-point Poisson 256^3, b = ones, tol 1e-8 — reference: 611 iterations, info 0."""
    from pytorch_sparse_solver import problems
    dg = manifest["survey_digests"]["cg_p3d256_ones_tol1e-8"]
    A = problems.poisson3d_csr(256, device="cuda")
    b = torch.ones(A.shape[0], dtype=torch.float64, device="cuda")
    x, info = ma.cg(A, b, tol=1e-8)
    res = _last()
    assert info == dg["info"]
    assert abs(res["iterations"] - dg["iterations"]) <= 2
    assert abs(float(torch.linalg.norm(x)) - dg["x_norm"]) <= 1e-9 * dg["x_norm"]
    assert abs(float(x[0]) - dg["x_0"]) <= 1e-8 * abs(dg["x_0"])
    assert abs(float(x[8388608]) - dg["x_8388608"]) <= 1e-8 * abs(dg["x_8388608"])
    assert res["final_residual"] / res["b_norm"] <= 1e-8
    # size-independent property: CG is linear in b for a fixed iteration window
    x10, _ = ma.cg(A, b, tol=0.0, atol=0.0, maxiter=10)
    dg10 = manifest["survey_digests"]["cg_p3d256_ones_maxiter10"]
    assert abs(float(torch.linalg.norm(x10)) - dg10["x_norm"]) <= 1e-10 * dg10["x_norm"]
    x10s, _ = ma.cg(A, 4.0 * b, tol=0.0, atol=0.0, maxiter=10)
    assert rel_diff(x10s, 4.0 * x10) <= 1e-13


def test_bicgstab_convdiff3d_256_full_size(ma, manifest):
    """Config 3: BiCGStab fp64, upwind convection-diffusion 256^3, b = A randn(seed 0), tol 1e-8 — reference: 399 its."""
    from pytorch_sparse_solver import problems
    dg = manifest["survey_digests"]["bicgstab_cd3d256_rand_tol1e-8"]
    A = problems.convdiff3d_csr(256, device="cuda")
    b, xt = problems.manufactured_rhs(A, 0)
    assert abs(float(torch.linalg.norm(b)) - dg["b_norm"]) <= 1e-12 * dg["b_norm"]
    x, info = ma.bicgstab(A, b, tol=1e-8)
    res = _last()
    assert info == dg["info"]
    # the reference's own self-noise at tol 1e-8 is a few iterations / 2e-10 in x (BASELINE.md §2)
    assert abs(res["iterations"] - dg["iterations"]) <= 8
    assert abs(float(torch.linalg.norm(x)) - dg["x_norm"]) <= 1e-8 * dg["x_norm"]
    assert res["final_residual"] / res["b_norm"] <= 1e-8
    assert rel_diff(x, xt) <= 1e-5


def test_bicgstab_convdiff3d_256_tol1e10_parity_gate(ma, manifest):
    """Config 3 at the tolerance SURVEY 8c / 8d prescribe for the x gate (tol 1e-10), against the digest of the unmodified
    reference (oracle/pin_round2.py --full: 477 iterations, ||x||, 4096 sampled entries).

    What the gate can be at this size was MEASURED with the reference itself (oracle/ref_selfnoise.py, manifest
    round2.ref_selfnoise_bicgstab_cd3d256): run with 8 and with 3 OpenMP threads — i.e. with two summation orders in
    torch's CPU dot / SpMV — the reference takes 477 vs 475 iterations and its two solutions differ by 1.5e-9 (SURVEY's
    4e-13 was measured at 128^3 and does not carry over to 256^3).  Two runs are a lower bound of that spread; its scale
    is the forward error: the reference's x is 1.3e-8 away from the manufactured solution (conditioning x residual), and
    so is ours — two such iterates can differ by up to the sum.  Round 2 changed our summation order twice (kernel 6,
    kernel 7 with two rows per lane): 472 iterations / 2.6e-9 and then 8.6e-9 from the digest.  The gate therefore is:
    iterations within 6 of the digest; OUR forward error no worse than 1.25 x the reference's own (measured here from
    the digest's samples against the manufactured solution); x within max(5e-9, 3 x self-noise, 2 x the reference's
    forward error) of the digest; the TRUE residual meets tol."""
    from pytorch_sparse_solver import problems
    dg = manifest["survey_digests"]["bicgstab_cd3d256_rand_tol1e-10"]
    d2 = manifest["round2"]["digest_bicgstab_cd3d256_tol1e-10"]
    noise = manifest["round2"]["ref_selfnoise_bicgstab_cd3d256"]
    data = load_case("digest_bicgstab_cd3d256_tol1e-10")
    assert d2["x_norm"] == dg["x_norm"] and d2["info"] == dg["info"] == 0
    assert noise["rel_diff_between_runs"] > 1e-10 and abs(noise["8"]["iterations_est"] - noise["3"]["iterations_est"]) >= 2
    A = problems.convdiff3d_csr(256, device="cuda")
    b, xt = problems.manufactured_rhs(A, 0)
    x, info = ma.bicgstab(A, b, tol=1e-10)
    res = _last()
    assert info == 0
    assert abs(res["iterations"] - dg["iterations"]) <= 6, (res["iterations"], dg["iterations"])
    idx = data["x_sample_idx"]
    xs, xts = x.cpu()[idx], xt.cpu()[idx]
    e_ref = rel_diff(data["x_sample"], xts)       # the reference's own forward error on the sampled entries
    e_ours = rel_diff(xs, xts)
    assert 1e-9 < e_ref < 1e-7, e_ref
    assert e_ours <= 1.25 * e_ref, (e_ours, e_ref)
    gate = max(5e-9, 3.0 * noise["rel_diff_between_runs"], 2.0 * e_ref)
    assert abs(float(torch.linalg.norm(x)) - dg["x_norm"]) <= gate * dg["x_norm"]
    assert rel_diff(xs, data["x_sample"]) <= gate, (rel_diff(xs, data["x_sample"]), gate)
    assert res["final_residual"] / res["b_norm"] <= 1e-10
    assert rel_diff(x, xt) <= 1e-7      # forward error = conditioning x residual
    # at a size where the reference does not differ from itself the gate is the north star's: 64^3, tol 1e-10
    entry, data64, x64, info64 = _solve_case(ma, "bicgstab_cd3d64_rand_digest", manifest)
    _check_against_golden(entry, data64, x64, info64)


@pytest.mark.parametrize("kind", ["cg", "bicgstab", "gmres"])
@pytest.mark.parametrize("layout", ["csr", "dense", "coo"])
def test_autograd_with_callable_preconditioner(ma, manifest, kind, layout):
    """The reference attaches the implicit-diff backward whenever A is a 2-D tensor, also with a callable M
    (:1079-1086, :1145-1152, :775-782); the adjoint solve reuses M.  Goldens: the reference's own b.grad."""
    entry = manifest["round2"][f"autograd_{kind}_jacobi"]
    data = load_case(f"autograd_{kind}_jacobi")
    A = build_matrix(entry["gen"])
    Ad = {"csr": A.cuda(), "dense": A.to_dense().cuda(), "coo": A.to_sparse_coo().cuda()}[layout]
    d = data["d"].cuda()
    b = data["b"].cuda().requires_grad_(True)
    x, info = getattr(ma, kind)(Ad, b, M=lambda r: r / d, **entry["kwargs"])
    assert _last()["route"] == "generic" and info == entry["info"]
    assert x.grad_fn is not None
    (x ** 2).sum().backward()
    assert b.grad is not None and torch.isfinite(b.grad).all()
    assert rel_diff(x, data["x"]) <= 1e-9          # scaled systems (cond ~1e6 before preconditioning)
    assert rel_diff(b.grad, data["grad_b"]) <= 1e-8
    # the built-in Jacobi object takes the native route and must give the same gradient
    b2 = data["b"].cuda().requires_grad_(True)
    x2, info2 = getattr(ma, kind)(Ad, b2, M=ma.JacobiPreconditioner(Ad), **entry["kwargs"])
    assert _last()["route"] == "native" and info2 == entry["info"]
    (x2 ** 2).sum().backward()
    assert rel_diff(b2.grad, data["grad_b"]) <= 1e-8


def test_autograd_ldc100_gmres_config4_full_size(ma, manifest):
    """BASELINE configs[3] at the LDC default size (nx = 100, ldc_solver_common.py:35): GMRES(30), tol 1e-10, with the
    implicit-diff backward; x and b.grad against the reference (run with COO A, pinned by oracle/pin_round2.py)."""
    entry = manifest["round2"]["autograd_gmres_ldc100"]
    data = load_case("autograd_gmres_ldc100")
    A = build_matrix(entry["gen"], device="cuda")
    b = data["b"].cuda().requires_grad_(True)
    x, info = ma.gmres(A, b, **entry["kwargs"])
    assert info == entry["info"]
    (x ** 2).sum().backward()
    assert rel_diff(x, data["x"]) <= 5e-10
    assert rel_diff(b.grad, data["grad_b"]) <= 1e-8
    # the LDC time loop: same A, many right-hand sides — the registration (and its transpose) is cached
    from pytorch_sparse_solver import _native
    m1 = _native.register_matrix(A)
    for scale in (1.0, 0.5, 2.0):
        xs, _ = ma.gmres(A, scale * data["b"].cuda(), **entry["kwargs"])
        assert _native.register_matrix(A) is m1
    assert rel_diff(xs, 2.0 * data["x"]) <= 1e-9


def test_cache_detects_in_place_value_update(ma):
    """ADVICE r1 (high): updating `vals` in place and re-solving must not hit a stale registration (pattern / pair
    dictionaries, tails, cached transpose are value dependent) — torch's version counter cannot be relied on."""
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import _native, problems
    A0 = problems.poisson3d_csr(10)
    crow, col = A0.crow_indices().cuda(), A0.col_indices().cuda()
    vals = A0.values().clone().cuda()
    A = torch.sparse_csr_tensor(crow, col, vals, size=A0.shape)
    b = torch.ones(A0.shape[0], dtype=torch.float64, device="cuda")
    x1, _ = ma.cg(A, b, tol=1e-10)
    m1 = _native.register_matrix(A)
    assert _native.register_matrix(A) is m1                       # unchanged content: cache hit
    v0 = A.values()._version
    vals.mul_(2.0)                                                # the user's handle, not A.values()
    assert A.values()._version == v0, "torch does not bump the wrapper's version: the cache must not rely on it"
    x2, info2 = ma.cg(A, b, tol=1e-10)
    assert _native.register_matrix(A) is not m1, "same storage, new content: must be re-registered"
    assert info2 == 0 and rel_diff(x2, 0.5 * x1) <= 1e-12       # (2A) x = b  =>  x = x1 / 2, same Krylov iterates
    x_ref, info_ref, _ = orc.cg(torch.sparse_csr_tensor(A0.crow_indices(), A0.col_indices(), vals.cpu(), size=A0.shape),
                                b.cpu(), tol=1e-10)
    assert info_ref == 0 and rel_diff(x2, x_ref) <= FP64_TOL
    vals[::7] *= 1.5                                              # now non-symmetric: check the SpMV and its transpose
    A_cpu = torch.sparse_csr_tensor(A0.crow_indices(), A0.col_indices(), vals.cpu(), size=A0.shape)
    xv = torch.randn(A0.shape[0], dtype=torch.float64, device="cuda")
    m3 = _native.register_matrix(A)
    assert rel_diff(m3.spmv(xv), torch.matmul(A_cpu, xv.cpu())) <= 1e-14
    assert rel_diff(m3.transpose().spmv(xv), torch.matmul(A_cpu.to_dense().T, xv.cpu())) <= 1e-14
    # a re-wrapped tensor over the same (mutated again) storages
    vals.mul_(0.5)
    A2 = torch.sparse_csr_tensor(crow, col, vals, size=A0.shape)
    A2_cpu = torch.sparse_csr_tensor(A0.crow_indices(), A0.col_indices(), vals.cpu(), size=A0.shape)
    assert rel_diff(_native.register_matrix(A2).spmv(xv), torch.matmul(A2_cpu, xv.cpu())) <= 1e-14
    # dense input mutated through .data
    D = A0.to_dense().cuda()
    y1 = _native.register_matrix(D).spmv(xv)
    D.data[0, 0] = 60.0
    y2 = _native.register_matrix(D).spmv(xv)
    assert float((y2 - y1)[0]) == pytest.approx(54.0 * float(xv[0]), rel=1e-12)
    # explicit API + orphan pruning
    _native.invalidate(A)
    assert _native._key_and_parts(A, torch.float64)[0] not in _native._CACHE
    for k in range(4):
        T = problems.poisson2d_csr(9 + k, 8).cuda()
        _native.register_matrix(T)
        del T
    import gc
    gc.collect()
    _native.register_matrix(problems.poisson2d_csr(5, 5).cuda())
    orphans = [e for e in _native._CACHE.values() if e["src"]() is None]
    assert len(orphans) <= _native._CACHE_MAX_ORPHANS + 1


def test_result_reports_loop_mode_and_device_time(ma, manifest):
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    entry, data, x, info = _solve_case(ma, "cg_p3d16_rand", manifest)
    r = _last()
    assert r["loop_mode_used"] == 3 and r["device_ms"] > 0.0          # small system: persistent cooperative kernel
    try:
        h.set_option("persistent", 0)
        entry, data, x, info = _solve_case(ma, "cg_p3d16_rand", manifest)
        assert _last()["loop_mode_used"] == 2
        h.set_option("loop_mode", 1)
        entry, data, x, info = _solve_case(ma, "cg_p3d16_rand", manifest)
        assert _last()["loop_mode_used"] == 1
        h.set_option("nvtx", 1)                                       # ranges are no-ops outside a profiler
        entry, data, x2, info = _solve_case(ma, "cg_p3d16_rand", manifest)
        assert torch.equal(x, x2)
    finally:
        h.set_option("persistent", 1)
        h.set_option("loop_mode", 0)
        h.set_option("nvtx", 0)
    for name in ("bicgstab_cd3d16_rand", "gmres_cd3d12_batched"):
        _solve_case(ma, name, manifest)
        assert _last()["loop_mode_used"] in (2, 3) and _last()["device_ms"] > 0.0


@pytest.mark.parametrize("loop_mode", [0, 1])
def test_cg_lagged_x_cut_bitwise(loop_mode):
    """Large systems update x every second iteration with both pending terms (bk_op_cg_p_lag / bk_op_cg_xp_lag): the
    same additions in the same order, so x must be bit-identical to the plain 3-kernel cut — whatever the parity of the
    iteration the loop stops in (maxiter 1..7: odd counts end with the flush of K3e, even counts inside K3o), with and
    without x0, through graphs and plain launches."""
    from pytorch_sparse_solver import _native, problems
    dev = torch.device("cuda")
    h = _native.Handle.get(dev)
    A = problems.poisson3d_csr(24, device=dev)
    m = _native.register_matrix(A)
    g = torch.Generator().manual_seed(5)
    b = torch.randn(A.shape[0], dtype=torch.float64, generator=g).to(dev)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=g).to(dev)
    try:
        h.set_option("persistent", 0)
        h.set_option("fuse_xpay", 0)
        h.set_option("loop_mode", loop_mode)
        for maxiter in (1, 2, 3, 4, 5, 6, 7, 40, 41, None):
            for start in (None, x0):
                out = {}
                for lag in (0, 1):
                    h.set_option("cg_lag_x", lag)
                    x, res = m.cg(b, start, 1e-9, 0.0, maxiter)
                    out[lag] = (x.clone(), res["iterations"], res["info"], res["final_residual"])
                assert out[0][1] == out[1][1] and out[0][2] == out[1][2]
                assert out[0][3] == out[1][3]
                assert torch.equal(out[0][0], out[1][0]), (maxiter, start is not None)
    finally:
        h.set_option("persistent", 1)
        h.set_option("fuse_xpay", -1)
        h.set_option("loop_mode", 0)
        h.set_option("cg_lag_x", 1)


@pytest.mark.parametrize("name", ["gmres_ldc100_step1_batched", "gmres_ldc32_step1_incremental", "gmres_cd3d12_x0",
                                  "gmres_scd3d12_jacobi_incremental", "gmres_cd3d12_batched_2cycles", "gmres_zero_rhs"])
def test_gmres_persistent_kernel_vs_multi_kernel(ma, manifest, name):
    """Launch-bound systems run the whole GMRES solve in ONE cooperative kernel (bk_gmres_persist.cuh); it must agree
    with the graph-launched multi-kernel path to rounding (sums are reduced over a different partition), take the same
    number of cycles and matvecs, and be bitwise reproducible."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    entry, data, xp, infop = _solve_case(ma, name, manifest)
    rp = dict(_last())
    assert rp["loop_mode_used"] == 3 or rp["iterations"] == 0
    _e, _d, xp2, _i = _solve_case(ma, name, manifest)
    assert torch.equal(xp, xp2)
    try:
        h.set_option("persistent", 0)
        _e, _d, xm, infom = _solve_case(ma, name, manifest)
        rm = dict(_last())
    finally:
        h.set_option("persistent", 1)
    assert rm["loop_mode_used"] == 2
    assert infop == infom == entry["info"]
    assert rp["iterations"] == rm["iterations"] == entry["iterations"]
    assert abs(rp["matvecs"] - rm["matvecs"]) <= 1
    if float(torch.linalg.norm(xm)) > 0:
        assert rel_diff(xp, xm) <= (1e-9 if "ldc" in name else 1e-11)
    else:
        assert float(xp.abs().max()) == 0.0


@pytest.mark.parametrize("name", ["bicgstab_cd3d16_rand", "bicgstab_cd3d16_x0", "bicgstab_cd3d16_fixed10",
                                  "bicgstab_cd3d16_fixed1", "bicgstab_zero_rhs", "bicgstab_cd3d64_rand_digest"])
def test_bicgstab_persistent_kernel_vs_multi_kernel(ma, manifest, name):
    """Launch-bound systems run the whole BiCGStab loop in ONE persistent kernel (bk_bicgstab_persist.cuh: a thread-block
    cluster with its hardware barrier up to 16384 rows, a cooperative grid above): same iteration counts and info as the
    graph-launched path, x to rounding, bitwise reproducible."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    entry, data, xp, infop = _solve_case(ma, name, manifest)
    rp = dict(_last())
    _check_against_golden(entry, data, xp, infop)
    if entry["n"] <= 200000:
        assert rp["loop_mode_used"] == 3 or rp["iterations"] == 0
    _e, _d, xp2, _i = _solve_case(ma, name, manifest)
    assert torch.equal(xp, xp2)
    try:
        h.set_option("persistent", 0)
        _e, _d, xm, infom = _solve_case(ma, name, manifest)
        rm = dict(_last())
        h.set_option("persistent", 1)
        h.set_option("persistent_cluster", 0)       # cooperative-grid variant
        _e, _d, xg, infog = _solve_case(ma, name, manifest)
        rg = dict(_last())
    finally:
        h.set_option("persistent", 1)
        h.set_option("persistent_cluster", 1)
    assert rm["loop_mode_used"] == 2
    assert infop == infom == infog == entry["info"]
    assert abs(rp["iterations"] - rm["iterations"]) <= 1 and rg["iterations"] == rp["iterations"]
    if float(torch.linalg.norm(xm)) > 0:
        assert rel_diff(xp, xm) <= 1e-10 and rel_diff(xg, xm) <= 1e-10
    else:
        assert float(xp.abs().max()) == 0.0


@pytest.mark.parametrize("name", ["complex_cg_herm48", "complex_bicgstab_gen48", "complex_gmres_gen48"])
@pytest.mark.parametrize("layout", ["dense", "csr"])
def test_complex_systems_vs_reference(ma, manifest, name, layout):
    """complex128 systems (reference :86-127, :1220) through the real-equivalent registration + bk_cdot / bk_caxpby;
    goldens: the unmodified reference on the same dense complex matrices."""
    entry = manifest["round2"][name]
    data = load_case(name)
    A = data["A"].cuda()
    if layout == "csr":
        A = A.to_sparse_csr()
    b = data["b"].cuda()
    x, info = getattr(ma, entry["kind"])(A, b, **entry["kwargs"])
    assert _last()["route"] == "complex" and info == entry["info"]
    assert x.dtype == torch.complex128 and x.is_cuda
    assert float(torch.linalg.norm(x.cpu() - data["x"]) / torch.linalg.norm(data["x"])) <= 1e-9
    Ad = data["A"].cuda()
    assert float(torch.linalg.norm(b - Ad @ x) / torch.linalg.norm(b)) <= 1e-9
    if entry["kind"] == "gmres":
        xi, infoi = ma.gmres(A, b, solve_method="incremental", **entry["kwargs"])
        assert infoi == 0 and float(torch.linalg.norm(xi - x) / torch.linalg.norm(x)) <= 1e-7
    # CPU tensors are staged through the device; the adjoint solve uses A^H
    xc, infoc = getattr(ma, entry["kind"])(data["A"], data["b"], **entry["kwargs"])
    assert not xc.is_cuda and infoc == 0 and float(torch.linalg.norm(xc - data["x"]) / torch.linalg.norm(data["x"])) <= 1e-9
    b1 = b.clone().requires_grad_(True)
    x1, _ = getattr(ma, entry["kind"])(A, b1, **entry["kwargs"])
    torch.view_as_real(x1).pow(2).sum().backward()
    g_exact = torch.linalg.solve(Ad.conj().T, 2 * x1.detach())
    assert float(torch.linalg.norm(b1.grad - g_exact) / torch.linalg.norm(g_exact)) <= 1e-7


@pytest.mark.parametrize("name", ["cg_blockjacobi_bs4", "bicgstab_blockjacobi_bs8", "gmres_blockjacobi_bs3"])
def test_block_jacobi_preconditioner(ma, manifest, name):
    """BlockJacobiPreconditioner (one library kernel per application) against the reference run with the equivalent
    torch.bmm lambda; same matvec counts within the +-2 iteration band, x to 1e-9 (badly scaled systems)."""
    from pytorch_sparse_solver import _native
    entry = manifest["round2"][name]
    data = load_case(name)
    A_cpu = build_matrix(entry["gen"])
    A = A_cpu.cuda()
    bs = entry["block_size"]
    M = ma.BlockJacobiPreconditioner(A, block_size=bs)
    # the kernel against a dense product
    r = torch.randn(A.shape[0], dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    Binv = ma.BlockJacobiPreconditioner.diagonal_block_inverses(A_cpu, bs)
    ref = torch.block_diag(*Binv)[:A.shape[0], :A.shape[0]] @ r.cpu()
    assert rel_diff(M(r), ref) <= 1e-14
    calls = {"n": 0}
    reg = _native.register_matrix(A)

    def Aop(v):
        calls["n"] += 1
        return reg.spmv(v)
    x, info = getattr(ma, entry["kind"])(Aop, data["b"].cuda(), M=M, **entry["kwargs"])
    assert info == entry["info"] and _last()["route"] == "generic"
    per_it = 2 if entry["kind"] == "bicgstab" else 1
    assert abs(calls["n"] - entry["matvecs_ref"]) <= 2 * per_it + (30 if entry["kind"] == "gmres" else 0)
    assert rel_diff(x, data["x"]) <= 1e-9
    # tensor A: the implicit-diff backward re-uses M on A^T
    b1 = data["b"].cuda().requires_grad_(True)
    x1, _ = getattr(ma, entry["kind"])(A, b1, M=M, **entry["kwargs"])
    (x1 ** 2).sum().backward()
    Ad = A_cpu.to_dense()
    g_exact = torch.linalg.solve(Ad.T, 2.0 * torch.linalg.solve(Ad, data["b"]))
    assert rel_diff(b1.grad, g_exact) <= 1e-5      # badly scaled systems: the analytic gradient is itself ill-conditioned


@pytest.mark.parametrize("method", ["cg", "bicgstab", "gmres"])
def test_mixed_precision_iterative_refinement(ma, manifest, method):
    """fp32 inner solves + fp64 residual (SURVEY 8f-4): the final fp64 x must meet the fp64 tolerance and agree with
    the reference's fp64 solution."""
    name = "cg_p3d64_ones_digest" if method == "cg" else "bicgstab_cd3d64_rand_digest"
    entry = manifest["cases"][name]
    data = load_case(name)
    A_cpu = build_matrix(entry["gen"])
    A = A_cpu.cuda()
    from pytorch_sparse_solver import problems
    b = (torch.ones(entry["n"], dtype=torch.float64) if method == "cg" else problems.manufactured_rhs(A_cpu, 0)[0]).cuda()
    x, info = ma.refined_solve(A, b, method=method, tol=1e-11, inner_tol=1e-4, restart=30)
    r = _last()
    assert info == 0 and x.dtype == torch.float64 and r["refinements"] >= 2
    assert r["final_residual"] <= 1e-11 * r["b_norm"] * 1.01
    idx = data["x_sample_idx"]
    assert rel_diff(x.cpu()[idx], data["x_sample"]) <= 1e-8      # the digests were solved to tol 1e-8 / 1e-10
    assert abs(float(torch.linalg.norm(x)) - entry["x_norm"]) <= 1e-8 * entry["x_norm"]


def test_gmres_restart_above_native_limit(ma, manifest):
    """The reference accepts any restart; above the native limit (256) the solve runs on the generic route."""
    entry = manifest["cases"]["gmres_cd3d12_batched"]
    data = load_case("gmres_cd3d12_batched")
    A = build_matrix(entry["gen"], device="cuda")
    x, info = ma.gmres(A, data["b"].cuda(), tol=1e-8, restart=300)
    assert info == 0 and _last()["route"] == "generic"
    assert rel_diff(x, data["x"]) <= 1e-7


def test_reference_api_on_dist_matrix_single_rank(ma, manifest):
    """module_a.cg / bicgstab / gmres accept a DistMatrix as A (SURVEY 8e: the API stays additive)."""
    from pytorch_sparse_solver import distributed as bkd
    entry = manifest["cases"]["cg_p3d16_rand"]
    data = load_case("cg_p3d16_rand")
    A = build_matrix(entry["gen"], device="cuda")
    D = bkd.DistMatrix(A.crow_indices(), A.col_indices(), A.values(), [0, A.shape[0]], 0, 1)
    x, info = ma.cg(D, data["b"].cuda(), tol=1e-10)
    assert info == 0 and _last()["route"] == "dist" and _last()["iterations"] == entry["iterations"]
    assert rel_diff(x, data["x"]) <= FP64_TOL
    xb, infob = ma.bicgstab(D, data["b"].cuda(), tol=1e-10)
    xg, infog = ma.gmres(D, data["b"].cuda(), tol=1e-10, restart=30)
    assert infob == 0 and infog == 0 and rel_diff(xb, data["x"]) <= 1e-8 and rel_diff(xg, data["x"]) <= 1e-8
    with pytest.raises(ValueError):
        ma.cg(D, data["b"].cuda()[:-1])
    D.close()


def test_dist_worker_world1_both_paths():
    """The multi-GPU parity worker with ONE rank (peer-memory and NCCL code paths, graph and stream loops), so the
    distributed kernels are exercised on a single-GPU box too."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    env = dict(os.environ)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=1", "--master-addr",
           "127.0.0.1", "--master-port", "29641", str(ROOT / "tests" / "dist_gpu_worker.py"), "12"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "dist worker OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# --------------------------------------------------------------------------------------------------
# generic route (callable A, preconditioner M, pytrees) and the row-partitioned path
# --------------------------------------------------------------------------------------------------
def test_generic_route_callable_and_preconditioner(ma, manifest):
    from pytorch_sparse_solver import _native
    entry = manifest["cases"]["cg_p3d16_rand"]
    data = load_case("cg_p3d16_rand")
    A = build_matrix(entry["gen"], device="cuda")
    m = _native.register_matrix(A)
    b = data["b"].cuda()
    x, info = ma.cg(lambda v: m.spmv(v), b, tol=1e-10)
    assert info == 0 and _last()["route"] == "generic" and _last()["iterations"] == entry["iterations"]
    assert rel_diff(x, data["x"]) <= FP64_TOL
    diag = torch.full_like(b, 6.0)
    xj, info = ma.cg(A, b, tol=1e-10, M=lambda r: r / diag)          # Jacobi preconditioner
    assert info == 0 and rel_diff(xj, data["x"]) <= 1e-9
    # pytree right-hand side with a callable operator
    half = b.numel() // 2

    def op(tree):
        y = m.spmv(torch.cat([tree["a"], tree["b"]]))
        return {"a": y[:half], "b": y[half:]}
    xt, info = ma.cg(op, {"a": b[:half], "b": b[half:]}, tol=1e-10)
    assert info == 0 and rel_diff(torch.cat([xt["a"], xt["b"]]), data["x"]) <= FP64_TOL
    for name, fn in (("bicgstab_cd3d16_rand", ma.bicgstab), ("gmres_cd3d12_incremental", ma.gmres),
                     ("gmres_cd3d12_batched", ma.gmres)):
        entry = manifest["cases"][name]
        data = load_case(name)
        mm = _native.register_matrix(build_matrix(entry["gen"], device="cuda"))
        xg, info = fn(lambda v, mm=mm: mm.spmv(v), data["b"].cuda(), **entry["kwargs"])
        assert info == entry["info"] and rel_diff(xg, data["x"]) <= FP64_TOL, name


def test_dist_single_rank(manifest):
    """world_size 1 through the bk_dist_* entries (NCCL communicator of one rank) equals the plain solver."""
    from pytorch_sparse_solver import _native
    from pytorch_sparse_solver import distributed as bkd
    entry = manifest["cases"]["cg_p3d16_rand"]
    data = load_case("cg_p3d16_rand")
    A = build_matrix(entry["gen"], device="cuda")
    D = bkd.DistMatrix(A.crow_indices(), A.col_indices(), A.values(), [0, A.shape[0]], 0, 1)
    x, res = D.cg(data["b"].cuda(), None, 1e-10, 0.0, None)
    assert res["info"] == 0 and res["iterations"] == entry["iterations"]
    assert rel_diff(x, data["x"]) <= FP64_TOL
    xv = torch.randn(A.shape[0], dtype=torch.float64, device="cuda")
    assert rel_diff(D.spmv(xv), _native.register_matrix(A).spmv(xv)) <= 1e-15
    D.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_dist_two_gpus():
    import subprocess
    import sys
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29631", str(ROOT / "tests" / "dist_gpu_worker.py"), "16"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "dist worker OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# --------------------------------------------------------------------------------------------------
# the reference's own test systems (dense inputs, tests/test_module_a.py) and edge cases, against the oracle run
# on the same seeded inputs
# --------------------------------------------------------------------------------------------------
def _oracle():
    from oracle import krylov_oracle as orc
    return orc


def _dense_cases():
    g = torch.Generator().manual_seed(42)
    n = 100
    tri = (2.0 * torch.eye(n, dtype=torch.float64) - torch.diag(torch.ones(n - 1, dtype=torch.float64), 1)
           - torch.diag(torch.ones(n - 1, dtype=torch.float64), -1))
    nonsym = tri + 0.1 * torch.randn(n, n, dtype=torch.float64, generator=g) + 5.0 * torch.eye(n, dtype=torch.float64)
    gen = torch.randn(n, n, dtype=torch.float64, generator=g) + 10.0 * torch.eye(n, dtype=torch.float64)
    B = torch.randn(50, 50, dtype=torch.float64, generator=g)
    spd = B @ B.T + 50.0 * torch.eye(50, dtype=torch.float64)
    tiny = torch.randn(6, 6, dtype=torch.float64, generator=g) + 4.0 * torch.eye(6, dtype=torch.float64)
    return {
        "bicgstab_nonsym100": ("bicgstab", nonsym, dict(tol=1e-10, maxiter=1000)),          # test_bicgstab_basic :126-161
        "gmres_general100": ("gmres", gen, dict(tol=1e-10, maxiter=1000, restart=30)),       # test_gmres_basic :163-195
        "gmres_spd50_batched": ("gmres", spd, dict(tol=1e-8, restart=30, solve_method="batched")),       # :273-315
        "gmres_spd50_incremental": ("gmres", spd, dict(tol=1e-8, restart=30, solve_method="incremental")),
        "gmres_tiny_restart_gt_n_batched": ("gmres", tiny, dict(tol=1e-10, restart=20, maxiter=5)),
        "gmres_tiny_restart_gt_n_incremental": ("gmres", tiny, dict(tol=1e-10, restart=20, maxiter=5,
                                                                     solve_method="incremental")),
        "cg_spd50": ("cg", spd, dict(tol=1e-10, maxiter=1000)),
        "cg_maxiter0": ("cg", spd, dict(tol=1e-10, maxiter=0)),
        "bicgstab_maxiter0": ("bicgstab", nonsym, dict(tol=1e-10, maxiter=0)),
        "gmres_maxiter0": ("gmres", gen, dict(tol=1e-10, maxiter=0, restart=5)),
    }


@pytest.mark.parametrize("name", sorted(_dense_cases().keys()))
def test_reference_dense_test_systems_vs_oracle(ma, name):
    kind, A, kw = _dense_cases()[name]
    g = torch.Generator().manual_seed(7)
    b = A @ torch.randn(A.shape[0], dtype=torch.float64, generator=g)
    x_ref, info_ref, st = getattr(_oracle(), kind)(A, b, None, **kw)
    x, info = getattr(ma, kind)(A.cuda(), b.cuda(), **kw)            # dense CUDA input, as the reference's tests pass it
    assert info == info_ref, (info, info_ref, st)
    if "tiny" in name:
        # Krylov space exhausted (restart > n): the breakdown decision `||w|| <= eps*||Av||` sits on rounding noise,
        # so only the solution is compared
        assert rel_diff(x, x_ref) <= 1e-9
    else:
        assert abs(_last()["iterations"] - st["iterations"]) <= 2
        assert rel_diff(x, x_ref) <= FP64_TOL if float(torch.linalg.norm(x_ref)) > 0 else float(torch.linalg.norm(x)) == 0.0


def test_zero_size_and_shape_errors(ma):
    A = build_matrix(dict(matrix="poisson2d", nx=5, ny=4), device="cuda")
    with pytest.raises(ValueError):
        ma.cg(A, torch.ones(19, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        ma.cg(A, torch.ones(20, dtype=torch.float64))            # device mismatch
    with pytest.raises(ValueError):
        ma.gmres(A, torch.ones(20, dtype=torch.float64, device="cuda"), restart=0)


def test_c_abi_argument_validation_on_gpu():
    import ctypes as C
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    lib = h.lib
    A = build_matrix(dict(matrix="poisson2d", nx=6, ny=5), device="cuda")
    crow, col, val = A.crow_indices().int(), A.col_indices().int(), A.values()
    out = C.c_void_p()
    s = torch.cuda.current_stream().cuda_stream
    assert lib.bk_csr_create(h.ptr, 30, val.numel(), crow.data_ptr(), col.data_ptr(), 16, val.data_ptr(), 0, 0, s, C.byref(out)) == -1
    assert lib.bk_csr_create(h.ptr, 30, val.numel(), crow.data_ptr(), col.data_ptr(), 32, val.data_ptr(), 7, 0, s, C.byref(out)) == -1
    bad = col.clone()
    bad[3] = 1000                                        # column out of range -> malformed CSR
    assert lib.bk_csr_create(h.ptr, 30, val.numel(), crow.data_ptr(), bad.data_ptr(), 32, val.data_ptr(), 0, 0, s, C.byref(out)) == -1
    assert b"malformed" in lib.bk_last_error()
    assert lib.bk_set_option(h.ptr, b"no_such_option", 1) == -1
    m = _native.register_matrix(A)
    res = _native.bk_result()
    b = torch.ones(30, dtype=torch.float64, device="cuda")
    x = torch.empty_like(b)
    assert lib.bk_gmres(h.ptr, m.ptr, b.data_ptr(), x.data_ptr(), 0, 1e-8, 0.0, 0, -1, 0, C.byref(res), s) == -4   # restart 0
    assert lib.bk_gmres(h.ptr, m.ptr, b.data_ptr(), x.data_ptr(), 0, 1e-8, 0.0, 1000, -1, 0, C.byref(res), s) == -4  # > 256
    assert lib.bk_gmres(h.ptr, m.ptr, b.data_ptr(), x.data_ptr(), 0, 1e-8, 0.0, 10, -1, 5, C.byref(res), s) == -1   # method
    assert lib.bk_spmv(h.ptr, m.ptr, b.data_ptr(), b.data_ptr(), s) == -1                                        # aliasing


# --------------------------------------------------------------------------------------------------
# built-in Jacobi preconditioner (SURVEY §8f-1): device PCG vs the reference run with M = lambda r: r / d
# --------------------------------------------------------------------------------------------------
def test_jacobi_pcg_routes_and_autograd(ma, manifest):
    """cg(M=JacobiPreconditioner) stays native; any other M and any other solver take the generic route with the
    same numbers; the adjoint solve reuses M (reference :1079-1084)."""
    from pytorch_sparse_solver import problems
    from pytorch_sparse_solver.module_a import krylov
    entry = manifest["cases"]["cg_sp3d12_jacobi"]
    data = load_case("cg_sp3d12_jacobi")
    A = build_matrix(entry["gen"], device="cuda")
    b = data["b"].cuda()
    M = ma.JacobiPreconditioner(A)
    d = problems.csr_diagonal(A)
    assert torch.equal(M.d, d), "bk_csr_diagonal"
    x, info = ma.cg(A, b, tol=1e-10, M=M)
    assert krylov.last_result["route"] == "native" and info == 0
    assert abs(krylov.last_result["iterations"] - entry["iterations"]) <= 2
    assert rel_diff(x, data["x"]) <= FP64_TOL
    xg, infog = ma.cg(A, b, tol=1e-10, M=lambda r: r / d)            # user lambda: generic route
    assert infog == 0 and rel_diff(xg, data["x"]) <= FP64_TOL
    xb, infob = ma.bicgstab(A, b, tol=1e-10, M=M)                    # BiCGStab has a device path for it too
    assert krylov.last_result["route"] == "native"
    assert infob == 0 and rel_diff(xb, data["x"]) <= 1e-5   # ill-conditioned system: x follows the residual loosely
    xg2, infog2 = ma.gmres(A, b, tol=1e-10, restart=30, M=M)         # and GMRES (left preconditioning)
    assert krylov.last_result["route"] == "native"
    assert infog2 == 0 and rel_diff(xg2, data["x"]) <= 1e-5
    xg3, infog3 = ma.gmres(A, b, tol=1e-10, restart=30, M=lambda r: r / d)   # user lambda: generic route, same answer
    assert infog3 == 0 and rel_diff(xg3, xg2) <= 1e-8
    # dense and COO inputs build the same preconditioner
    assert torch.equal(ma.JacobiPreconditioner(A.to_dense()).d, d)
    assert torch.equal(ma.JacobiPreconditioner(A.to_sparse_coo()).d, d)
    # gradient w.r.t. b through the preconditioned adjoint solve == A^-T (2 x)
    b1 = b.clone().requires_grad_(True)
    x1, _ = ma.cg(A, b1, tol=1e-12, M=M)
    (x1 ** 2).sum().backward()
    Ad = A.to_dense()
    g_exact = torch.linalg.solve(Ad.T, 2.0 * torch.linalg.solve(Ad, b))
    assert rel_diff(b1.grad, g_exact) <= 1e-8
    with pytest.raises(ValueError):
        ma.JacobiPreconditioner(torch.zeros(3, 3, device="cuda"))
    # through the router: SolverResult.residual stays the UNpreconditioned ||b - A x|| / ||b|| (solver.py:362-368)
    import pytorch_sparse_solver as pss
    xr, resr = pss.SparseSolver().solve(A, b, method='cg', backend='module_a', tol=1e-10, M=M)
    true_rel = float(torch.linalg.norm(b - torch.mv(Ad, xr)) / torch.linalg.norm(b))
    assert resr.converged and resr.iterations == krylov.last_result["iterations"]
    assert abs(resr.residual - true_rel) <= 1e-3 * true_rel + 1e-16


def test_jacobi_pcg_edge_cases(ma):
    from pytorch_sparse_solver.module_a import krylov
    A = build_matrix(dict(matrix="scaled_poisson3d", n=6), device="cuda")
    M = ma.JacobiPreconditioner(A)
    z = torch.zeros(A.shape[0], dtype=torch.float64, device="cuda")
    x, info = ma.cg(A, z, M=M)
    assert info == 0 and float(x.abs().max()) == 0.0 and krylov.last_result["iterations"] == 0
    b = torch.ones(A.shape[0], dtype=torch.float64, device="cuda")
    x5, info5 = ma.cg(A, b, tol=0.0, atol=0.0, maxiter=5, M=M)
    assert info5 == -1 and krylov.last_result["iterations"] == 5
    x5b, _ = ma.cg(A, b, tol=0.0, atol=0.0, maxiter=5, M=M)
    assert torch.equal(x5, x5b)
    # fp32 native path
    A32 = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values().float(), size=A.shape)
    x32, info32 = ma.cg(A32, b.float(), tol=1e-5, M=ma.JacobiPreconditioner(A32))
    x64, _ = ma.cg(A, b, tol=1e-10, M=M)
    assert info32 == 0 and x32.dtype == torch.float32 and rel_diff(x32, x64) <= 1e-4


# --------------------------------------------------------------------------------------------------
# dense / COO ingestion by the library's own kernels (SURVEY §8f-2) against torch's conversions
# --------------------------------------------------------------------------------------------------
def _csr_triplet(m):
    crow, col, val = m.arrays()
    return crow.cpu().long(), col.cpu().long(), val.cpu()


@pytest.mark.parametrize("n,density,dtype", [(1, 1.0, torch.float64), (37, 0.3, torch.float64), (300, 0.02, torch.float64),
                                              (257, 1.0, torch.float32), (1000, 0.004, torch.float64)])
def test_dense_ingestion_matches_torch(n, density, dtype):
    from pytorch_sparse_solver import _native
    g = torch.Generator().manual_seed(n)
    D = torch.randn(n, n, dtype=dtype, generator=g)
    D[torch.rand(n, n, generator=g) > density] = 0.0
    if n > 30:
        D[5, :] = 0.0                                   # an empty row
    ref = D.to_sparse_csr()
    _native.clear_cache()
    m = _native.register_matrix(D.cuda(), dtype)
    crow, col, val = _csr_triplet(m)
    assert torch.equal(crow, ref.crow_indices()) and torch.equal(col, ref.col_indices())
    assert torch.equal(val, ref.values())
    # a non-contiguous view (transposed) and an fp32 matrix registered as fp64
    mt = _native.register_matrix(D.cuda().t(), torch.float64)
    rt = D.t().contiguous().double().to_sparse_csr()
    crow, col, val = _csr_triplet(mt)
    assert torch.equal(crow, rt.crow_indices()) and torch.equal(col, rt.col_indices()) and torch.equal(val, rt.values())
    x = torch.randn(n, dtype=dtype, generator=g)
    assert rel_diff(m.spmv(x.cuda()), D.double() @ x.double()) <= (1e-13 if dtype == torch.float64 else 1e-5)


@pytest.mark.parametrize("n,nnz,dups", [(1, 1, False), (50, 400, True), (3000, 20000, True), (70000, 300000, False)])
def test_coo_ingestion_matches_torch(n, nnz, dups):
    from pytorch_sparse_solver import _native
    g = torch.Generator().manual_seed(nnz)
    rows = torch.randint(0, n, (nnz,), generator=g)
    cols = torch.randint(0, n, (nnz,), generator=g)
    if dups:                                            # force repeated positions, some cancelling exactly
        rows[nnz // 2:] = rows[:nnz - nnz // 2]
        cols[nnz // 2:] = cols[:nnz - nnz // 2]
    vals = torch.randn(nnz, dtype=torch.float64, generator=g)
    if dups:
        vals[nnz // 2] = -vals[0]
    C = torch.sparse_coo_tensor(torch.stack([rows, cols]), vals, (n, n))
    ref = C.coalesce().to_sparse_csr()
    _native.clear_cache()
    m = _native.register_matrix(C.cuda())
    crow, col, val = _csr_triplet(m)
    assert torch.equal(crow, ref.crow_indices()) and torch.equal(col, ref.col_indices())
    assert rel_diff(val, ref.values()) <= 1e-15 and m.nnz == ref.values().numel()
    x = torch.randn(n, dtype=torch.float64, generator=g)
    assert rel_diff(m.spmv(x.cuda()), torch.sparse.mm(C.coalesce(), x[:, None])[:, 0]) <= 1e-12
    # bad index -> error, not a crash
    badC = torch.sparse_coo_tensor(torch.tensor([[0], [0]]), torch.ones(1, dtype=torch.float64), (1, 1)).cuda()
    bad_idx = badC._indices().clone()
    h = _native.Handle.get(torch.device("cuda"))
    p = _native._VP()
    bad_idx[0, 0] = (1 << 32)            # would alias index 0 if it were narrowed to int32 before the check
    rc = h.lib.bk_csr_from_coo(h.ptr, 1, 1, bad_idx[0].contiguous().data_ptr(), bad_idx[1].contiguous().data_ptr(), 64,
                               badC._values().data_ptr(), _native.BK_F64, _native.BK_F64, None, _native.C.byref(p))
    assert rc == -1


def _banded_coded_matrix(n, offsets, drop, seed, dtype=torch.float64, per_offset_values=1):
    """n x n matrix with entries at (r, r + o) for o in `offsets`, each kept with probability 1 - drop; the value of
    an entry depends only on its offset (and r % per_offset_values), so a block holds few distinct (offset, value)
    pairs although the row lengths vary wildly."""
    g = torch.Generator().manual_seed(seed)
    offs = torch.tensor(sorted(offsets))
    base = torch.randn(len(offs), per_offset_values, dtype=torch.float64, generator=g)
    r = torch.arange(n)[:, None]
    c = r + offs[None, :]
    keep = (c >= 0) & (c < n) & (torch.rand(n, len(offs), generator=g) >= drop)
    keep[n // 3] = False                                          # an empty row
    v = base[torch.arange(len(offs))[None, :].expand(n, -1), (r % per_offset_values).expand(-1, len(offs))]
    rows = r.expand(-1, len(offs))[keep]
    A = torch.sparse_coo_tensor(torch.stack([rows, c[keep]]), v[keep].to(dtype), (n, n)).coalesce().to_sparse_csr()
    return A


@pytest.mark.parametrize("n,offsets,drop,pov,expect5", [
    (1000, [-37, -1, 0, 1, 37], 0.0, 1, True),
    (777, [-300, -64, -5, -1, 0, 1, 2, 9, 64, 300], 0.4, 1, True),        # ragged rows, n % 32 != 0
    (4099, list(range(-9, 10)), 0.5, 1, True),                            # up to 19 entries: several 8-entry batches
    (2050, list(range(-15, 16)), 0.2, 1, True),                           # 31 pairs: the limit
    (2050, list(range(-16, 16)), 0.2, 1, False),                          # 32 pairs: falls back
    (1500, [-40, -1, 0, 1, 40], 0.1, 6, True),                            # 30 pairs from 5 offsets x 6 values
    (1500, [-40, -1, 0, 1, 40], 0.1, 7, False),                           # 35 pairs: falls back
    (31, [0, 1], 0.0, 1, True),
])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_pair_coded_spmv_stress(n, offsets, drop, pov, expect5, dtype):
    """Kernel 5 on adversarial 'few distinct pairs' matrices: bit-identical to the plain CSR kernel, every fused variant
    (dots, residual form), and the fall-back when a block exceeds 31 pairs."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    A = _banded_coded_matrix(n, offsets, drop, seed=n + len(offsets), dtype=dtype, per_offset_values=pov).cuda()
    g = torch.Generator("cuda").manual_seed(3)
    x = torch.randn(n, dtype=dtype, device="cuda", generator=g)
    w = torch.randn(n, dtype=dtype, device="cuda", generator=g)
    try:
        h.set_option("use_compress", 0)
        _native.clear_cache()
        m2 = _native.register_matrix(A, dtype)
        y2, d2 = m2.spmv_dot(x, w)
        k2 = m2.info()["kernel"]
        h.set_option("use_compress", 2)
        _native.clear_cache()
        m5 = _native.register_matrix(A, dtype)
        y5, d5 = m5.spmv_dot(x, w)
        k5 = m5.info()["kernel"]
        y5b = m5.spmv(x)
        h.set_option("use_compress", 3)
        _native.clear_cache()
        m6 = _native.register_matrix(A, dtype)
        y6, d6 = m6.spmv_dot(x, w)
        k6 = m6.info()["kernel"]
        h.set_option("mask_window", 1)           # gathers from TMA-staged shared-memory windows instead of LDG: same bits
        y6l, d6l = m6.spmv_dot(x, w)
        h.set_option("mask_wgroup", 2)
        h.set_option("tma_stages", 2)
        y6w, d6w = m6.spmv_dot(x, w)
    finally:
        h.set_option("use_compress", 3)
        h.set_option("mask_window", 0)
        h.set_option("mask_wgroup", 4)
        h.set_option("tma_stages", 0)
        _native.clear_cache()
    assert torch.equal(y6, y6l) and torch.equal(y6, y6w)
    assert abs(float(d6) - float(d6l)) <= 1e-12 * float(w.abs() @ y6.abs() + 1e-300)
    assert k2 in (0, 2)
    if k2 == 2:
        assert (k5 == 5) == expect5, (k5, expect5)
    assert torch.equal(y2, y5) and torch.equal(y5, y5b) and float(d2) == float(d5)
    # kernel 6 needs <= 8 entries per row and <= 8 pairs per 32-row chunk; whatever was selected must agree bit for bit
    if max(len(offsets), 1) * pov <= 8:
        assert k6 == 6, k6
    assert torch.equal(y2, y6) and abs(float(d2) - float(d6)) <= 1e-12 * float(w.abs() @ y2.abs() + 1e-300)
    ref = torch.matmul(A.cpu().to_dense().double(), x.cpu().double())
    assert rel_diff(y5, ref) <= (1e-13 if dtype == torch.float64 else 2e-5)


@pytest.mark.parametrize("kind", ["poisson3d", "convdiff3d"])
def test_full_size_spmv_all_stagings_bitwise(kind):
    """BASELINE's full size (256^3, 117 M entries): the stencil fast path (kernel 7), the row-bitmask stream (6), the
    pair-coded stream (5), the coded-column stream (3) and the TMA-staged CSR stream (2) must produce the same bits; the
    LDG-staged kernel (0) agrees to rounding."""
    from pytorch_sparse_solver import _native
    h = _native.Handle.get(torch.device("cuda"))
    A = build_matrix(dict(matrix=kind, n=256), device="cuda")
    N = A.shape[0]
    g = torch.Generator("cuda").manual_seed(11)
    x = torch.randn(N, dtype=torch.float64, device="cuda", generator=g)
    w = torch.randn(N, dtype=torch.float64, device="cuda", generator=g)
    outs = {}
    saved = {k: h.get_option(k) for k in ("use_tma", "use_compress", "mask_const")}
    try:
        for label, opts, want in (("k7", dict(use_tma=1, use_compress=3, mask_const=1), 7),
                                  ("k6", dict(use_tma=1, use_compress=3, mask_const=0), 6),
                                  ("k5", dict(use_tma=1, use_compress=2), 5), ("k3", dict(use_tma=1, use_compress=1), 3),
                                  ("k2", dict(use_tma=1, use_compress=0), 2), ("k0", dict(use_tma=0, use_compress=0), 0)):
            for k, v in opts.items():
                h.set_option(k, v)
            _native.clear_cache()
            m = _native.register_matrix(A)
            assert m.info()["kernel"] == want, (label, m.info()["kernel"])
            y, d = m.spmv_dot(x, w)
            outs[label] = (y.clone(), float(d))
            del m
    finally:
        for k, v in saved.items():
            h.set_option(k, v)
        _native.clear_cache()
    for label in ("k7", "k6", "k3", "k2"):
        assert torch.equal(outs["k5"][0], outs[label][0]), label
    # kernel 0 parks rounded products in shared memory and adds them (mul + add), the TMA kernels use fma chains
    assert rel_diff(outs["k0"][0], outs["k5"][0]) <= 1e-15
    # the dot is reduced over a kernel-specific grid, so it may differ in the last bits between stagings
    scale = float(w.abs() @ outs["k5"][0].abs())
    for label in ("k7", "k6", "k3", "k2", "k0"):
        assert abs(outs["k5"][1] - outs[label][1]) <= 1e-13 * scale, (label, outs["k5"][1], outs[label][1])
    # a size-independent property: row sums of the Poisson matrix are 0 away from the boundary => A * ones is
    # non-zero only on boundary rows; for both matrices A*(2x) == 2*(A x) exactly (scaling by 2 is exact)
    _native.clear_cache()
    m = _native.register_matrix(A)
    assert torch.equal(m.spmv(2.0 * x), 2.0 * outs["k5"][0])


def test_bench_dump_outputs_match_oracle(tmp_path):
    """`bench.py --dump-outputs` writes the solution of the timed call (module_a.cg on the GPU), the same bits from run to
    run, and it agrees with the oracle's solve of the same system; --steps sets the number of timed solves."""
    import json
    import subprocess
    import sys
    import numpy as np
    from conftest import ROOT
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import problems

    def run(out, steps):
        cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--n", "32", "--steps", str(steps), "--warmup", "1",
               "--no-e2e", "--no-cpu", "--no-extra", "--dump-outputs", str(out)]
        p = subprocess.run(cmd, cwd=str(ROOT), capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-4000:]
        (line,) = [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")]
        assert line["steps"] == steps and line["details"]["info"] == 0
        return line, {f.stem: np.load(f) for f in sorted(out.iterdir())}

    line2, a = run(tmp_path / "a", 2)
    line4, b = run(tmp_path / "b", 4)
    its = line2["details"]["iterations_per_solve"]
    assert line4["details"]["iterations_per_solve"] == its
    assert abs(line2["ms_per_step"] * 2 * line2["value"] * 1e-3 - 2 * its) <= 1e-6 * its
    assert abs(line4["ms_per_step"] * 4 * line4["value"] * 1e-3 - 4 * its) <= 1e-6 * its
    assert sorted(a) == ["info", "x"] and all(v.dtype == np.float64 for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)
    A = problems.poisson3d_csr(32)
    x_ref, info_ref, _ = orc.cg(A, torch.ones(A.shape[0], dtype=torch.float64), tol=1e-8)
    assert float(a["info"]) == info_ref == 0
    assert rel_diff(torch.from_numpy(a["x"]), x_ref) <= FP64_TOL
