"""Multicolor symmetric Gauss-Seidel preconditioner (bk_sgs_*, module_a.SymmetricGaussSeidelPreconditioner).

`restate_coloring` and `restate_sgs` are numpy restatements of the library's definition:
  neighbours  j != i with (i, j) or (j, i) stored (explicit zeros count)
  priority    (fmix32(i) << 32) | i
  rounds      Jones-Plassmann on a snapshot: an uncolored row whose priority exceeds that of every uncolored neighbour
              takes the smallest color no neighbour colored in an earlier round holds
  apply       z = 0, forward sweep over colors 0..C-1, backward over C-2..0, z_i = (r_i - sum_{j!=i} a_ij z_j) / a_ii
The CPU tests pin the restatement (valid coloring, color bound, closed form B = (D+U)^-1 D (D+L)^-1 in color order,
SPD for SPD A); the GPU tests hold the device to it and run the three preconditioned solvers against the oracle.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import rel_diff
from pytorch_sparse_solver import problems
from test_stencil_plans import stencil_grid


# ---- restatement ------------------------------------------------------------------------------------------------
def _csr(A):
    A = A.to_sparse_csr() if A.layout != torch.sparse_csr else A
    crow = A.crow_indices().cpu().numpy().astype(np.int64)
    col = A.col_indices().cpu().numpy().astype(np.int64)
    val = A.values().cpu().double().numpy()
    return sp.csr_matrix((val, col, crow), shape=A.shape)


def fmix32(i):
    h = np.asarray(i, dtype=np.uint64) & np.uint64(0xFFFFFFFF)
    m = np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85EBCA6B)) & m
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xC2B2AE35)) & m
    h ^= h >> np.uint64(16)
    return h


def prio(i):
    i = np.asarray(i, dtype=np.uint64)
    return (fmix32(i) << np.uint64(32)) | i


def restate_coloring(S):
    """(colors uint8[n], rounds) of the csr_matrix S's pattern."""
    n = S.shape[0]
    rows = np.repeat(np.arange(n), np.diff(S.indptr))
    I = np.concatenate([rows, S.indices])
    J = np.concatenate([S.indices, rows])
    keep = I != J
    I, J = I[keep], J[keep]
    pr = prio(np.arange(n))
    color = np.full(n, -1, dtype=np.int64)
    rounds = 0
    while (color < 0).any():
        unc = color < 0
        e = unc[I] & unc[J]
        beaten = np.zeros(n, dtype=bool)
        beaten[I[e][pr[J[e]] > pr[I[e]]]] = True
        sel = unc & ~beaten
        used = np.zeros((n, 257), dtype=bool)
        e = sel[I] & (color[J] >= 0)
        used[I[e], color[J[e]]] = True
        c = np.argmin(used, axis=1)
        color[sel] = c[sel]
        rounds += 1
    assert color.max() < 255
    return color.astype(np.uint8), rounds


def restate_sgs(S, colors, r):
    """z = M r in float64 (rows of one color in CSR order, one at a time)."""
    d = S.diagonal()
    off = sp.csr_matrix((S.data * (S.indices != np.repeat(np.arange(S.shape[0]), np.diff(S.indptr))),
                         S.indices, S.indptr), shape=S.shape)
    r = np.asarray(r, dtype=np.float64)
    z = np.zeros_like(r)
    C = int(colors.max()) + 1
    lists = [np.nonzero(colors == c)[0] for c in range(C)]
    for c in list(range(C)) + list(range(C - 2, -1, -1)):
        rows = lists[c]
        z[rows] = (r[rows] - off[rows] @ z) / d[rows]
    return z


def closed_form(S, colors):
    """B = P^T (D+U)^-1 D (D+L)^-1 P with P the stable sort of the rows by color."""
    perm = np.argsort(colors, kind="stable")
    Ap = S[perm][:, perm].toarray()
    D = np.diag(np.diag(Ap))
    L, U = np.tril(Ap, -1), np.triu(Ap, 1)
    n = Ap.shape[0]
    Bp = np.linalg.solve(D + U, D @ np.linalg.solve(D + L, np.eye(n)))
    B = np.empty_like(Bp)
    B[np.ix_(perm, perm)] = Bp
    return B


def random_nonsym(n=300, seed=3):
    rng = np.random.default_rng(seed)
    M = sp.random(n, n, density=0.02, random_state=rng, format="csr")
    M = M + sp.diags(4.0 + rng.random(n))
    M.sort_indices()
    return torch.sparse_csr_tensor(torch.from_numpy(M.indptr.astype(np.int64)), torch.from_numpy(M.indices.astype(np.int64)),
                                   torch.from_numpy(M.data), size=M.shape)


def holes_grid():
    return stencil_grid((24, 20, 18), holes=0.1, seed=5)


SMALL = {
    "p3d8": lambda: problems.poisson3d_csr(8),
    "p2d12x10": lambda: problems.poisson2d_csr(12, 10),
    "ldc16": lambda: problems.ldc_pressure_csr(16),
    "nonsym300": random_nonsym,
}


def _max_degree(S):
    G = sp.csr_matrix((np.ones_like(S.indices), S.indices, S.indptr), shape=S.shape)
    G = ((G + G.T) > 0).astype(np.int8)
    G.setdiag(0)
    G.eliminate_zeros()
    return int(np.diff(G.indptr).max())


# ---- CPU: the restatement ---------------------------------------------------------------------------------------
def test_fmix32_known_values():
    # murmur3's finalizer: fmix32(0) = 0, fmix32(1) = 0x514e28b7
    assert int(fmix32(0)) == 0 and int(fmix32(1)) == 0x514E28B7
    assert int(prio(1)) == (0x514E28B7 << 32) | 1


@pytest.mark.parametrize("name", sorted(SMALL))
def test_coloring_is_valid_and_bounded(name):
    S = _csr(SMALL[name]())
    colors, rounds = restate_coloring(S)
    coo = S.tocoo()
    off = coo.row != coo.col
    assert not np.any(colors[coo.row[off]] == colors[coo.col[off]])
    assert int(colors.max()) + 1 <= _max_degree(S) + 1
    assert rounds >= int(colors.max()) + 1


def test_p3d32_uses_six_colors():
    colors, _ = restate_coloring(_csr(problems.poisson3d_csr(32)))
    assert int(colors.max()) + 1 == 6


@pytest.mark.parametrize("name", sorted(SMALL))
def test_application_equals_closed_form(name):
    S = _csr(SMALL[name]())
    colors, _ = restate_coloring(S)
    B = closed_form(S, colors)
    r = np.random.default_rng(1).standard_normal(S.shape[0])
    z = restate_sgs(S, colors, r)
    ref = B @ r
    assert np.linalg.norm(z - ref) <= 1e-13 * np.linalg.norm(ref)


@pytest.mark.parametrize("name", ["p3d8", "p2d12x10"])
def test_symmetric_matrix_gives_spd_preconditioner(name):
    S = _csr(SMALL[name]())
    colors, _ = restate_coloring(S)
    B = closed_form(S, colors)
    assert np.abs(B - B.T).max() <= 1e-13 * np.abs(B).max()
    assert np.linalg.eigvalsh(0.5 * (B + B.T)).min() > 0


def test_preconditioner_rejects_cpu_complex_and_dist():
    from pytorch_sparse_solver import _native
    from pytorch_sparse_solver.module_a import SymmetricGaussSeidelPreconditioner as SGS
    A = problems.poisson2d_csr(4, 4)
    with pytest.raises(ValueError):
        SGS(torch.complex(A.to_dense(), A.to_dense()))
    with pytest.raises(ValueError):
        SGS(type("DistMatrix", (), {"n_global": 4})())
    with pytest.raises(_native.NativeLibraryError):
        SGS(A)


def test_exported():
    from pytorch_sparse_solver import module_a
    assert "SymmetricGaussSeidelPreconditioner" in module_a.__all__


# ---- GPU ----------------------------------------------------------------------------------------------------------
GPU_COLORING = {
    "p3d32": lambda: problems.poisson3d_csr(32),
    "ldc32": lambda: problems.ldc_pressure_csr(32),
    "ldc100": lambda: problems.ldc_pressure_csr(100),
    "cd3d16": lambda: problems.convdiff3d_csr(16),
    "holes": holes_grid,
    "nonsym300": random_nonsym,
    "p3d12_int32": lambda: problems.poisson3d_csr(12, index_dtype=torch.int32),
    "p3d12_int64": lambda: problems.poisson3d_csr(12, index_dtype=torch.int64),
}


def _sgs_of(A, dtype=torch.float64):
    from pytorch_sparse_solver.module_a import SymmetricGaussSeidelPreconditioner
    M = SymmetricGaussSeidelPreconditioner(A)
    return M, M.sgs(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GPU_COLORING))
def test_device_coloring_equals_restatement(name):
    from pytorch_sparse_solver import _native
    A = GPU_COLORING[name]()
    colors, rounds = restate_coloring(_csr(A))
    M, S = _sgs_of(A.cuda())
    got = S.colors().cpu().numpy()
    assert np.array_equal(got, colors)
    assert (S.num_colors, S.rounds) == (int(colors.max()) + 1, rounds)
    # a second creation (a fresh registration) gives the same bytes
    _native.clear_cache()
    M2, S2 = _sgs_of(A.cuda())
    assert S2 is not S and torch.equal(S2.colors().cpu(), torch.from_numpy(colors))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-12), (torch.float32, 1e-5)])
@pytest.mark.parametrize("name", ["p3d32", "ldc32", "nonsym300", "holes"])
def test_device_application_matches_restatement(name, dtype, tol):
    A = GPU_COLORING[name]().to(dtype)
    Sc = _csr(A)
    colors, _ = restate_coloring(Sc)
    r = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    M, S = _sgs_of(A.cuda(), dtype)
    z = S.apply(r.to(dtype).cuda())
    ref = restate_sgs(Sc, colors, r.to(dtype).double().numpy())
    assert rel_diff(z, torch.from_numpy(ref)) <= tol
    assert torch.equal(z, S.apply(r.to(dtype).cuda()))
    assert torch.equal(M(r.to(dtype).cuda()), z)


@pytest.mark.gpu
def test_in_place_value_scaling_is_picked_up():
    A = problems.poisson3d_csr(16).cuda()
    M, S = _sgs_of(A)
    r = torch.randn(A.shape[0], dtype=torch.float64, device="cuda")
    z = M(r)
    A.values().mul_(2.0)
    z2 = M(r)
    assert torch.equal(z2, z / 2)


@pytest.mark.gpu
def test_missing_or_zero_diagonal_raises():
    from pytorch_sparse_solver.module_a import SymmetricGaussSeidelPreconditioner as SGS
    A = problems.poisson2d_csr(6, 5)
    dense = A.to_dense()
    dense[7, 7] = 0.0                                    # missing diagonal entry
    with pytest.raises(ValueError, match="row 7"):
        SGS(dense.to_sparse_csr().cuda())
    vals = A.values().clone()
    crow, col = A.crow_indices(), A.col_indices()
    rows = torch.repeat_interleave(torch.arange(30), crow.diff())
    vals[(rows == 11) & (col == 11)] = 0.0               # stored explicit zero on the diagonal
    with pytest.raises(ValueError, match="row 11"):
        SGS(torch.sparse_csr_tensor(crow, col, vals, size=A.shape).cuda())


def _oracle_M(A, dtype=torch.float64):
    Sc = _csr(A)
    colors, _ = restate_coloring(Sc)
    return lambda r: torch.from_numpy(restate_sgs(Sc, colors, r.double().cpu().numpy()))


SOLVES = [
    ("cg", "p3d32", lambda: problems.poisson3d_csr(32), dict(tol=1e-8), False, torch.float64),
    ("cg", "p3d32_x0", lambda: problems.poisson3d_csr(32), dict(tol=1e-8), True, torch.float64),
    ("cg", "sp3d12", lambda: problems.scaled_poisson3d_csr(12), dict(tol=1e-8), False, torch.float64),
    ("cg", "sp3d12_x0", lambda: problems.scaled_poisson3d_csr(12), dict(tol=1e-8), True, torch.float64),
    ("cg", "p3d32_fp32", lambda: problems.poisson3d_csr(32), dict(tol=1e-5), False, torch.float32),
    ("bicgstab", "cd3d16", lambda: problems.convdiff3d_csr(16), dict(tol=1e-8), False, torch.float64),
    ("gmres", "ldc32_batched", lambda: problems.ldc_pressure_csr(32),
     dict(tol=1e-10, restart=30, solve_method="batched"), False, torch.float64),
    ("gmres", "ldc32_incremental", lambda: problems.ldc_pressure_csr(32),
     dict(tol=1e-10, restart=30, solve_method="incremental"), False, torch.float64),
]


@pytest.fixture
def cpu_gmres_tolerances():
    from pytorch_sparse_solver.module_a import krylov
    saved = krylov.GMRES_TOLERANCE_DEVICE
    krylov.GMRES_TOLERANCE_DEVICE = "cpu"
    yield
    krylov.GMRES_TOLERANCE_DEVICE = saved


@pytest.mark.gpu
@pytest.mark.parametrize("solver,name,make,kw,with_x0,dtype", SOLVES, ids=[s[1] for s in SOLVES])
def test_solves_match_oracle(solver, name, make, kw, with_x0, dtype, cpu_gmres_tolerances):
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import module_a
    A = make()
    n = A.shape[0]
    b = A.to(torch.float64) @ torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    x0 = 0.1 * torch.ones(n, dtype=torch.float64) if with_x0 else None
    Ag = A.to(dtype).cuda()
    M = module_a.SymmetricGaussSeidelPreconditioner(Ag)
    res = {}
    x, info = getattr(module_a, solver)(Ag, b.to(dtype).cuda(), None if x0 is None else x0.to(dtype).cuda(), M=M,
                                        _result=res, **kw)
    xo, info_o, stats = getattr(orc, solver)(A.to(torch.float64), b, x0, M=_oracle_M(A.to(dtype)), **kw)
    assert info == info_o
    assert rel_diff(x, xo) <= (1e-10 if dtype == torch.float64 else 1e-4)
    if dtype == torch.float64:
        assert abs(res["iterations"] - stats["iterations"]) <= 2
    assert res["route"] == "native"


@pytest.mark.gpu
def test_loop_modes_runs_and_jacobi_comparison():
    from pytorch_sparse_solver import _native, module_a
    A = problems.poisson3d_csr(32).cuda()
    b = A @ torch.randn(A.shape[0], dtype=torch.float64, device="cuda")
    M = module_a.SymmetricGaussSeidelPreconditioner(A)
    h = _native.Handle.get(A.device)
    saved = h.get_option("loop_mode")
    xs = []
    try:
        for mode in (2, 1):   # CUDA graph of chunks, plain stream launches
            h.set_option("loop_mode", mode)
            res = {}
            x, info = module_a.cg(A, b, tol=1e-8, M=M, _result=res)
            assert info == 0 and res["loop_mode_used"] == mode
            xs.append(x)
    finally:
        h.set_option("loop_mode", saved)
    assert torch.equal(xs[0], xs[1])
    runs = [module_a.cg(A, b, tol=1e-8, M=M)[0] for _ in range(3)]
    assert all(torch.equal(runs[0], x) for x in runs)
    rs, rj = {}, {}
    module_a.cg(A, b, tol=1e-8, M=M, _result=rs)
    module_a.cg(A, b, tol=1e-8, M=module_a.JacobiPreconditioner(A), _result=rj)
    assert rs["iterations"] < rj["iterations"]


@pytest.mark.gpu
@pytest.mark.parametrize("solver,kw", [("cg", dict(tol=1e-8)), ("bicgstab", dict(tol=1e-8)),
                                       ("gmres", dict(tol=1e-10, restart=30))])
def test_generic_route_agrees_with_native(solver, kw):
    from pytorch_sparse_solver import module_a
    A = (problems.poisson3d_csr(12) if solver == "cg" else problems.convdiff3d_csr(12)).cuda()
    b = A @ torch.randn(A.shape[0], dtype=torch.float64, device="cuda")
    M = module_a.SymmetricGaussSeidelPreconditioner(A)
    fn = getattr(module_a, solver)
    x_native, info_n = fn(A, b, M=M, **kw)
    x_generic, info_g = fn(lambda v: A @ v, b, M=M, **kw)
    assert info_n == info_g == 0
    assert rel_diff(x_generic, x_native) <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("solver,make,kw", [
    ("cg", lambda: problems.poisson3d_csr(12), dict(tol=1e-10)),
    ("gmres", lambda: problems.convdiff3d_csr(12), dict(tol=1e-10, restart=30)),
])
def test_gradient_matches_oracle_adjoint(solver, make, kw, cpu_gmres_tolerances):
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import module_a
    A = make()
    n = A.shape[0]
    b = (A @ torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(0))).cuda()
    b.requires_grad_(True)
    w = torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(4))
    Ag = A.cuda()
    M = module_a.SymmetricGaussSeidelPreconditioner(Ag)
    x, info = getattr(module_a, solver)(Ag, b, M=M, **kw)
    (x * w.cuda()).sum().backward()
    g_ref = orc.adjoint_grad_b(solver, A, w, None, M=_oracle_M(A), **kw)
    assert rel_diff(b.grad, g_ref) <= 1e-9
