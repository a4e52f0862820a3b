"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol the header declares,
argument validation mirrors the reference's exceptions, tolerance helpers mirror the reference's roundings,
pytree helpers, problem generators.  No compute call is made (there is no GPU here)."""
import re

import pytest
import torch

from conftest import ROOT


def test_library_exports_every_header_symbol():
    from pytorch_sparse_solver import _native
    header = (ROOT / "include" / "bk_krylov.h").read_text()
    declared = set(re.findall(r"^\s*(?:int|int64_t|const char\*)\s+(bk_[a-z0-9_]+)\s*\(", header, flags=re.M))
    assert len(declared) >= 25
    lib = _native.load_library()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/bk_krylov.h but not exported"
    assert declared == set(_native._SIGNATURES), "ctypes signature table out of sync with the header"
    assert lib.bk_version() == 200


def test_library_result_struct_layout():
    from pytorch_sparse_solver import _native
    import ctypes
    assert ctypes.sizeof(_native.bk_result) == 8 + 8 + 8 + 4 + 4 + 5 * 8 + 4 + 4 + 8
    assert ctypes.sizeof(_native.bk_csr_info) == 8 + 8 + 4 * 4 + 8 + 8 + 8


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_cuda():
    from pytorch_sparse_solver import _native, module_a
    A = torch.eye(4, dtype=torch.float64).to_sparse_csr()
    b = torch.ones(4, dtype=torch.float64)
    with pytest.raises(_native.NativeLibraryError):
        module_a.cg(A, b)
    with pytest.raises(_native.NativeLibraryError):
        module_a.gmres(A, b)


def test_argument_validation_matches_reference():
    from pytorch_sparse_solver import module_a
    b = torch.ones(4, dtype=torch.float64)
    with pytest.raises(ValueError, match="square"):
        module_a.cg(torch.ones(4, 3, dtype=torch.float64), b)
    with pytest.raises(TypeError):
        module_a.cg("not a matrix", b)
    with pytest.raises(ValueError, match="matching shapes"):
        module_a.bicgstab(torch.eye(4, dtype=torch.float64), b, torch.ones(3, dtype=torch.float64))
    with pytest.raises(ValueError, match="Unsupported solve_method"):
        module_a.gmres(torch.eye(4, dtype=torch.float64), b, solve_method="qr")
    with pytest.raises(ValueError, match="2D tensor"):
        module_a.cg_differentiable(lambda v: v, b)


def test_gmres_tolerance_mirror():
    """_gmres_effective_tolerances must reproduce the reference's atol_tensor / ptol (oracle copy of :733-753)."""
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver.module_a import krylov
    import warnings
    for dev in ("cpu", "cuda"):
        for tol, atol, n, bn in ((1e-10, 0.0, 10_000, 7071.07), (1e-5, 1e-3, 100, 3.0), (1e-14, 0.0, 16_777_216, 4096.0),
                                 (1e-8, 0.0, 1024, 0.0)):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                a_ref, p_ref = orc.gmres_tolerances(tol, atol, n, torch.tensor(bn, dtype=torch.float64), dev)
            t_eff, a_eff = krylov._gmres_effective_tolerances(tol, atol, n, dev)
            a = max(t_eff * bn, a_eff)
            assert a == float(a_ref)
            if bn > 0:
                assert bn * min(1.0, a / bn) == float(p_ref)


def test_fp32_tolerance_rounding_constants():
    """bk_state_fill_tol reproduces torch.tensor(tol) (fp32) and torch.square on it (reference :816)."""
    import numpy as np
    t = np.float32(1e-8)
    assert float(t) == float(torch.tensor(1e-8))
    assert float(t * t) == float(torch.square(torch.tensor(1e-8)))


def test_tree_utils():
    from pytorch_sparse_solver.module_a import tree_flatten, tree_leaves, tree_map, tree_unflatten, Partial
    from pytorch_sparse_solver.module_a.torch_tree_util import tree_reduce, tree_structure
    t = {"b": [torch.ones(2), (torch.zeros(1), None)], "a": torch.full((3,), 2.0)}
    leaves, td = tree_flatten(t)
    assert [tuple(x.shape) for x in leaves] == [(3,), (2,), (1,)]
    back = tree_unflatten(td, leaves)
    assert isinstance(back["b"][1], tuple) and back["b"][1][1] is None
    doubled = tree_map(lambda x: 2 * x, t)
    assert float(doubled["a"][0]) == 4.0
    summed = tree_map(lambda x, y: x + y, t, doubled)
    assert float(summed["a"][0]) == 6.0
    assert float(tree_reduce(lambda a, c: a + c.sum(), t, 0.0)) == 8.0
    assert tree_structure(t) == tree_structure(doubled)
    with pytest.raises(ValueError):
        tree_map(lambda x, y: x, t, [1, 2])
    assert Partial(lambda a, b, c=0: a + b + c, 1, c=3)(2) == 6
    assert len(tree_leaves(None)) == 0


def test_generators_match_reference_conventions():
    import pytorch_sparse_solver as pss
    from pytorch_sparse_solver import problems
    A = problems.poisson2d_csr(7, 5)
    B = pss.create_poisson_2d_sparse_coo(7, 5).to_sparse_csr()
    assert torch.equal(A.crow_indices(), B.crow_indices()) and torch.equal(A.col_indices(), B.col_indices())
    assert torch.equal(A.values(), B.values())
    T = pss.create_tridiagonal_sparse_coo(6).to_dense()
    assert torch.equal(T, 2 * torch.eye(6, dtype=torch.float64) - torch.diag(torch.ones(5, dtype=torch.float64), 1)
                       - torch.diag(torch.ones(5, dtype=torch.float64), -1))
    P = problems.poisson3d_csr(5)
    D = P.to_dense()
    assert torch.equal(D, D.T) and P.values().numel() == 7 * 125 - 6 * 25
    C = problems.convdiff3d_csr(4).to_dense()
    assert not torch.equal(C, C.T) and float(C.sum(1).min()) >= 0.0        # M-matrix row sums >= 0
    L = problems.ldc_pressure_csr(6).to_dense()
    assert torch.equal(L, L.T) and float(L.sum(1).abs().max()) == 0.0       # all-Neumann: singular
    assert problems.cg_bytes_per_iteration(16_777_216, 117_047_296) == 2_948_071_428
    assert problems.bicgstab_bytes_per_iteration(16_777_216, 117_047_296) == 5_493_489_672
    slab = problems.stencil3d_csr(4, nz=2)
    assert slab.shape[0] == 32


def test_router_errors_and_availability():
    import pytorch_sparse_solver as pss
    have = torch.cuda.is_available()   # module_a IS the CUDA library: no device -> not available (no CPU fallback)
    assert pss.get_available_backends() == {"module_a": have, "module_b": False, "module_c": False}
    s = pss.SparseSolver()
    A = torch.eye(3, dtype=torch.float64)
    b = torch.ones(3, dtype=torch.float64)
    if not have:
        assert s.available_backends == []
        with pytest.raises(RuntimeError, match="No sparse solver backends"):
            s.solve(A, b)
        return
    assert s.available_backends == ["module_a"]
    with pytest.raises(ValueError, match="not available"):
        s.solve(A, b, backend="module_c")
    with pytest.raises(ValueError):
        s.solve(A, b, method="direct")
    with pytest.raises(ValueError):
        pss.amg(A, b)
    assert "module_a" in repr(s)


def test_c_abi_error_paths_without_gpu():
    """Argument validation of the C ABI: negative bk_error codes + a message, never a crash.  (No compute call.)"""
    import ctypes as C
    from pytorch_sparse_solver import _native
    lib = _native.load_library()
    h = C.c_void_p()
    rc = lib.bk_create(0, None)
    assert rc == -1 and b"out is null" in lib.bk_last_error()
    if not torch.cuda.is_available():
        rc = lib.bk_create(0, C.byref(h))
        assert rc < 0 and h.value is None and len(lib.bk_last_error()) > 0
    assert lib.bk_set_option(None, b"chunk", 4) == -1
    assert lib.bk_get_option(None, b"chunk") == -1
    out = C.c_void_p()
    assert lib.bk_csr_create(None, 4, 4, None, None, 32, None, 0, 0, None, C.byref(out)) == -1
    assert lib.bk_spmv(None, None, None, None, None) == -1
    res = _native.bk_result()
    assert lib.bk_cg(None, None, None, None, 0, 1e-5, 0.0, -1, C.byref(res), None) == -1
    assert lib.bk_gmres(None, None, None, None, 0, 1e-5, 0.0, 20, -1, 0, C.byref(res), None) == -1
    assert lib.bk_solve_host(None, 0, 4, 4, None, None, 32, None, 0, None, None, 0, 1e-5, 0.0, -1, 20, 0, C.byref(res)) == -1
    assert lib.bk_dist_p2p_export(None, None) == -1
    assert lib.bk_csr_destroy(None) == 0 and lib.bk_destroy(None) == 0 and lib.bk_dist_destroy(None) == 0


def test_matrix_wrapper_exposes_every_solver_entry():
    """krylov.py reaches the C solvers through these CsrMatrix methods: a missing one would only show up on a GPU."""
    from pytorch_sparse_solver import _native
    for name in ("spmv", "spmv_dot", "cg", "bicgstab", "gmres", "cg_jacobi", "bicgstab_jacobi", "gmres_jacobi",
                 "diagonal", "transpose", "arrays", "grad_pattern", "info"):
        assert callable(getattr(_native.CsrMatrix, name, None)), name
    for sym in ("bk_cg", "bk_bicgstab", "bk_gmres", "bk_cg_jacobi", "bk_bicgstab_jacobi", "bk_gmres_jacobi",
                "bk_csr_from_dense", "bk_csr_from_coo", "bk_dist_cg", "bk_dist_bicgstab", "bk_dist_gmres"):
        assert sym in _native._SIGNATURES, sym


def test_problem_generators_scaled_systems():
    """The badly scaled fixtures: same sparsity as their parents, S A S values, symmetric iff the parent is."""
    from pytorch_sparse_solver import problems
    P = problems.poisson3d_csr(5)
    S = problems.scaled_poisson3d_csr(5)
    C = problems.scaled_convdiff3d_csr(5)
    assert torch.equal(P.crow_indices(), S.crow_indices()) and torch.equal(P.col_indices(), S.col_indices())
    Sd, Cd = S.to_dense(), C.to_dense()
    assert torch.allclose(Sd, Sd.T, rtol=0, atol=0), "S A S of a symmetric A is symmetric bit for bit"
    assert not torch.allclose(Cd, Cd.T)
    assert torch.equal(problems.csr_diagonal(S), torch.diagonal(Sd))
    assert torch.equal(problems.csr_diagonal(C), torch.diagonal(Cd))
    assert float(torch.linalg.eigvalsh(Sd).min()) > 0.0, "still positive definite"
    d = torch.diagonal(Sd)
    assert float(d.max() / d.min()) > 100.0, "strongly varying diagonal (what Jacobi is for)"


def test_oracle_preconditioned_solvers_agree_with_dense_solve():
    """Oracle with M = r / d (the form pinned against the reference) on a small badly scaled system."""
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import problems
    A = problems.scaled_convdiff3d_csr(5)
    d = problems.csr_diagonal(A)
    xt = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    b = torch.mv(A.to_dense(), xt)
    M = lambda r: r / d  # noqa: E731
    for kind, kw in (("bicgstab", dict(tol=1e-12)), ("gmres", dict(tol=1e-12, restart=20))):
        x, info, st = getattr(orc, kind)(A, b, None, M=M, **kw)
        x0, info0, st0 = getattr(orc, kind)(A, b, None, **kw)
        assert info == 0 and float(torch.linalg.norm(x - xt) / torch.linalg.norm(xt)) <= 1e-8
        assert st["matvecs"] < st0["matvecs"], (kind, st["matvecs"], st0["matvecs"])
    S = problems.scaled_poisson3d_csr(5)
    ds = problems.csr_diagonal(S)
    bs = torch.mv(S.to_dense(), xt)
    x, info, st = orc.cg(S, bs, None, tol=1e-12, M=lambda r: r / ds)
    x0, info0, st0 = orc.cg(S, bs, None, tol=1e-12)
    assert info == 0 and st["iterations"] < st0["iterations"]
    assert float(torch.linalg.norm(x - xt) / torch.linalg.norm(xt)) <= 1e-8


def test_bench_reference_arm_contract_on_cpu():
    """`bench.py --impl reference` (the oracle port timed on the host cores) runs without a GPU; its JSON line carries the
    keys the driver reads, at N = 1 and under a torchrun-style environment with N > 1 (rank 0 prints, the others exit 0
    without work), with the SAME workload string this repo's arm prints for that N."""
    import json
    import os
    import subprocess
    import sys

    def run(extra_env, gpus):
        env = dict(os.environ, **extra_env)
        cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", str(gpus), "--n", "12", "--steps", "1",
               "--warmup", "1", "--ref-window", "5"]
        p = subprocess.run(cmd, env=env, cwd=str(ROOT), capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-2000:]
        return [json.loads(line) for line in p.stdout.splitlines() if line.startswith("{")]

    (line,) = run({}, 1)
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "cg_iterations_per_second" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert "12^3" in line["config"]["workload"]
    (line2,) = run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, 2)
    assert line2["n_gpus"] == 2 and "row-partitioned over 2 GPUs" in line2["config"]["workload"]
    assert run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, 2) == []


def test_bench_dump_outputs_reference_arm(tmp_path):
    """`--dump-outputs DIR` writes the last timed step's (x, info) as float64 arrays; the same arguments give the same
    files, and x is what the timed call computes."""
    import json
    import subprocess
    import sys
    import numpy as np
    from oracle import krylov_oracle as orc
    from pytorch_sparse_solver import problems

    def run(out, steps):
        cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--n", "10", "--steps", str(steps),
               "--warmup", "1", "--ref-window", "7", "--dump-outputs", str(out)]
        p = subprocess.run(cmd, cwd=str(ROOT), capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-2000:]
        (line,) = [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")]
        assert line["steps"] == steps
        return {f.stem: np.load(f) for f in sorted(out.iterdir())}

    a, b = run(tmp_path / "a", 2), run(tmp_path / "b", 3)
    assert sorted(a) == ["info", "x"] and all(v.dtype == np.float64 for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)
    A = problems.poisson3d_csr(10)
    x, info, _ = orc.cg(A, torch.ones(A.shape[0], dtype=torch.float64), tol=0.0, atol=0.0, maxiter=7)
    assert np.array_equal(a["x"], x.numpy()) and float(a["info"]) == info


def test_bench_dump_outputs_sample(tmp_path, monkeypatch):
    """An x larger than DUMP_MAX_ENTRIES is stored as a fixed sample of rows plus the sampled row indices."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_ENTRIES", 100)
    x = torch.randn(1000, dtype=torch.float64)
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(a, x, 0)
    bench.dump_outputs(b, x, 0)
    idx, xs = np.load(a / "x_index.npy"), np.load(a / "x.npy")
    assert idx.dtype == xs.dtype == np.float64 and idx.shape == xs.shape == (100,)
    assert np.all(np.diff(idx) > 0) and np.array_equal(xs, x.numpy()[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(b / "x_index.npy"))
    bench.dump_outputs(a, x[:50].float(), 1)
    assert sorted(f.name for f in a.iterdir()) == ["info.npy", "x.npy"]
    assert np.load(a / "x.npy").dtype == np.float64 and float(np.load(a / "info.npy")) == 1.0
