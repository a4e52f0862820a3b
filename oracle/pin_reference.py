#!/usr/bin/env python3
"""Pin the oracle to the UNMODIFIED reference and write the golden fixtures (tests/golden/).

Run in the build container only (needs /root/reference):   python oracle/pin_reference.py

For every case it runs
  (1) the reference  (sys.path -> /root/reference/src, pytorch_sparse_solver.module_a.{cg,bicgstab,gmres}, CPU)
      with A wrapped in a counting callable to obtain matvec counts (bit-identical results, SURVEY.md §0), and
  (2) oracle/krylov_oracle.py on the same tensors,
requires torch.equal(x_ref, x_oracle), equal info and equal matvec counts, and stores inputs + reference outputs
as small .npz files plus a manifest.  The reference has no golden vectors of its own (SURVEY.md §4), so these
fixtures ARE the pin: tests/test_oracle_golden.py re-checks the oracle against them on every machine, and the
GPU parity tests compare the CUDA path against the same vectors.
"""
import importlib
import json
import os
import sys
import time
import warnings
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"
REF_SRC = "/root/reference/src"
PKG_DIR = ROOT / "pytorch-sparse-linalg-torch-amgx.cg.bicg.gmres_b200"

warnings.filterwarnings("ignore")


def load_reference():
    """Import the reference package under its own name, then detach it so ours can be imported too."""
    sys.path.insert(0, REF_SRC)
    for k in list(sys.modules):
        if k.startswith("pytorch_sparse_solver"):
            del sys.modules[k]
    ref = importlib.import_module("pytorch_sparse_solver.module_a")
    ref_mods = {k: v for k, v in sys.modules.items() if k.startswith("pytorch_sparse_solver")}
    for k in ref_mods:
        del sys.modules[k]
    sys.path.remove(REF_SRC)
    return ref, ref_mods


def main():
    torch.set_num_threads(os.cpu_count())
    ref, ref_mods = load_reference()
    sys.path.insert(0, str(PKG_DIR))
    sys.path.insert(0, str(ROOT))
    from pytorch_sparse_solver import problems           # our generators (product code; no solver involved)
    from oracle import krylov_oracle as orc
    GOLD.mkdir(parents=True, exist_ok=True)
    manifest = {"torch": torch.__version__, "torch_threads": torch.get_num_threads(),
                "generated": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), "cases": {}}

    def run_ref(kind, A, b, x0=None, **kw):
        calls = {"n": 0}

        def Aop(v):
            calls["n"] += 1
            return torch.matmul(A, v)
        fn = getattr(ref, kind)
        x, info = fn(Aop, b, x0=x0, **kw)
        # same call with the tensor itself must be bit-identical (and is what users do)
        x2, info2 = fn(A, b, x0=x0, **kw)
        assert torch.equal(x, x2) and info == info2, "reference: callable vs tensor differ"
        return x, int(info), calls["n"]

    def run_orc(kind, A, b, x0=None, **kw):
        x, info, stats = getattr(orc, kind)(A, b, x0, **kw)
        return x, info, stats

    def pin(name, kind, A, b, x0=None, store_vectors=True, gen=None, jacobi=False, **kw):
        t0 = time.time()
        if jacobi:  # M = diag(A)^-1 written the way users of the reference write it
            d = problems.csr_diagonal(A)
            kw_run = dict(kw, M=lambda r: r / d)
        else:
            kw_run = kw
        xr, inf_r, mv_r = run_ref(kind, A, b, x0, **kw_run)
        xo, inf_o, st = run_orc(kind, A, b, x0, **kw_run)
        # reference matvecs include its final residual check (1), ours are counted before it
        assert torch.equal(xr, xo), f"{name}: oracle x differs from reference (max {float((xr - xo).abs().max()):.3e})"
        assert inf_r == inf_o, f"{name}: info {inf_r} vs {inf_o}"
        assert mv_r == st["matvecs"] + 1, f"{name}: matvecs {mv_r} vs {st['matvecs']}+1"
        entry = dict(kind=kind, n=int(b.numel()), info=inf_r, matvecs_ref=mv_r, iterations=st["iterations"],
                     final_residual=st["final_residual"], b_norm=st["b_norm"], gen=gen or {},
                     kwargs={k: v for k, v in kw.items()}, jacobi=bool(jacobi), x_norm=float(torch.linalg.norm(xr)),
                     x_sum=float(xr.sum()), seconds=round(time.time() - t0, 2))
        arrays = {}
        if store_vectors:
            arrays["x"] = xr.numpy()
            arrays["b"] = b.numpy()
            if x0 is not None:
                arrays["x0"] = x0.numpy()
        else:
            idx = torch.linspace(0, b.numel() - 1, 512).long()
            arrays["x_sample_idx"] = idx.numpy()
            arrays["x_sample"] = xr[idx].numpy()
        np.savez_compressed(GOLD / f"{name}.npz", **arrays)
        manifest["cases"][name] = entry
        print(f"  pinned {name}: iters={st['iterations']} matvecs={mv_r} info={inf_r} ({entry['seconds']} s)")
        return xr

    g = torch.Generator().manual_seed(1)

    # ---- CG --------------------------------------------------------------------------------------
    A = problems.poisson2d_csr(32, 32)
    ones = torch.ones(A.shape[0], dtype=torch.float64)
    pin("cg_p2d32_ones", "cg", A, ones, gen=dict(matrix="poisson2d", nx=32, ny=32), tol=1e-8)
    A = problems.poisson3d_csr(16)
    b, _ = problems.manufactured_rhs(A, 0)
    pin("cg_p3d16_rand", "cg", A, b, gen=dict(matrix="poisson3d", n=16), tol=1e-10)
    pin("cg_p3d16_fixed10", "cg", A, b, gen=dict(matrix="poisson3d", n=16), tol=0.0, atol=0.0, maxiter=10)
    pin("cg_p3d16_fixed1", "cg", A, b, gen=dict(matrix="poisson3d", n=16), tol=0.0, atol=0.0, maxiter=1)
    A = problems.poisson2d_csr(24, 20)
    b, _ = problems.manufactured_rhs(A, 3)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=g)
    pin("cg_p2d24x20_x0", "cg", A, b, x0, gen=dict(matrix="poisson2d", nx=24, ny=20), tol=1e-9, atol=1e-12)
    pin("cg_p2d24x20_maxiter5", "cg", A, b, gen=dict(matrix="poisson2d", nx=24, ny=20), tol=1e-12, maxiter=5)
    z = torch.zeros(A.shape[0], dtype=torch.float64)
    pin("cg_zero_rhs", "cg", A, z, gen=dict(matrix="poisson2d", nx=24, ny=20), tol=1e-8)
    # the reference's own test matrix: dense tridiag(2,-1), n=100 (test_module_a.py:93-124), fed as CSR here
    n = 100
    Ad = (2.0 * torch.eye(n, dtype=torch.float64) - torch.diag(torch.ones(n - 1, dtype=torch.float64), 1)
          - torch.diag(torch.ones(n - 1, dtype=torch.float64), -1))
    bt = Ad @ torch.randn(n, dtype=torch.float64, generator=g)
    xd, infd, _ = run_ref("cg", Ad, bt, tol=1e-10, maxiter=1000)
    xs = pin("cg_tridiag100", "cg", Ad.to_sparse_csr(), bt, gen=dict(matrix="tridiag", n=100), tol=1e-10, maxiter=1000)
    manifest["cases"]["cg_tridiag100"]["dense_vs_csr_maxdiff"] = float((xd - xs).abs().max())
    # digests at larger sizes (x too big to ship: 512 samples + norms)
    A = problems.poisson2d_csr(256, 256)
    pin("cg_p2d256_ones_digest", "cg", A, torch.ones(A.shape[0], dtype=torch.float64), store_vectors=False,
        gen=dict(matrix="poisson2d", nx=256, ny=256), tol=1e-8)
    A = problems.poisson3d_csr(64)
    pin("cg_p3d64_ones_digest", "cg", A, torch.ones(A.shape[0], dtype=torch.float64), store_vectors=False,
        gen=dict(matrix="poisson3d", n=64), tol=1e-8)

    # Jacobi-preconditioned CG (M = lambda r: r / diag(A)) on a badly scaled SPD system
    A = problems.scaled_poisson3d_csr(12)
    b, _ = problems.manufactured_rhs(A, 2)
    gsp = dict(matrix="scaled_poisson3d", n=12, seed=7)
    # (without M this system needs 8747 iterations at tol 1e-10; with Jacobi 53)
    pin("cg_sp3d12_jacobi", "cg", A, b, gen=gsp, jacobi=True, tol=1e-10)
    pin("cg_sp3d12_jacobi_fixed7", "cg", A, b, gen=gsp, jacobi=True, tol=0.0, atol=0.0, maxiter=7)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(11))
    pin("cg_sp3d12_jacobi_x0", "cg", A, b, x0, gen=gsp, jacobi=True, tol=1e-9, atol=1e-14)
    pin("cg_p3d16_jacobi", "cg", problems.poisson3d_csr(16), problems.manufactured_rhs(problems.poisson3d_csr(16), 0)[0],
        gen=dict(matrix="poisson3d", n=16), jacobi=True, tol=1e-10)

    # ---- BiCGStab --------------------------------------------------------------------------------
    A = problems.convdiff3d_csr(16)
    b, _ = problems.manufactured_rhs(A, 0)
    pin("bicgstab_cd3d16_rand", "bicgstab", A, b, gen=dict(matrix="convdiff3d", n=16), tol=1e-10)
    pin("bicgstab_cd3d16_fixed10", "bicgstab", A, b, gen=dict(matrix="convdiff3d", n=16), tol=0.0, atol=0.0, maxiter=10)
    pin("bicgstab_cd3d16_fixed1", "bicgstab", A, b, gen=dict(matrix="convdiff3d", n=16), tol=0.0, atol=0.0, maxiter=1)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=g)
    pin("bicgstab_cd3d16_x0", "bicgstab", A, b, x0, gen=dict(matrix="convdiff3d", n=16), tol=1e-10)
    pin("bicgstab_zero_rhs", "bicgstab", A, torch.zeros(A.shape[0], dtype=torch.float64),
        gen=dict(matrix="convdiff3d", n=16), tol=1e-8)
    A = problems.convdiff3d_csr(64)
    b, _ = problems.manufactured_rhs(A, 0)
    pin("bicgstab_cd3d64_rand_digest", "bicgstab", A, b, store_vectors=False, gen=dict(matrix="convdiff3d", n=64),
        tol=1e-10)

    # Jacobi-preconditioned BiCGStab on a badly scaled non-symmetric system (S A S, A = upwind convection-diffusion)
    A = problems.scaled_convdiff3d_csr(12)
    b, _ = problems.manufactured_rhs(A, 4)
    gsc = dict(matrix="scaled_convdiff3d", n=12, seed=7)
    pin("bicgstab_scd3d12_jacobi", "bicgstab", A, b, gen=gsc, jacobi=True, tol=1e-10)
    pin("bicgstab_scd3d12_jacobi_fixed5", "bicgstab", A, b, gen=gsc, jacobi=True, tol=0.0, atol=0.0, maxiter=5)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(12))
    pin("bicgstab_scd3d12_jacobi_x0", "bicgstab", A, b, x0, gen=gsc, jacobi=True, tol=1e-9)

    # ---- GMRES -----------------------------------------------------------------------------------
    A = problems.convdiff3d_csr(12)
    b, _ = problems.manufactured_rhs(A, 0)
    for sm in ("batched", "incremental"):
        pin(f"gmres_cd3d12_{sm}", "gmres", A, b, gen=dict(matrix="convdiff3d", n=12), tol=1e-8, restart=20,
            solve_method=sm)
        pin(f"gmres_cd3d12_{sm}_2cycles", "gmres", A, b, gen=dict(matrix="convdiff3d", n=12), tol=0.0, atol=0.0,
            restart=10, maxiter=2, solve_method=sm)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=g)
    pin("gmres_cd3d12_x0", "gmres", A, b, x0, gen=dict(matrix="convdiff3d", n=12), tol=1e-9, restart=15)
    pin("gmres_zero_rhs", "gmres", A, torch.zeros(A.shape[0], dtype=torch.float64), gen=dict(matrix="convdiff3d", n=12),
        tol=1e-8, restart=10)

    # Jacobi (left-)preconditioned GMRES on the badly scaled non-symmetric system
    A = problems.scaled_convdiff3d_csr(12)
    b, _ = problems.manufactured_rhs(A, 4)
    gsc = dict(matrix="scaled_convdiff3d", n=12, seed=7)
    for sm in ("batched", "incremental"):
        pin(f"gmres_scd3d12_jacobi_{sm}", "gmres", A, b, gen=gsc, jacobi=True, tol=1e-9, restart=20, solve_method=sm)
    pin("gmres_scd3d12_jacobi_2cycles", "gmres", A, b, gen=gsc, jacobi=True, tol=0.0, atol=0.0, restart=8, maxiter=2)
    x0 = torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(13))
    pin("gmres_scd3d12_jacobi_x0", "gmres", A, b, x0, gen=gsc, jacobi=True, tol=1e-9, restart=15)

    # LDC pressure systems: matrix from our vectorised builder must equal the reference driver's, RHS sequence is
    # produced by the reference driver itself (ldc_solver_common.py:185-201)
    sys.path.insert(0, "/root/reference/FVM_example/LDC_by_torchsp")
    saved = {k: v for k, v in sys.modules.items() if k.startswith("pytorch_sparse_solver")}
    for k in saved:
        del sys.modules[k]
    sys.modules.update(ref_mods)
    import contextlib
    import io
    ldc_mod = importlib.import_module("ldc_solver_module_a")
    for nx, nsteps, re_ in ((32, 3, 100.0), (100, 2, 400.0)):
        with contextlib.redirect_stdout(io.StringIO()):
            s = ldc_mod.LDCSolverModuleA(nx=nx, Re=re_, method="gmres", device="cpu")
        rhs_list = []
        orig = s._solve_linear_system

        def capture(prhs, _orig=orig, _l=rhs_list):
            _l.append(prhs.clone())
            # advance the flow with BiCGStab (fast); the GMRES parity solves are done below on the captured RHS
            pt, info = ref.bicgstab(s.A_csr, prhs, tol=1e-10, maxiter=1000)
            return pt, info
        s._solve_linear_system = capture
        for _ in range(nsteps):
            s.step()
        A_ref = s.A_csr
        A_ours = problems.ldc_pressure_csr(nx)
        assert torch.equal(A_ref.crow_indices(), A_ours.crow_indices())
        assert torch.equal(A_ref.col_indices(), A_ours.col_indices())
        assert torch.equal(A_ref.values(), A_ours.values()), "LDC matrix builder differs from the reference driver"
        for t, prhs in enumerate(rhs_list):
            for sm in ("batched", "incremental"):
                if nx == 100 and (t > 0 and sm == "incremental"):
                    continue
                pin(f"gmres_ldc{nx}_step{t}_{sm}", "gmres", A_ours, prhs, store_vectors=True,
                    gen=dict(matrix="ldc", nx=nx), tol=1e-10, maxiter=1000, restart=30, solve_method=sm)
    for k in list(sys.modules):
        if k.startswith("pytorch_sparse_solver") or k.startswith("ldc_solver"):
            del sys.modules[k]
    sys.modules.update(saved)

    # ---- autograd (implicit adjoint, :1227-1248): reference needs dense / COO A --------------------
    auto = {}
    for kind, A, kw in (("cg", problems.poisson2d_csr(12, 12), dict(tol=1e-12)),
                        ("bicgstab", problems.convdiff3d_csr(6), dict(tol=1e-12)),
                        ("gmres", problems.convdiff3d_csr(6), dict(tol=1e-12, restart=30))):
        Ad = A.to_dense()
        b0, _ = problems.manufactured_rhs(A, 5)
        b1 = b0.clone().requires_grad_(True)
        x, info = getattr(ref, kind)(Ad, b1, **kw)
        loss = (x ** 2).sum()
        loss.backward()
        g_ref = b1.grad.clone()
        # oracle adjoint
        xo, _, _ = getattr(orc, kind)(A, b0, None, **kw)
        g_orc = orc.adjoint_grad_b(kind, A, 2.0 * xo, None, **kw)
        assert torch.allclose(g_ref, g_orc, rtol=0, atol=1e-13 * float(g_ref.abs().max())), kind
        g_exact = torch.linalg.solve(Ad.T, 2.0 * torch.linalg.solve(Ad, b0))
        name = f"autograd_{kind}"
        np.savez_compressed(GOLD / f"{name}.npz", b=b0.numpy(), grad_b=g_ref.numpy(), x=x.detach().numpy())
        auto[name] = dict(kind=kind, info=int(info), kwargs=kw, n=int(b0.numel()),
                          gen=(dict(matrix="poisson2d", nx=12, ny=12) if kind == "cg" else dict(matrix="convdiff3d", n=6)),
                          grad_vs_exact=float((g_ref - g_exact).abs().max() / g_exact.abs().max()))
        print(f"  pinned {name}: grad rel err vs analytic {auto[name]['grad_vs_exact']:.2e}")
    # BASELINE configs[3]: GMRES(30) on the LDC pressure system with autograd backward (reference needs COO A: CSR .T raises)
    A = problems.ldc_pressure_csr(32)
    with np.load(GOLD / "gmres_ldc32_step1_batched.npz") as z:
        b0 = torch.from_numpy(z["b"].copy())
    kw = dict(tol=1e-10, maxiter=1000, restart=30)
    b1 = b0.clone().requires_grad_(True)
    x, info = ref.gmres(A.to_sparse_coo(), b1, **kw)
    (x ** 2).sum().backward()
    xo, _, _ = orc.gmres(A, b0, None, **kw)
    g_orc = orc.adjoint_grad_b("gmres", A, 2.0 * xo, None, **kw)
    assert torch.equal(b1.grad, g_orc), "oracle adjoint differs from the reference on LDC-32"
    np.savez_compressed(GOLD / "autograd_gmres_ldc32.npz", b=b0.numpy(), grad_b=b1.grad.numpy(), x=x.detach().numpy())
    auto["autograd_gmres_ldc32"] = dict(kind="gmres", info=int(info), kwargs=kw, n=int(b0.numel()), gen=dict(matrix="ldc", nx=32),
                                        note="GMRES(30) on the LDC pressure system with autograd backward; reference run with COO A")
    manifest["autograd"] = auto

    # ---- full-size digests measured with the reference at survey time (BASELINE.md §2; 3-6 CPU-minutes each,
    # not re-run here).  Used by the GPU tests at BASELINE.json's full sizes.
    manifest["survey_digests"] = {
        "cg_p3d256_ones_tol1e-8": dict(iterations=611, info=0, relres=9.787e-9, x_norm=6799410.672531194,
                                       x_sum=22609955493.50508, x_0=0.7157477149852747,
                                       x_8388608=3.1720422387358913),
        "cg_p3d256_ones_maxiter10": dict(iterations=10, x_norm=1.232426453129e+06),
        "bicgstab_cd3d256_rand_tol1e-8": dict(iterations=399, info=0, relres=4.845e-9, x_norm=4096.465821813488,
                                              b_norm=34480.55109333533),
        "bicgstab_cd3d256_rand_tol1e-10": dict(iterations=477, info=0, relres=9.253e-11, x_norm=4096.465821360726),
    }
    with open(GOLD / "manifest.json", "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)
    print(f"wrote {len(manifest['cases'])} cases to {GOLD}")


if __name__ == "__main__":
    main()
