#!/usr/bin/env python3
"""Multicolor symmetric Gauss-Seidel against no preconditioner and Jacobi, on one GPU.

Systems (b = A randn, seed 0): P3D-256 CG at tol 1e-8, CD3D-256 BiCGStab at tol 1e-8, scaled P3D-128 CG at tol 1e-8,
LDC-100 GMRES(30) at tol 1e-10 (maxiter only bounds a run that does not converge).  For each (system, M): iterations,
device ms of one solve after a warm-up solve (bk_result.device_ms), the SGS set-up ms (coloring + row lists, host clock
around a synchronised call), the number of colors and rounds, and the true relative residual ||b - A x|| / ||b|| computed with torch's sparse matmul.  The
first line records the card and its power limit.  One JSON line per record.

    python tools/sgs_bench.py [--out profiles/r03_sgs_bench.jsonl]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "pytorch-sparse-linalg-torch-amgx.cg.bicg.gmres_b200"))
import torch  # noqa: E402

from pytorch_sparse_solver import _native, module_a, problems  # noqa: E402

CASES = [
    ("P3D-256", "cg", lambda d: problems.poisson3d_csr(256, device=d), dict(tol=1e-8, maxiter=20000)),
    ("CD3D-256", "bicgstab", lambda d: problems.convdiff3d_csr(256, device=d), dict(tol=1e-8, maxiter=20000)),
    ("scaled P3D-128", "cg", lambda d: problems.scaled_poisson3d_csr(128, device=d), dict(tol=1e-8, maxiter=100000)),
    ("LDC-100", "gmres", lambda d: problems.ldc_pressure_csr(100, device=d), dict(tol=1e-10, restart=30,
                                                                               maxiter=1000)),
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"record": "card", "torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_sgs_bench.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sgs_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = [card()]
    for name, solver, make, kw in CASES:
        A = make(dev)
        b = A @ torch.randn(A.shape[0], dtype=torch.float64, generator=torch.Generator().manual_seed(0)).to(dev)
        mat = _native.register_matrix(A, torch.float64)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        S = mat.sgs()
        torch.cuda.synchronize()
        setup_ms = 1e3 * (time.perf_counter() - t0)
        M_sgs = module_a.SymmetricGaussSeidelPreconditioner(A)
        for label, M in (("none", None), ("jacobi", module_a.JacobiPreconditioner(A)), ("sgs", M_sgs)):
            fn = getattr(module_a, solver)
            fn(A, b, M=M, **kw)                                  # warm-up: graphs, modules
            res = {}
            x, info = fn(A, b, M=M, _result=res, **kw)
            rel = float(torch.linalg.norm(b - A @ x) / torch.linalg.norm(b))
            rec = {"record": "solve", "system": name, "n": A.shape[0], "solver": solver, "M": label, "tol": kw["tol"],
                   "info": info, "iterations": res["iterations"], "matvecs": res["matvecs"],
                   "kernel_launches": res["kernel_launches"], "device_ms": res["device_ms"],
                   "loop_mode_used": res["loop_mode_used"], "true_rel_residual": rel}
            if solver == "gmres":
                rec["restart"] = kw["restart"]
            if label == "sgs":
                rec.update(setup_ms=setup_ms, colors=S.num_colors, rounds=S.rounds)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        del A, b, mat, S, M_sgs
        _native.clear_cache()
        torch.cuda.empty_cache()
    print(json.dumps(lines[0]))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
