"""module_a front end: the reference's Python API over the B200-native Krylov library.

Mirrors (names, argument meaning, return values, error behaviour) of the reference file
src/pytorch_sparse_solver/module_a/torch_sparse_linalg.py:

    cg        :1019-1088      bicgstab :1091-1158      gmres :641-784
    cg/bicgstab/gmres_differentiable :1261-1367        LinearSolveFunction :1161-1224
    ImplicitAdjointFunction :1227-1248 (here: _ImplicitAdjoint)

What is different underneath: the whole iteration loop of each solver is ONE call into
libbk_krylov.so (hand-written sm_100a kernels, device-resident loop, deterministic reductions).
Routes:

  * native   A is a 2-D CUDA tensor (CSR / COO / dense), b a CUDA tensor, M is None
             -> bk_cg / bk_bicgstab / bk_gmres on the registered CSR matrix.
  * host     the same with CPU tensors: the arrays are copied to the current CUDA device, solved
             there and x is copied back (bk_solve_host).  Still the CUDA path — this build has no
             CPU solver, and raises if no CUDA device exists.
  * generic  callable A, preconditioner M or pytree b: the reference's recurrences driven from
             Python (one host sync per iteration, as in the reference) with every dot / axpy done
             by the library's deterministic kernels (see generic.py).  With a TENSOR A (and a callable
             M) the implicit-differentiation backward is attached exactly as on the native route
             (reference :1079-1086, :1145-1152, :775-782): the adjoint solve runs the same generic
             solver on the cached device transpose with the same M.  A callable A cannot be
             differentiated here (the reference lets autograd unroll its torch ops; our kernels are
             not autograd ops): a warning says so once.
  * dist     A is a distributed.DistMatrix (row-partitioned over the ranks of a process group), b this
             rank's slab: bk_dist_cg / bk_dist_bicgstab / bk_dist_gmres (SURVEY §8e "API stays additive").
"""
from __future__ import annotations

import warnings
from typing import Any, Callable, Optional, Tuple, Union

import torch

from .. import _native
from .preconditioners import JacobiPreconditioner, SymmetricGaussSeidelPreconditioner
from .torch_tree_util import tree_leaves

__all__ = [
    "cg", "bicgstab", "gmres",
    "cg_differentiable", "bicgstab_differentiable", "gmres_differentiable",
    "LinearSolveFunction",
]

# Tests comparing against the CPU oracle set this to 'cpu' so that gmres uses the reference's CPU
# tolerance constants even though the tensors live on a CUDA device (reference :737-744).
GMRES_TOLERANCE_DEVICE: Optional[str] = None

# Opt-in extension (SURVEY §8f-3): also return dL/dA = -(A^-T dL/dx) x^T on A's sparsity pattern when A requires grad.
# Off by default because the reference returns None for A (:1248).
GRAD_WRT_A: bool = False

# Filled by every PUBLIC solve (cg / bicgstab / gmres / *_differentiable): the native bk_result of the most recent
# call (iterations, matvecs, device_ms, loop_mode_used ...).  The reference returns no iteration count
# (solver.py:373); this is strictly extra information.  Adjoint solves run inside backward() do not touch it, and
# callers that must not depend on a module global (the router, re-entrant code) pass `_result={}` to the solver
# functions and read the same dictionary from there.
last_result: dict = {}

# restarts above this run on the generic route (the native GMRES keeps its small dense arrays in shared memory)
NATIVE_MAX_RESTART = 256


# --------------------------------------------------------------------------------------------------
# validation helpers (same exceptions as the reference)
# --------------------------------------------------------------------------------------------------
def _check_operator(A):
    """_normalize_matvec :176-208: ValueError for a non-square tensor, TypeError for junk."""
    if callable(A) and not isinstance(A, torch.Tensor):
        return "callable"
    if isinstance(A, torch.Tensor):
        if A.ndim != 2 or A.shape[0] != A.shape[1]:
            raise ValueError(f'linear operator must be a square matrix, but has shape: {A.shape}')
        return "tensor"
    raise TypeError(f'linear operator must be either a function or tensor: {A}')


def _check_x0(b, x0):
    """_isolve :992-1002 / gmres :723-727."""
    b_leaves, x0_leaves = tree_leaves(b), tree_leaves(x0)
    if len(b_leaves) != len(x0_leaves):
        raise ValueError('x0 and b must have matching tree structure')
    for bl, xl in zip(b_leaves, x0_leaves):
        if bl.shape != xl.shape:
            raise ValueError(f'arrays in x0 and b must have matching shapes: {xl.shape} vs {bl.shape}')


def _route(A, b, x0, M, native_M: bool = False) -> str:
    """native_M: the solver has a device implementation for a built-in preconditioner object (Jacobi, SGS)."""
    kind = _check_operator(A)
    if kind == "tensor" and isinstance(b, torch.Tensor) and (A.is_complex() or b.is_complex()):
        return "complex"
    builtin = native_M and isinstance(M, _BUILTIN_M) and kind == "tensor" and A.is_cuda
    if kind == "callable" or (M is not None and not builtin) or not isinstance(b, torch.Tensor):
        return "generic"
    if b.ndim != 1 or b.shape[0] != A.shape[0]:
        raise ValueError(f"b must be a vector of length {A.shape[0]}, got shape {tuple(b.shape)}")
    if A.is_complex() or b.is_complex():
        return "complex"
    if A.is_cuda != b.is_cuda:
        raise ValueError("A and b must live on the same device")
    return "native" if A.is_cuda else "host"


_BUILTIN_M = (JacobiPreconditioner, SymmetricGaussSeidelPreconditioner)


def _work_dtype(A: torch.Tensor, b: torch.Tensor) -> torch.dtype:
    """fp64 unless BOTH A and b are fp32 (the reference always computes in fp64, :979-980; it raises
    for fp32 A — here that combination selects the native fp32 kernels)."""
    if A.dtype == torch.float32 and b.dtype == torch.float32:
        return torch.float32
    return torch.float64


def _use_implicit_diff(A: Any, b: Any) -> bool:
    """:1251-1258"""
    return (isinstance(A, torch.Tensor) and isinstance(b, torch.Tensor) and A.ndim == 2
            and (A.requires_grad or b.requires_grad))


def _gmres_effective_tolerances(tol: float, atol: float, size: int, device_type: str) -> Tuple[float, float]:
    """The host-only part of gmres' tolerance set-up (:733-748), including its fp32 roundings.

    atol_tensor = max(tensor(adaptive_tol) * ||b||, max(tensor(atol), tensor(base_atol)))
    where torch.tensor(<python float>) is fp32 and torch.tensor(<fp64 tensor>) stays fp64.
    Returns (tol_eff, atol_eff); the device finishes with ||b||.
    """
    if GMRES_TOLERANCE_DEVICE is not None:
        device_type = GMRES_TOLERANCE_DEVICE
    eps = torch.finfo(torch.float64).eps
    root = torch.sqrt(torch.tensor(size, dtype=torch.float64))
    scaled = (1e-12 if device_type == 'cuda' else 1e-14) * root
    base_atol = eps * (1000 if device_type == 'cuda' else 100) * size
    adaptive = max(tol, scaled)  # python max: keeps `tol` (a float) unless the tensor is larger
    tol_eff = float(torch.tensor(adaptive)) if not isinstance(adaptive, torch.Tensor) else float(adaptive)
    atol_eff = max(float(torch.tensor(atol)), float(torch.tensor(base_atol)))
    return tol_eff, atol_eff


# --------------------------------------------------------------------------------------------------
# the three solver cores (no autograd)
# --------------------------------------------------------------------------------------------------
def _solve_core(name: str, A: torch.Tensor, b: torch.Tensor, x0: Optional[torch.Tensor], tol: float, atol: float,
                maxiter: Optional[int], restart: int = 20, solve_method: str = 'batched',
                transpose: bool = False, precond=None) -> Tuple[torch.Tensor, int, dict]:
    """Run one solver on (A or A^T).  Returns (x, info, result dict) with x of the work dtype on b's device."""
    route = "native" if A.is_cuda else "host"
    wdt = _work_dtype(A, b)
    if precond is not None and route != "native":
        raise _native.NativeLibraryError("built-in preconditioners run on the native CUDA route only")
    if name == "gmres":
        if solve_method == 'incremental':
            method = _native.BK_GMRES_INCREMENTAL
        elif solve_method == 'batched':
            method = _native.BK_GMRES_BATCHED
        else:
            raise ValueError(f"Unsupported solve_method: {solve_method}")
    with torch.no_grad():
        bw = b.detach().to(wdt)
        x0w = None if x0 is None else x0.detach().to(wdt)
        n = bw.numel()
        if route == "native":
            mat = _native.register_matrix(A, wdt)
            if transpose:
                mat = mat.transpose()
            sgs = precond.sgs(wdt) if isinstance(precond, SymmetricGaussSeidelPreconditioner) else None
            if sgs is not None:   # the adjoint solve runs on A^T with the M of A, as the reference does with a callable M
                if name == "gmres":
                    tol_eff, atol_eff = _gmres_effective_tolerances(tol, atol, n, 'cuda')
                    x, res = mat.gmres_sgs(sgs, bw, x0w, tol_eff, atol_eff, restart, maxiter, method)
                else:
                    x, res = getattr(mat, name + "_sgs")(sgs, bw, x0w, tol, atol, maxiter)
            elif name == "cg" and precond is not None:   # diag(A^T) == diag(A): the adjoint solve reuses M (:1079-1084)
                x, res = mat.cg_jacobi(precond.diagonal(wdt, bw.device), bw, x0w, tol, atol, maxiter)
            elif name == "cg":
                x, res = mat.cg(bw, x0w, tol, atol, maxiter)
            elif name == "bicgstab" and precond is not None:
                x, res = mat.bicgstab_jacobi(precond.diagonal(wdt, bw.device), bw, x0w, tol, atol, maxiter)
            elif name == "bicgstab":
                x, res = mat.bicgstab(bw, x0w, tol, atol, maxiter)
            else:
                tol_eff, atol_eff = _gmres_effective_tolerances(tol, atol, n, 'cuda')
                if precond is not None:
                    x, res = mat.gmres_jacobi(precond.diagonal(wdt, bw.device), bw, x0w, tol_eff, atol_eff, restart,
                                              maxiter, method)
                else:
                    x, res = mat.gmres(bw, x0w, tol_eff, atol_eff, restart, maxiter, method)
        else:
            Ad = A.detach()
            if transpose:
                Ad = Ad.t()
            if Ad.layout != torch.sparse_csr:
                Ad = (Ad.coalesce() if Ad.layout == torch.sparse_coo else Ad).to_sparse_csr()
            crow, col, val = Ad.crow_indices(), Ad.col_indices(), Ad.values().to(wdt)
            if name == "gmres":
                t, a = _gmres_effective_tolerances(tol, atol, n, 'cpu')
                x, res = _native.solve_host(_native.METHOD_GMRES, crow, col, val, bw, x0w, t, a, maxiter, restart,
                                            method)
            else:
                code = _native.METHOD_CG if name == "cg" else _native.METHOD_BICGSTAB
                x, res = _native.solve_host(code, crow, col, val, bw, x0w, tol, atol, maxiter)
    return x.reshape(b.shape), int(res["info"]), dict(res, solver=name, route=route)


def _publish(res: dict, sink: Optional[dict]):
    global last_result
    last_result = res
    if sink is not None:
        sink.clear()
        sink.update(res)


class _ImplicitAdjoint(torch.autograd.Function):
    """Attach the implicit-differentiation backward to a precomputed solution (:1227-1248).

    backward: grad_b = solve(A^T, grad_x) with the forward's x0 / tolerances (:1246); no gradient for
    A (reference returns None, :1248).  A^T is the library's cached device transpose, so CSR inputs
    work (the reference's `A.T` raises for CSR on torch 2.11).
    """

    @staticmethod
    def forward(ctx, A, b, x, name, x0, tol, atol, restart, maxiter, solve_method, precond=None):
        ctx.A = A
        ctx.x = x.detach()
        ctx.meta = (name, x0, tol, atol, restart, maxiter, solve_method, precond)
        return x.clone()

    @staticmethod
    def backward(ctx, grad_output):
        name, x0, tol, atol, restart, maxiter, solve_method, precond = ctx.meta
        grad_b = grad_A = None
        want_A = GRAD_WRT_A and ctx.needs_input_grad[0]
        if ctx.needs_input_grad[1] or want_A:
            g, _, _ = _solve_core(name, ctx.A, grad_output.contiguous(), x0, tol, atol, maxiter, restart, solve_method,
                                  transpose=True, precond=precond)
            if ctx.needs_input_grad[1]:
                grad_b = g.to(grad_output.dtype)
            if want_A:
                grad_A = _grad_wrt_matrix(ctx.A, g, ctx.x)
        return (grad_A, grad_b) + (None,) * 9


def _grad_wrt_matrix(A: torch.Tensor, g: torch.Tensor, x: torch.Tensor) -> Optional[torch.Tensor]:
    """dL/dA in A's own layout: -g x^T restricted to the stored pattern for CSR / coalesced COO, dense outer product
    for strided A."""
    with torch.no_grad():
        if A.layout == torch.strided:
            return -torch.outer(g.to(A.dtype), x.to(A.dtype))
        if not A.is_cuda:
            return None
        wdt = torch.float32 if (A.dtype == torch.float32 and g.dtype == torch.float32) else torch.float64
        if A.layout == torch.sparse_coo and not A.is_coalesced():
            return None
        vals = _native.register_matrix(A, wdt).grad_pattern(g.to(wdt), x.to(wdt)).to(A.dtype)
        if A.layout == torch.sparse_csr:
            return torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), vals, size=A.shape)
        return torch.sparse_coo_tensor(A._indices(), vals, A.shape).coalesce()


def _finish(name, A, b, x, info, x0, tol, atol, restart, maxiter, solve_method, precond=None):
    if _use_implicit_diff(A, b):
        x = _ImplicitAdjoint.apply(A, b, x, name, x0, tol, atol, restart, maxiter, solve_method, precond)
    return x, info


class _GenericAdjoint(torch.autograd.Function):
    """The implicit-differentiation backward for the generic route with a TENSOR A and a callable M: the reference
    attaches ImplicitAdjointFunction whenever A is a 2-D tensor, with or without M (:1079-1086 cg, :1145-1152 bicgstab,
    :775-782 gmres), and its transpose_solve_fn re-uses M, x0 and the tolerances."""

    @staticmethod
    def forward(ctx, A, b, x, name, x0, tol, atol, restart, maxiter, solve_method, M):
        ctx.A = A
        ctx.meta = (name, x0, tol, atol, restart, maxiter, solve_method, M)
        return x.clone()

    @staticmethod
    def backward(ctx, grad_output):
        from . import generic
        name, x0, tol, atol, restart, maxiter, solve_method, M = ctx.meta
        grad_b = None
        if ctx.needs_input_grad[1]:
            global last_result
            saved = last_result          # the adjoint solve must not overwrite the forward's record
            try:
                with torch.no_grad():
                    g = grad_output.detach().contiguous()
                    if name == "cg":
                        gb, _ = generic.generic_cg(ctx.A, g, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, transpose=True)
                    elif name == "bicgstab":
                        gb, _ = generic.generic_bicgstab(ctx.A, g, x0, tol=tol, atol=atol, maxiter=maxiter, M=M,
                                                         transpose=True)
                    else:
                        gb, _ = generic.generic_gmres(ctx.A, g, x0, tol=tol, atol=atol, restart=restart,
                                                      maxiter=maxiter, M=M, solve_method=solve_method, transpose=True)
            finally:
                last_result = saved
            grad_b = gb.to(grad_output.dtype)
        return (None, grad_b) + (None,) * 9


_warned_callable_grad = False


def _generic(name, A, b, x0, tol, atol, maxiter, M, restart=20, solve_method='batched', _result=None):
    """Generic route + the autograd semantics of the reference for it."""
    global _warned_callable_grad
    from . import generic
    fn = {"cg": generic.generic_cg, "bicgstab": generic.generic_bicgstab, "gmres": generic.generic_gmres}[name]
    kw = dict(tol=tol, atol=atol, maxiter=maxiter, M=M)
    if name == "gmres":
        kw.update(restart=restart, solve_method=solve_method)
    x, info = fn(A, b, x0, **kw)
    _publish(dict(last_result), _result)
    if _use_implicit_diff(A, b):
        if A.is_complex() or b.is_complex():
            return x, info
        x = _GenericAdjoint.apply(A, b, x, name, x0, tol, atol, restart, maxiter, solve_method, M)
    elif not _warned_callable_grad and any(isinstance(t, torch.Tensor) and t.requires_grad for t in tree_leaves(b)):
        _warned_callable_grad = True
        warnings.warn("module_a: b requires grad but A is a callable — this build cannot differentiate through a "
                      "callable operator (pass A as a tensor to get the implicit-differentiation backward)")
    return x, info


def _is_dist(A) -> bool:
    return type(A).__name__ == "DistMatrix" and hasattr(A, "n_global")


# --------------------------------------------------------------------------------------------------
# public API
# --------------------------------------------------------------------------------------------------
def cg(A: Union[torch.Tensor, Callable[[Any], Any]], b: Any, x0: Optional[Any] = None, *, tol: float = 1e-5,
       atol: float = 0.0, maxiter: Optional[int] = None, M: Optional[Callable[[Any], Any]] = None,
       _result: Optional[dict] = None) -> Tuple[Any, Optional[int]]:
    """Conjugate gradient for hermitian positive definite A.  Same contract as reference cg (:1019-1088):
    returns (x, info), x fp64 (fp32 when A and b are both fp32), info 0 if ||b - A x|| <= max(tol*||b||, atol)
    else -1; gradients w.r.t. b by implicit differentiation with a second (transposed) solve."""
    if _is_dist(A):
        return A._module_a_solve("cg", b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, _result=_result)
    route = _route(A, b, x0, M, native_M=True)
    if route == "complex":
        from .complex_route import complex_solve
        return complex_solve("cg", A, b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, _result=_result)
    if route == "generic":
        return _generic("cg", A, b, x0, tol, atol, maxiter, M, _result=_result)
    if x0 is not None:
        _check_x0(b, x0)
    x, info, res = _solve_core("cg", A, b, x0, tol, atol, maxiter, precond=M)
    _publish(res, _result)
    return _finish("cg", A, b, x, info, x0, tol, atol, 20, maxiter, 'batched', precond=M)


def bicgstab(A: Union[torch.Tensor, Callable[[Any], Any]], b: Any, x0: Optional[Any] = None, *, tol: float = 1e-5,
             atol: float = 0.0, maxiter: Optional[int] = None, M: Optional[Callable[[Any], Any]] = None,
             _result: Optional[dict] = None) -> Tuple[Any, Optional[int]]:
    """Bi-conjugate gradient stabilised for general A.  Same contract as reference bicgstab (:1091-1158)."""
    if _is_dist(A):
        return A._module_a_solve("bicgstab", b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, _result=_result)
    route = _route(A, b, x0, M, native_M=True)
    if route == "complex":
        from .complex_route import complex_solve
        return complex_solve("bicgstab", A, b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, _result=_result)
    if route == "generic":
        return _generic("bicgstab", A, b, x0, tol, atol, maxiter, M, _result=_result)
    if x0 is not None:
        _check_x0(b, x0)
    x, info, res = _solve_core("bicgstab", A, b, x0, tol, atol, maxiter, precond=M)
    _publish(res, _result)
    return _finish("bicgstab", A, b, x, info, x0, tol, atol, 20, maxiter, 'batched', precond=M)


def gmres(A: Union[torch.Tensor, Callable[[Any], Any]], b: Any, x0: Optional[Any] = None, *, tol: float = 1e-5,
          atol: float = 0.0, restart: int = 20, maxiter: Optional[int] = None,
          M: Optional[Callable[[Any], Any]] = None, solve_method: str = 'batched',
          _result: Optional[dict] = None) -> Tuple[Any, Optional[int]]:
    """Restarted GMRES.  Same contract as reference gmres (:641-784): `maxiter` counts restart cycles,
    solve_method 'batched' (default; always `restart` Arnoldi steps per cycle) or 'incremental' (Givens QR with
    early exit inside a cycle); info 0 iff ||b - A x|| <= 10*atol_eff and x is finite."""
    if solve_method not in ('batched', 'incremental'):
        raise ValueError(f"Unsupported solve_method: {solve_method}")
    if _is_dist(A):
        return A._module_a_solve("gmres", b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, restart=restart,
                                 solve_method=solve_method, _result=_result)
    route = _route(A, b, x0, M, native_M=True)
    if route == "complex":
        from .complex_route import complex_solve
        return complex_solve("gmres", A, b, x0, tol=tol, atol=atol, maxiter=maxiter, M=M, restart=restart,
                             solve_method=solve_method, _result=_result)
    if route != "generic" and restart > NATIVE_MAX_RESTART:
        route = "generic"         # the reference accepts any restart; very long cycles run Python-driven
    if route == "generic":
        return _generic("gmres", A, b, x0, tol, atol, maxiter, M, restart, solve_method, _result=_result)
    if x0 is not None:
        _check_x0(b, x0)
    if restart < 1:
        raise ValueError("restart must be >= 1")
    x, info, res = _solve_core("gmres", A, b, x0, tol, atol, maxiter, restart, solve_method, precond=M)
    _publish(res, _result)
    return _finish("gmres", A, b, x, info, x0, tol, atol, restart, maxiter, solve_method, precond=M)


class LinearSolveFunction(torch.autograd.Function):
    """Legacy differentiable wrapper with the reference's signature (:1161-1224):
    forward(A_matrix, b, solve_fn, transpose_solve_fn, *solve_args) -> x ; backward gives only grad_b."""

    @staticmethod
    def forward(ctx, A_matrix, b, solve_fn, transpose_solve_fn, *solve_args):
        x, _info = solve_fn(A_matrix, b, *solve_args)
        ctx.A = A_matrix
        ctx.transpose_solve_fn = transpose_solve_fn
        ctx.solve_args = solve_args
        return x

    @staticmethod
    def backward(ctx, grad_output):
        grad_b = None
        if ctx.needs_input_grad[1]:
            fn = ctx.transpose_solve_fn
            if getattr(fn, "_bk_accepts_transposed", False):
                A_T = _Transposed(ctx.A)          # library-cached device transpose, works for CSR
            else:                                 # user-supplied solver: materialise A^T like the reference (:1215)
                A_T = ctx.A.T.conj() if torch.is_complex(ctx.A) else ctx.A.T
            grad_b, _ = fn(A_T, grad_output, *ctx.solve_args)
        return (None, grad_b, None, None) + (None,) * len(ctx.solve_args)


class _Transposed:
    """Marker handed to a LinearSolveFunction transpose_solve_fn: "solve with A^T" without materialising A.T
    (which raises for CSR tensors on torch 2.11)."""

    def __init__(self, A):
        self.A = A


def _legacy(name, A, b, x0, tol, atol, maxiter, restart=20):
    if not isinstance(A, torch.Tensor) or A.ndim != 2:
        raise ValueError(f"For differentiable {name.upper() if name != 'bicgstab' else 'BiCGStab'}, "
                         "A must be a 2D tensor")

    def solve_fn(A_mat, rhs, x_init=None, tol_=1e-5, atol_=0.0, *rest):
        transpose = isinstance(A_mat, _Transposed)
        A_use = A_mat.A if transpose else A_mat
        _route(A_use, rhs, x_init, None)
        if name == "gmres":
            restart_, maxiter_ = rest
        else:
            (maxiter_,) = rest
            restart_ = 20
        x_, info_, res_ = _solve_core(name, A_use, rhs, x_init, tol_, atol_, maxiter_, restart_, 'batched',
                                      transpose=transpose)
        if not transpose:
            _publish(res_, None)
        return x_, info_

    solve_fn._bk_accepts_transposed = True
    args = (x0, tol, atol, restart, maxiter) if name == "gmres" else (x0, tol, atol, maxiter)
    return LinearSolveFunction.apply(A, b, solve_fn, solve_fn, *args)


def cg_differentiable(A: torch.Tensor, b: torch.Tensor, x0: Optional[torch.Tensor] = None, *, tol: float = 1e-5,
                      atol: float = 0.0, maxiter: Optional[int] = None) -> torch.Tensor:
    """:1261-1296 — returns x only; gradient of b via an adjoint CG solve."""
    return _legacy("cg", A, b, x0, tol, atol, maxiter)


def bicgstab_differentiable(A: torch.Tensor, b: torch.Tensor, x0: Optional[torch.Tensor] = None, *,
                            tol: float = 1e-5, atol: float = 0.0, maxiter: Optional[int] = None) -> torch.Tensor:
    """:1299-1330"""
    return _legacy("bicgstab", A, b, x0, tol, atol, maxiter)


def gmres_differentiable(A: torch.Tensor, b: torch.Tensor, x0: Optional[torch.Tensor] = None, *, tol: float = 1e-5,
                         atol: float = 0.0, restart: int = 20, maxiter: Optional[int] = None) -> torch.Tensor:
    """:1333-1367"""
    return _legacy("gmres", A, b, x0, tol, atol, maxiter, restart)
