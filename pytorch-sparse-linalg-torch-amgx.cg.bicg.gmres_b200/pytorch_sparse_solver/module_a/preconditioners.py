"""Built-in preconditioners for Module A (SURVEY §8f-1).

The reference takes `M` as an arbitrary Python callable (torch_sparse_linalg.py:821, :849), which forces every
application through the interpreter.  `JacobiPreconditioner(A)` is such a callable — `M(r) = r / diag(A)`, exactly
what users of the reference write as `M = lambda r: r / d` — that `cg()`, `bicgstab()` and `gmres()` additionally
recognise: for a CUDA matrix the whole preconditioned iteration then stays on the device (`bk_cg_jacobi`,
`bk_bicgstab_jacobi`, `bk_gmres_jacobi`), with results identical to passing the lambda to the reference (golden
fixtures `*_jacobi*`).  With a callable `A` or on CPU tensors it behaves like any other callable `M`.
`SymmetricGaussSeidelPreconditioner(A)` is the stronger built-in: one multicolor symmetric Gauss-Seidel sweep
(`bk_cg_sgs`, `bk_bicgstab_sgs`, `bk_gmres_sgs` on the device route; a library call per application elsewhere).
"""
from __future__ import annotations

import torch

from .. import _native


class JacobiPreconditioner:
    """M = diag(A)^-1, applied as r / d."""

    def __init__(self, A: torch.Tensor):
        if type(A).__name__ == "DistMatrix" and hasattr(A, "diagonal"):   # row-partitioned: this rank's slice
            d = A.diagonal()
            if bool((d == 0).any()):
                raise ValueError("JacobiPreconditioner: the matrix has a zero on its diagonal")
            self.d = d
            self.shape = (A.n_global, A.n_global)
            return
        if not isinstance(A, torch.Tensor) or A.ndim != 2 or A.shape[0] != A.shape[1]:
            raise ValueError("JacobiPreconditioner needs a square 2-D tensor (dense, COO or CSR)")
        with torch.no_grad():
            Ad = A.detach()
            if Ad.layout == torch.strided:
                d = torch.diagonal(Ad).clone()
            elif Ad.is_cuda and not Ad.is_complex():
                wdt = torch.float32 if Ad.dtype == torch.float32 else torch.float64
                d = _native.register_matrix(Ad, wdt).diagonal()
            else:
                C = Ad.coalesce() if Ad.layout == torch.sparse_coo else Ad.to_sparse_coo().coalesce()
                i, v = C.indices(), C.values()
                m = i[0] == i[1]
                d = torch.zeros(A.shape[0], dtype=v.dtype, device=v.device).index_add_(0, i[0][m], v[m])
        if bool((d == 0).any()):
            raise ValueError("JacobiPreconditioner: the matrix has a zero on its diagonal")
        self.d = d
        self.shape = tuple(A.shape)

    def diagonal(self, dtype: torch.dtype, device) -> torch.Tensor:
        return self.d.to(device=device, dtype=dtype)

    def __call__(self, r):
        if isinstance(r, torch.Tensor):
            return r / self.d.to(device=r.device, dtype=r.dtype)
        raise TypeError("JacobiPreconditioner applies to a single tensor")


class BlockJacobiPreconditioner:
    """M = blockdiag(A)^-1 with square diagonal blocks of `block_size` rows (SURVEY §8f-1).

    The inverses of the diagonal blocks are formed once at construction (set-up: a batched torch.linalg.inv of
    [n / bs, bs, bs]); every application `M(r)` is ONE library kernel (bk_block_apply) — no Python per block, no
    torch.bmm on the path.  It is a callable like any user-supplied M, so cg / bicgstab / gmres take the generic route
    with it (the user's-callable route, vector work in the library's kernels) and the implicit-diff backward re-uses
    it on A^T.  Equivalent to what users of the reference write as
    `M = lambda r: torch.bmm(Binv, r.view(-1, bs, 1)).view(-1)` (fixtures `*_blockjacobi*`)."""

    def __init__(self, A: torch.Tensor, block_size: int = 4):
        if not isinstance(A, torch.Tensor) or A.ndim != 2 or A.shape[0] != A.shape[1]:
            raise ValueError("BlockJacobiPreconditioner needs a square 2-D tensor (dense, COO or CSR)")
        if block_size < 1 or block_size > 64:
            raise ValueError("block_size must be in [1, 64]")
        self.bs = int(block_size)
        n = int(A.shape[0])
        self.shape = (n, n)
        with torch.no_grad():
            self.inv = self.diagonal_block_inverses(A.detach(), self.bs)

    @staticmethod
    def diagonal_block_inverses(A: torch.Tensor, bs: int) -> torch.Tensor:
        """[ceil(n / bs), bs, bs] inverses of the diagonal blocks of A (the last block is padded with the identity)."""
        n = int(A.shape[0])
        nb = (n + bs - 1) // bs
        if A.layout == torch.strided:
            idx = A.nonzero(as_tuple=False)
            r, c, v = idx[:, 0], idx[:, 1], A[idx[:, 0], idx[:, 1]]
        else:
            Cc = A.coalesce() if A.layout == torch.sparse_coo else A.to_sparse_coo().coalesce()
            r, c, v = Cc.indices()[0], Cc.indices()[1], Cc.values()
        wdt = torch.float32 if v.dtype == torch.float32 else torch.float64
        keep = (r // bs) == (c // bs)
        r, c, v = r[keep], c[keep], v[keep].to(wdt)
        blocks = torch.zeros(nb * bs * bs, dtype=wdt, device=v.device)
        blocks.index_add_(0, (r // bs) * bs * bs + (r % bs) * bs + (c % bs), v)
        blocks = blocks.view(nb, bs, bs)
        pad = nb * bs - n
        if pad:
            k = torch.arange(bs - pad, bs, device=v.device)
            blocks[nb - 1, k, k] = 1.0
        return torch.linalg.inv(blocks).contiguous()

    def __call__(self, r):
        if not isinstance(r, torch.Tensor):
            raise TypeError("BlockJacobiPreconditioner applies to a single tensor")
        if not r.is_cuda:
            raise _native.NativeLibraryError("BlockJacobiPreconditioner applies on the CUDA device (no CPU fallback)")
        inv = self.inv.to(device=r.device, dtype=r.dtype)
        if inv is not self.inv:
            self.inv = inv
        return _native.block_apply(inv, r.detach(), self.bs).reshape(r.shape)


class SymmetricGaussSeidelPreconditioner:
    """M = one multicolor symmetric Gauss-Seidel sweep: z = 0, a forward sweep over the colors of A's pattern, then a
    backward sweep, every row z_i = (r_i - sum_{j != i} a_ij z_j) / a_ii.  For symmetric A this is
    M = (D + U)^-1 D (D + L)^-1 with the rows taken in color order, which is symmetric positive definite when A is.

    The coloring (deterministic Jones-Plassmann rounds) is built once per work dtype, when A is first registered for it.
    The sweeps read A's values at every application: when A is a CUDA CSR tensor of the work dtype, its values are
    borrowed, so an in-place update of A.values() is picked up by the next application (JacobiPreconditioner, by
    contrast, keeps the diagonal it read at construction).  Only a change of the sparsity pattern needs a new object.

    cg(), bicgstab() and gmres() run the whole preconditioned iteration on the device with it (and reuse it for the
    adjoint solve on A^T); as a callable `M(r)` it works on the generic route too, e.g. with a callable A."""

    def __init__(self, A: torch.Tensor):
        if type(A).__name__ == "DistMatrix":
            raise ValueError("SymmetricGaussSeidelPreconditioner does not support row-partitioned matrices")
        if not isinstance(A, torch.Tensor) or A.ndim != 2 or A.shape[0] != A.shape[1]:
            raise ValueError("SymmetricGaussSeidelPreconditioner needs a square 2-D tensor (dense, COO or CSR)")
        if A.is_complex():
            raise ValueError("SymmetricGaussSeidelPreconditioner supports real matrices only")
        if not A.is_cuda:
            raise _native.NativeLibraryError("SymmetricGaussSeidelPreconditioner runs on the CUDA device "
                                             "(no CPU fallback)")
        self.A = A.detach()
        self.shape = tuple(A.shape)
        self._by_dtype = {}
        self.sgs(torch.float32 if A.dtype == torch.float32 else torch.float64)   # checks the diagonal now

    def sgs(self, dtype: torch.dtype) -> "_native.SgsPreconditioner":
        """The device set-up for the work dtype `dtype` (registered and colored on first use, then cached)."""
        S = self._by_dtype.get(dtype)
        if S is None:
            with torch.no_grad():
                S = _native.register_matrix(self.A, dtype).sgs()
            self._by_dtype[dtype] = S
        return S

    def __call__(self, r):
        if not isinstance(r, torch.Tensor):
            raise TypeError("SymmetricGaussSeidelPreconditioner applies to a single tensor")
        if not r.is_cuda:
            raise _native.NativeLibraryError("SymmetricGaussSeidelPreconditioner applies on the CUDA device "
                                             "(no CPU fallback)")
        wdt = torch.float32 if r.dtype == torch.float32 else torch.float64
        return self.sgs(wdt).apply(r.detach().reshape(-1).to(wdt)).reshape(r.shape)
