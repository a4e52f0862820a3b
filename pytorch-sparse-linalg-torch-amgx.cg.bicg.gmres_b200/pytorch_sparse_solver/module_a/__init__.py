"""Module A — JAX-style Krylov solvers (cg, bicgstab, gmres) behind the reference's API, running on the
B200-native CUDA library.  Same exports as the reference module_a/__init__.py:40-63."""
from .krylov import (
    cg, bicgstab, gmres,
    cg_differentiable, bicgstab_differentiable, gmres_differentiable,
    LinearSolveFunction,
)
from .preconditioners import BlockJacobiPreconditioner, JacobiPreconditioner, SymmetricGaussSeidelPreconditioner
from .mixed_precision import refined_solve
from .torch_tree_util import tree_leaves, tree_map, tree_flatten, tree_unflatten, Partial

__all__ = [
    'cg', 'bicgstab', 'gmres',
    'cg_differentiable', 'bicgstab_differentiable', 'gmres_differentiable',
    'LinearSolveFunction',
    'JacobiPreconditioner',   # addition: built-in M that keeps cg() on the device (SURVEY §8f-1)
    'BlockJacobiPreconditioner',   # addition: block-diagonal M applied by one library kernel
    'SymmetricGaussSeidelPreconditioner',   # addition: multicolor symmetric Gauss-Seidel M, on the device
    'refined_solve',          # addition: mixed-precision iterative refinement (SURVEY §8f-4)
    'tree_leaves', 'tree_map', 'tree_flatten', 'tree_unflatten', 'Partial',
]

__version__ = '1.0.0'
