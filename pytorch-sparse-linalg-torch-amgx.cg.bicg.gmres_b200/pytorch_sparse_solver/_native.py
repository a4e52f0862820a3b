"""ctypes binding of libbk_krylov.so (C ABI declared in include/bk_krylov.h).

PyTorch is plumbing here: it owns device memory and the current stream; every numerical
operation of the Krylov loop happens inside the hand-written CUDA library.  There is no CPU
fallback: if the library is missing or there is no CUDA device, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from collections import OrderedDict
from pathlib import Path
from typing import Optional, Tuple

import torch

_LIB_NAME = "libbk_krylov.so"
_LIB_DIR = Path(__file__).resolve().parent / "_lib"

BK_F64, BK_F32 = 0, 1
BK_GMRES_BATCHED, BK_GMRES_INCREMENTAL = 0, 1
METHOD_CG, METHOD_BICGSTAB, METHOD_GMRES = 0, 1, 2
BK_ERR_ARG = -1


class NativeLibraryError(RuntimeError):
    """The CUDA library is missing/unloadable or reported an error."""


class bk_result(C.Structure):
    _fields_ = [
        ("iterations", C.c_int64),
        ("matvecs", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("info", C.c_int32),
        ("status", C.c_int32),
        ("final_residual", C.c_double),
        ("threshold", C.c_double),
        ("b_norm", C.c_double),
        ("x_norm", C.c_double),
        ("rr_last", C.c_double),
        ("loop_mode_used", C.c_int32),
        ("reserved0", C.c_int32),
        ("device_ms", C.c_double),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class bk_csr_info(C.Structure):
    _fields_ = [
        ("n", C.c_int64),
        ("nnz", C.c_int64),
        ("dtype", C.c_int32),
        ("kernel", C.c_int32),
        ("lanes_per_row", C.c_int32),
        ("max_row_nnz", C.c_int32),
        ("mean_row_nnz", C.c_double),
        ("bytes_matrix", C.c_int64),
        ("bytes_stream", C.c_int64),
    ]


# symbol -> (restype, argtypes); kept in one table so tests can check it against the header.
_VP = C.c_void_p
_SIGNATURES = {
    "bk_version": (C.c_int, []),
    "bk_last_error": (C.c_char_p, []),
    "bk_create": (C.c_int, [C.c_int, C.POINTER(_VP)]),
    "bk_destroy": (C.c_int, [_VP]),
    "bk_set_option": (C.c_int, [_VP, C.c_char_p, C.c_int64]),
    "bk_get_option": (C.c_int64, [_VP, C.c_char_p]),
    "bk_device_info": (C.c_int, [_VP, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bk_csr_create": (C.c_int, [_VP, C.c_int64, C.c_int64, _VP, _VP, C.c_int, _VP, C.c_int, C.c_int, _VP,
                                C.POINTER(_VP)]),
    "bk_csr_destroy": (C.c_int, [_VP]),
    "bk_csr_get_info": (C.c_int, [_VP, C.POINTER(bk_csr_info)]),
    "bk_csr_transpose": (C.c_int, [_VP, _VP, _VP, C.POINTER(_VP)]),
    "bk_csr_grad_pattern": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    "bk_csr_arrays": (C.c_int, [_VP, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_VP)]),
    "bk_checksum": (C.c_int, [_VP, _VP, C.c_int64, _VP, C.POINTER(C.c_uint64)]),
    "bk_spmv": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "bk_spmv_dot": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "bk_dot": (C.c_int, [_VP, C.c_int64, C.c_int, _VP, _VP, _VP, _VP]),
    "bk_nrm2": (C.c_int, [_VP, C.c_int64, C.c_int, _VP, _VP, _VP]),
    "bk_axpby": (C.c_int, [_VP, C.c_int64, C.c_int, C.c_double, _VP, C.c_double, _VP, _VP, _VP]),
    "bk_axpby_dev": (C.c_int, [_VP, C.c_int64, C.c_int, C.c_double, _VP, _VP, C.c_double, _VP, _VP, _VP, _VP]),
    "bk_div_scalar": (C.c_int, [_VP, C.c_int64, C.c_int, _VP, C.c_double, _VP, _VP]),
    "bk_block_apply": (C.c_int, [_VP, C.c_int64, C.c_int, C.c_int, _VP, _VP, _VP, _VP]),
    "bk_cdot": (C.c_int, [_VP, C.c_int64, _VP, _VP, _VP, _VP]),
    "bk_caxpby": (C.c_int, [_VP, C.c_int64, C.c_double, C.c_double, _VP, C.c_double, C.c_double, _VP, _VP, _VP]),
    "bk_cg": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64, C.POINTER(bk_result), _VP]),
    "bk_bicgstab": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64, C.POINTER(bk_result),
                              _VP]),
    "bk_gmres": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int64, C.c_int,
                           C.POINTER(bk_result), _VP]),
    "bk_solve_host": (C.c_int, [_VP, C.c_int, C.c_int64, C.c_int64, _VP, _VP, C.c_int, _VP, C.c_int, _VP, _VP,
                                C.c_int, C.c_double, C.c_double, C.c_int64, C.c_int, C.c_int, C.POINTER(bk_result)]),
    "bk_dist_unique_id": (C.c_int, [_VP]),
    "bk_dist_create": (C.c_int, [_VP, _VP, C.c_int, C.c_int, C.c_int64, C.c_int64, _VP, _VP, _VP, C.c_int64, _VP,
                                 C.c_int64, _VP, _VP, _VP, C.c_int64, C.c_int, _VP, _VP, _VP, _VP, C.c_int, _VP,
                                 C.POINTER(_VP)]),
    "bk_dist_destroy": (C.c_int, [_VP]),
    "bk_dist_set_extended": (C.c_int, [_VP, C.c_int64, _VP, _VP, _VP, _VP, C.c_int64, _VP, C.POINTER(C.c_int32)]),
    "bk_dist_cg_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_int64,
                                    C.POINTER(bk_result), _VP]),
    "bk_dist_bicgstab_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64,
                                          C.c_int64, C.POINTER(bk_result), _VP]),
    "bk_dist_gmres_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int64,
                                       C.c_int, C.c_int64, C.POINTER(bk_result), _VP]),
    "bk_dist_p2p_export": (C.c_int, [_VP, _VP]),
    "bk_dist_p2p_connect": (C.c_int, [_VP, _VP, _VP]),
    "bk_dist_spmv": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "bk_dist_cg": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_int64,
                             C.POINTER(bk_result), _VP]),
    "bk_csr_from_dense": (C.c_int, [_VP, C.c_int64, _VP, C.c_int64, C.c_int, C.c_int, _VP, C.POINTER(_VP)]),
    "bk_csr_from_coo": (C.c_int, [_VP, C.c_int64, C.c_int64, _VP, _VP, C.c_int, _VP, C.c_int, C.c_int, _VP,
                                  C.POINTER(_VP)]),
    "bk_cg_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64,
                               C.POINTER(bk_result), _VP]),
    "bk_bicgstab_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64,
                                     C.POINTER(bk_result), _VP]),
    "bk_gmres_jacobi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int64,
                                  C.c_int, C.POINTER(bk_result), _VP]),
    "bk_csr_diagonal": (C.c_int, [_VP, _VP, _VP, _VP]),
    "bk_sgs_create": (C.c_int, [_VP, _VP, _VP, C.POINTER(_VP)]),
    "bk_sgs_get_info": (C.c_int, [_VP, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "bk_sgs_colors": (C.c_int, [_VP, _VP, _VP]),
    "bk_sgs_apply": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "bk_cg_sgs": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64,
                            C.POINTER(bk_result), _VP]),
    "bk_bicgstab_sgs": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64,
                                  C.POINTER(bk_result), _VP]),
    "bk_gmres_sgs": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int64,
                               C.c_int, C.POINTER(bk_result), _VP]),
    "bk_dist_bicgstab": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_int64,
                                   C.POINTER(bk_result), _VP]),
    "bk_dist_gmres": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int64, C.c_int,
                                C.c_int64, C.POINTER(bk_result), _VP]),
}

_lib = None


def library_path() -> Path:
    return Path(os.environ.get("BK_KRYLOV_LIB", _LIB_DIR / _LIB_NAME))


def load_library():
    """dlopen the C-ABI library and attach signatures.  Raises NativeLibraryError when absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not path.exists():
        raise NativeLibraryError(
            f"{path} not found: build it with `python __graft_entry__.py` (or csrc/build.py). "
            "There is no CPU fallback for the module_a hot path.")
    try:
        lib = C.CDLL(str(path))
    except OSError as e:  # pragma: no cover
        raise NativeLibraryError(f"cannot load {path}: {e}") from e
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{path} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _check(rc: int, what: str):
    if rc != 0:
        msg = load_library().bk_last_error()
        raise NativeLibraryError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float64:
        return BK_F64
    if dt == torch.float32:
        return BK_F32
    raise TypeError(f"module_a native path supports float64/float32, got {dt}")


class Handle:
    """One bk_handle per CUDA device (created lazily, lives for the process)."""

    _by_device = {}

    def __init__(self, device_index: int):
        lib = load_library()
        if not torch.cuda.is_available():
            raise NativeLibraryError("a CUDA device is required: module_a has no CPU fallback in this build")
        torch.cuda.init()
        with torch.cuda.device(device_index):
            torch.cuda.current_stream()  # make sure the primary context exists
            p = _VP()
            _check(lib.bk_create(device_index, C.byref(p)), "bk_create")
        self.ptr = p
        self.device_index = device_index
        self.lib = lib

    @classmethod
    def get(cls, device) -> "Handle":
        load_library()
        if not torch.cuda.is_available():
            raise NativeLibraryError("a CUDA device is required: module_a has no CPU fallback in this build")
        idx = torch.device(device).index
        if idx is None:
            idx = torch.cuda.current_device()
        h = cls._by_device.get(idx)
        if h is None:
            h = cls(idx)
            cls._by_device[idx] = h
        return h

    def set_option(self, key: str, value: int):
        _check(self.lib.bk_set_option(self.ptr, key.encode(), int(value)), f"bk_set_option({key})")

    def get_option(self, key: str) -> int:
        return int(self.lib.bk_get_option(self.ptr, key.encode()))

    def device_info(self):
        sms, l2, mem = C.c_int32(), C.c_int64(), C.c_int64()
        _check(self.lib.bk_device_info(self.ptr, C.byref(sms), C.byref(l2), C.byref(mem)), "bk_device_info")
        return {"num_sms": sms.value, "l2_bytes": l2.value, "mem_bytes": mem.value}


class _DevPtr:
    """Minimal __cuda_array_interface__ carrier for a borrowed device pointer."""

    def __init__(self, ptr: int, count: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": typestr, "data": (ptr, False), "version": 2}


class CsrMatrix:
    """A registered CSR matrix.  Holds references to the torch tensors whose memory the library borrows."""

    def __init__(self, handle: Handle, crow: torch.Tensor, col: torch.Tensor, val: torch.Tensor, n: int):
        assert crow.is_cuda and col.is_cuda and val.is_cuda
        crow = crow.contiguous()
        col = col.contiguous()
        val = val.contiguous()
        if crow.dtype not in (torch.int32, torch.int64) or col.dtype != crow.dtype:
            raise TypeError("CSR indices must be int32 or int64")
        self.handle = handle
        self.n = int(n)
        self.nnz = int(val.numel())
        self.dtype = val.dtype
        self.device = val.device
        # what the library BORROWS must stay alive: the values always, the index arrays only when they are int32
        # (int64 indices are narrowed into a library-owned copy at registration)
        self._keep = (val,) if crow.dtype == torch.int64 else (crow, col, val)
        p = _VP()
        with torch.cuda.device(self.device):
            _check(handle.lib.bk_csr_create(handle.ptr, self.n, self.nnz, crow.data_ptr(), col.data_ptr(),
                                            32 if crow.dtype == torch.int32 else 64, val.data_ptr(),
                                            _dtype_code(val.dtype), 0, _stream_ptr(self.device), C.byref(p)),
                   "bk_csr_create")
        self.ptr = p
        self._owned = True
        self._transpose = None
        self._sgs = None
        self._finalizer = weakref.finalize(self, CsrMatrix._destroy, handle.lib, p)

    @staticmethod
    def _destroy(lib, p):
        try:
            lib.bk_csr_destroy(p)
        except Exception:  # pragma: no cover
            pass

    @classmethod
    def _wrap(cls, handle: Handle, ptr, n, nnz, dtype, device, keep):
        obj = cls.__new__(cls)
        obj.handle, obj.ptr, obj.n, obj.nnz, obj.dtype, obj.device = handle, ptr, n, nnz, dtype, device
        obj._keep = keep
        obj._owned = False
        obj._transpose = None
        obj._sgs = None
        return obj

    def info(self) -> dict:
        out = bk_csr_info()
        _check(self.handle.lib.bk_csr_get_info(self.ptr, C.byref(out)), "bk_csr_get_info")
        return {k: getattr(out, k) for k, _ in out._fields_}

    def transpose(self) -> "CsrMatrix":
        """Cached A^T (owned by this matrix on the C side)."""
        if self._transpose is None:
            p = _VP()
            with torch.cuda.device(self.device):
                _check(self.handle.lib.bk_csr_transpose(self.handle.ptr, self.ptr, _stream_ptr(self.device),
                                                        C.byref(p)), "bk_csr_transpose")
            self._transpose = CsrMatrix._wrap(self.handle, p, self.n, self.nnz, self.dtype, self.device, (self,))
        return self._transpose

    def sgs(self) -> "SgsPreconditioner":
        """Cached multicolor symmetric Gauss-Seidel set-up of this matrix (owned by it on the C side).
        ValueError when a row stores no nonzero diagonal."""
        if self._sgs is None:
            p = _VP()
            with torch.cuda.device(self.device):
                rc = self.handle.lib.bk_sgs_create(self.handle.ptr, self.ptr, _stream_ptr(self.device), C.byref(p))
            if rc == BK_ERR_ARG:
                msg = self.handle.lib.bk_last_error()
                raise ValueError(msg.decode() if msg else "bk_sgs_create: invalid matrix")
            _check(rc, "bk_sgs_create")
            self._sgs = SgsPreconditioner(self, p)
        return self._sgs

    def arrays(self) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Copy the (int32) CSR arrays of this matrix out as torch tensors (testing / debugging)."""
        rp, cp, vp = _VP(), _VP(), _VP()
        _check(self.handle.lib.bk_csr_arrays(self.ptr, C.byref(rp), C.byref(cp), C.byref(vp)), "bk_csr_arrays")
        torch.cuda.synchronize(self.device)

        def view(ptr, count, typestr, dtype):
            if count == 0:
                return torch.empty(0, dtype=dtype, device=self.device)
            return torch.as_tensor(_DevPtr(ptr.value, count, typestr), device=self.device).clone()

        crow = view(rp, self.n + 1, "<i4", torch.int32)
        col = view(cp, self.nnz, "<i4", torch.int32)
        val = view(vp, self.nnz, "<f8" if self.dtype == torch.float64 else "<f4", self.dtype)
        return crow, col, val

    # ---- building blocks -------------------------------------------------------------------
    def _vec(self, v: torch.Tensor) -> torch.Tensor:
        if v.dtype != self.dtype or not v.is_cuda or v.numel() != self.n:
            raise ValueError(f"vector must be a CUDA {self.dtype} tensor of {self.n} elements")
        return v.contiguous()

    def spmv(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        x = self._vec(x)
        y = torch.empty_like(x) if out is None else out
        with torch.cuda.device(self.device):
            _check(self.handle.lib.bk_spmv(self.handle.ptr, self.ptr, x.data_ptr(), y.data_ptr(),
                                           _stream_ptr(self.device)), "bk_spmv")
        return y

    def spmv_dot(self, x: torch.Tensor, w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        x = self._vec(x)
        w = self._vec(w)
        y = torch.empty_like(x)
        d = torch.empty(1, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.handle.lib.bk_spmv_dot(self.handle.ptr, self.ptr, x.data_ptr(), y.data_ptr(), w.data_ptr(),
                                               d.data_ptr(), _stream_ptr(self.device)), "bk_spmv_dot")
        return y, d[0]

    def grad_pattern(self, g: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        """-g_i x_j on the stored pattern (values in this matrix's CSR order)."""
        g, x = self._vec(g), self._vec(x)
        out = torch.empty(self.nnz, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.handle.lib.bk_csr_grad_pattern(self.handle.ptr, self.ptr, g.data_ptr(), x.data_ptr(),
                                                       out.data_ptr(), _stream_ptr(self.device)), "bk_csr_grad_pattern")
        return out

    # ---- solvers -----------------------------------------------------------------------------
    def _solve(self, which: str, b: torch.Tensor, x0: Optional[torch.Tensor], *args) -> Tuple[torch.Tensor, dict]:
        b = self._vec(b)
        if x0 is None:
            x = torch.empty_like(b)
            has_x0 = 0
        else:
            x = self._vec(x0).clone()
            has_x0 = 1
        res = bk_result()
        lib = self.handle.lib
        with torch.cuda.device(self.device):
            s = _stream_ptr(self.device)
            if which == "cg":
                tol, atol, maxiter = args
                rc = lib.bk_cg(self.handle.ptr, self.ptr, b.data_ptr(), x.data_ptr(), has_x0, tol, atol, maxiter,
                               C.byref(res), s)
            elif which == "bicgstab":
                tol, atol, maxiter = args
                rc = lib.bk_bicgstab(self.handle.ptr, self.ptr, b.data_ptr(), x.data_ptr(), has_x0, tol, atol,
                                     maxiter, C.byref(res), s)
            elif which == "gmres":
                tol_eff, atol_eff, restart, maxiter, method = args
                rc = lib.bk_gmres(self.handle.ptr, self.ptr, b.data_ptr(), x.data_ptr(), has_x0, tol_eff, atol_eff,
                                  restart, maxiter, method, C.byref(res), s)
            else:  # pragma: no cover
                raise ValueError(which)
        _check(rc, f"bk_{which}")
        return x, res.as_dict()

    def cg(self, b, x0, tol, atol, maxiter):
        return self._solve("cg", b, x0, float(tol), float(atol), -1 if maxiter is None else int(maxiter))

    def bicgstab(self, b, x0, tol, atol, maxiter):
        return self._solve("bicgstab", b, x0, float(tol), float(atol), -1 if maxiter is None else int(maxiter))

    def gmres(self, b, x0, tol_eff, atol_eff, restart, maxiter, method):
        return self._solve("gmres", b, x0, float(tol_eff), float(atol_eff), int(restart),
                           -1 if maxiter is None else int(maxiter), int(method))

    def diagonal(self) -> torch.Tensor:
        """diag(A) as a device vector of the matrix dtype (bk_csr_diagonal)."""
        out = torch.empty(self.n, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.handle.lib.bk_csr_diagonal(self.handle.ptr, self.ptr, out.data_ptr(),
                                                   _stream_ptr(self.device)), "bk_csr_diagonal")
        return out

    def _solve_jacobi(self, fn_name: str, diag: torch.Tensor, b, x0, tol, atol, maxiter):
        d = self._vec(diag)
        b = self._vec(b)
        if x0 is None:
            x, has_x0 = torch.empty_like(b), 0
        else:
            x, has_x0 = self._vec(x0).clone(), 1
        res = bk_result()
        with torch.cuda.device(self.device):
            rc = getattr(self.handle.lib, fn_name)(self.handle.ptr, self.ptr, d.data_ptr(), b.data_ptr(), x.data_ptr(),
                                                   has_x0, float(tol), float(atol),
                                                   -1 if maxiter is None else int(maxiter), C.byref(res),
                                                   _stream_ptr(self.device))
        _check(rc, fn_name)
        return x, res.as_dict()

    def cg_jacobi(self, diag: torch.Tensor, b, x0, tol, atol, maxiter):
        """CG preconditioned with M = (r -> r / diag), all on the device (bk_cg_jacobi)."""
        return self._solve_jacobi("bk_cg_jacobi", diag, b, x0, tol, atol, maxiter)

    def gmres_jacobi(self, diag: torch.Tensor, b, x0, tol_eff, atol_eff, restart, maxiter, method):
        """GMRES left-preconditioned with M = (v -> v / diag), all on the device (bk_gmres_jacobi)."""
        d = self._vec(diag)
        b = self._vec(b)
        if x0 is None:
            x, has_x0 = torch.empty_like(b), 0
        else:
            x, has_x0 = self._vec(x0).clone(), 1
        res = bk_result()
        with torch.cuda.device(self.device):
            rc = self.handle.lib.bk_gmres_jacobi(self.handle.ptr, self.ptr, d.data_ptr(), b.data_ptr(), x.data_ptr(),
                                                 has_x0, float(tol_eff), float(atol_eff), int(restart),
                                                 -1 if maxiter is None else int(maxiter), int(method), C.byref(res),
                                                 _stream_ptr(self.device))
        _check(rc, "bk_gmres_jacobi")
        return x, res.as_dict()

    def bicgstab_jacobi(self, diag: torch.Tensor, b, x0, tol, atol, maxiter):
        """BiCGStab right-preconditioned with M = (v -> v / diag), all on the device (bk_bicgstab_jacobi)."""
        return self._solve_jacobi("bk_bicgstab_jacobi", diag, b, x0, tol, atol, maxiter)

    def _solve_sgs(self, fn_name: str, S: "SgsPreconditioner", b, x0, *args):
        if S.n != self.n or S.dtype != self.dtype or S.device != self.device:
            raise ValueError("the preconditioner was built for another order, dtype or device")
        b = self._vec(b)
        if x0 is None:
            x, has_x0 = torch.empty_like(b), 0
        else:
            x, has_x0 = self._vec(x0).clone(), 1
        res = bk_result()
        with torch.cuda.device(self.device):
            rc = getattr(self.handle.lib, fn_name)(self.handle.ptr, self.ptr, S.ptr, b.data_ptr(), x.data_ptr(),
                                                   has_x0, *args, C.byref(res), _stream_ptr(self.device))
        _check(rc, fn_name)
        return x, res.as_dict()

    def cg_sgs(self, S: "SgsPreconditioner", b, x0, tol, atol, maxiter):
        """CG preconditioned with multicolor symmetric Gauss-Seidel, all on the device (bk_cg_sgs)."""
        return self._solve_sgs("bk_cg_sgs", S, b, x0, float(tol), float(atol), -1 if maxiter is None else int(maxiter))

    def bicgstab_sgs(self, S: "SgsPreconditioner", b, x0, tol, atol, maxiter):
        """BiCGStab right-preconditioned with symmetric Gauss-Seidel (bk_bicgstab_sgs)."""
        return self._solve_sgs("bk_bicgstab_sgs", S, b, x0, float(tol), float(atol),
                               -1 if maxiter is None else int(maxiter))

    def gmres_sgs(self, S: "SgsPreconditioner", b, x0, tol_eff, atol_eff, restart, maxiter, method):
        """GMRES left-preconditioned with symmetric Gauss-Seidel (bk_gmres_sgs)."""
        return self._solve_sgs("bk_gmres_sgs", S, b, x0, float(tol_eff), float(atol_eff), int(restart),
                               -1 if maxiter is None else int(maxiter), int(method))


class SgsPreconditioner:
    """A bk_sgs of a registered matrix (freed with it; this object keeps the matrix alive)."""

    def __init__(self, mat: CsrMatrix, ptr):
        self.mat, self.ptr = mat, ptr
        self.n, self.dtype, self.device = mat.n, mat.dtype, mat.device
        nc, rounds = C.c_int32(), C.c_int32()
        _check(mat.handle.lib.bk_sgs_get_info(ptr, C.byref(nc), C.byref(rounds)), "bk_sgs_get_info")
        self.num_colors, self.rounds = nc.value, rounds.value

    def colors(self) -> torch.Tensor:
        """The color of every row (uint8, on the device)."""
        out = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.mat.handle.lib.bk_sgs_colors(self.ptr, out.data_ptr(), _stream_ptr(self.device)),
                   "bk_sgs_colors")
        return out

    def apply(self, r: torch.Tensor) -> torch.Tensor:
        """z = M r (bk_sgs_apply)."""
        r = self.mat._vec(r)
        z = torch.empty_like(r)
        with torch.cuda.device(self.device):
            _check(self.mat.handle.lib.bk_sgs_apply(self.mat.handle.ptr, self.ptr, r.data_ptr(), z.data_ptr(),
                                                    _stream_ptr(self.device)), "bk_sgs_apply")
        return z


# ---- building-block vector ops (deterministic reductions) ------------------------------------------
def dot(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    h = Handle.get(x.device)
    x = x.contiguous()
    y = y.contiguous()
    out = torch.empty(1, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _check(h.lib.bk_dot(h.ptr, x.numel(), _dtype_code(x.dtype), x.data_ptr(), y.data_ptr(), out.data_ptr(),
                            _stream_ptr(x.device)), "bk_dot")
    return out[0]


def nrm2(x: torch.Tensor) -> torch.Tensor:
    h = Handle.get(x.device)
    x = x.contiguous()
    out = torch.empty(1, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _check(h.lib.bk_nrm2(h.ptr, x.numel(), _dtype_code(x.dtype), x.data_ptr(), out.data_ptr(),
                             _stream_ptr(x.device)), "bk_nrm2")
    return out[0]


def axpby(a: float, x: torch.Tensor, b: float, y: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    h = Handle.get(x.device)
    x = x.contiguous()
    y = y.contiguous()
    z = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        _check(h.lib.bk_axpby(h.ptr, x.numel(), _dtype_code(x.dtype), float(a), x.data_ptr(), float(b), y.data_ptr(),
                              z.data_ptr(), _stream_ptr(x.device)), "bk_axpby")
    return z


def axpby_dev(sa: float, a: Optional[torch.Tensor], x: torch.Tensor, sb: float, b: Optional[torch.Tensor],
              y: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """z = (sa * a) x + (sb * b) y with a, b 0-dim fp64 DEVICE tensors (None = 1): no host sync (bk_axpby_dev)."""
    h = Handle.get(x.device)
    x = x.contiguous()
    y = y.contiguous()
    z = torch.empty_like(x) if out is None else out
    for t in (a, b):
        if t is not None and (t.dtype != torch.float64 or not t.is_cuda):
            raise ValueError("device scalars must be fp64 CUDA tensors")
    with torch.cuda.device(x.device):
        _check(h.lib.bk_axpby_dev(h.ptr, x.numel(), _dtype_code(x.dtype), float(sa), None if a is None else a.data_ptr(),
                                  x.data_ptr(), float(sb), None if b is None else b.data_ptr(), y.data_ptr(),
                                  z.data_ptr(), _stream_ptr(x.device)), "bk_axpby_dev")
    return z


def div_scalar(x: torch.Tensor, d: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """z = x / d (true division; bk_div_scalar)."""
    h = Handle.get(x.device)
    x = x.contiguous()
    z = torch.empty_like(x) if out is None else out
    with torch.cuda.device(x.device):
        _check(h.lib.bk_div_scalar(h.ptr, x.numel(), _dtype_code(x.dtype), x.data_ptr(), float(d), z.data_ptr(),
                                   _stream_ptr(x.device)), "bk_div_scalar")
    return z


def block_apply(inv: torch.Tensor, r: torch.Tensor, bs: int) -> torch.Tensor:
    """z = blockdiag(inv) r (bk_block_apply); inv: [nblocks, bs, bs] contiguous, same dtype / device as r."""
    h = Handle.get(r.device)
    r = r.contiguous()
    z = torch.empty_like(r)
    with torch.cuda.device(r.device):
        _check(h.lib.bk_block_apply(h.ptr, r.numel(), int(bs), _dtype_code(r.dtype), inv.data_ptr(), r.data_ptr(),
                                    z.data_ptr(), _stream_ptr(r.device)), "bk_block_apply")
    return z


def cdot(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """sum conj(x) y for complex128 vectors given as interleaved fp64 (2n) tensors; returns a device tensor [re, im]."""
    h = Handle.get(x.device)
    out = torch.empty(2, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _check(h.lib.bk_cdot(h.ptr, x.numel() // 2, x.data_ptr(), y.data_ptr(), out.data_ptr(), _stream_ptr(x.device)),
               "bk_cdot")
    return out


def caxpby(a: complex, x: torch.Tensor, b: complex, y: torch.Tensor) -> torch.Tensor:
    """z = a x + b y for complex128 vectors given as interleaved fp64 (2n) tensors, complex scalars a, b."""
    h = Handle.get(x.device)
    z = torch.empty_like(x)
    a, b = complex(a), complex(b)
    with torch.cuda.device(x.device):
        _check(h.lib.bk_caxpby(h.ptr, x.numel() // 2, a.real, a.imag, x.data_ptr(), b.real, b.imag, y.data_ptr(),
                               z.data_ptr(), _stream_ptr(x.device)), "bk_caxpby")
    return z


# ---- matrix ingestion + cache ---------------------------------------------------------------------
# Registrations are cached per (layout, storage pointers, shape, dtypes, device).  torch offers no reliable way to
# notice that a user changed `vals` in place (the version counter of a CSR / COO wrapper's value tensor does not move
# when the tensor it was built from is written to, and `.data` writes never bump it), and the registration holds
# value-dependent artefacts (the pattern / pair dictionaries of kernels 5 and 6, tail copies, the cached transpose,
# dtype-converted copies).  A hit is therefore VALIDATED: the library checksums the arrays as they are now
# (bk_checksum, one pass, ~0.3 ms for a 256^3 matrix) and a mismatch re-registers the matrix.  BK_CACHE_VALIDATE=0
# turns the check off for callers who promise not to mutate registered matrices; `invalidate(A)` drops an entry.
# Entries hold only what the library borrows (never the source tensor itself): when the source tensor has been
# garbage-collected at most ONE such orphan is kept (the pattern `solve(torch.sparse_csr_tensor(...), b)` re-wraps the
# same storages on every call), so a loop over distinct large systems does not pin their memory.
_CACHE: "OrderedDict[tuple, dict]" = OrderedDict()
_CACHE_MAX = 8
_CACHE_MAX_ORPHANS = 1


def _csr_components(A: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """dense / COO / CSR torch tensor -> (crow, col, values).  Setup-time torch calls (not the hot path)."""
    if A.layout == torch.sparse_csr:
        return A.crow_indices(), A.col_indices(), A.values()
    if A.layout == torch.sparse_coo:
        A = A.coalesce().to_sparse_csr()
        return A.crow_indices(), A.col_indices(), A.values()
    if A.layout == torch.strided:
        A = A.to_sparse_csr()
        return A.crow_indices(), A.col_indices(), A.values()
    A = A.to_sparse_csr()
    return A.crow_indices(), A.col_indices(), A.values()


def _ingest_native(A: torch.Tensor, dtype: torch.dtype) -> Optional[CsrMatrix]:
    """dense / COO CUDA tensors -> CsrMatrix through the library's own conversion kernels (bk_csr_from_dense /
    bk_csr_from_coo).  Returns None for layouts / dtypes those entry points do not take (handled via torch)."""
    if A.layout not in (torch.strided, torch.sparse_coo) or A.dtype not in (torch.float64, torch.float32):
        return None
    if os.environ.get("BK_NATIVE_INGEST", "1") == "0":
        return None
    h = Handle.get(A.device)
    n = int(A.shape[0])
    p = _VP()
    with torch.no_grad(), torch.cuda.device(A.device):
        s = _stream_ptr(A.device)
        if A.layout == torch.strided:
            D = A.detach()
            if D.stride(1) != 1 and n > 1:
                D = D.contiguous()
            ld = int(D.stride(0)) if n > 1 else max(n, 1)
            if ld < n:
                D, ld = D.contiguous(), n
            _check(h.lib.bk_csr_from_dense(h.ptr, n, D.data_ptr(), ld, _dtype_code(D.dtype), _dtype_code(dtype), s,
                                           C.byref(p)), "bk_csr_from_dense")
        else:
            idx = A.detach()._indices()
            val = A.detach()._values().contiguous()
            rows, cols = idx[0].contiguous(), idx[1].contiguous()
            _check(h.lib.bk_csr_from_coo(h.ptr, n, int(val.numel()), rows.data_ptr(), cols.data_ptr(),
                                         64 if rows.dtype == torch.int64 else 32, val.data_ptr(),
                                         _dtype_code(val.dtype), _dtype_code(dtype), s, C.byref(p)), "bk_csr_from_coo")
        torch.cuda.current_stream(A.device).synchronize()
    m = CsrMatrix._wrap(h, p, n, 0, dtype, A.device, ())   # the library owns every array: nothing to keep alive
    m._owned = True
    m._finalizer = weakref.finalize(m, CsrMatrix._destroy, h.lib, p)
    m.nnz = int(m.info()["nnz"])
    return m


def checksum(t: torch.Tensor) -> int:
    """bk_checksum of a CUDA tensor's bytes (contiguous; 4-byte aligned size)."""
    h = Handle.get(t.device)
    t = t.contiguous()
    out = C.c_uint64(0)
    with torch.cuda.device(t.device):
        _check(h.lib.bk_checksum(h.ptr, t.data_ptr(), t.numel() * t.element_size(), _stream_ptr(t.device),
                                 C.byref(out)), "bk_checksum")
    return int(out.value)


def _key_and_parts(A: torch.Tensor, dtype: torch.dtype):
    """Cache key + the tensors whose CONTENT defines the registration (checksummed on a hit)."""
    if A.layout == torch.sparse_csr:
        crow, col, v = A.crow_indices(), A.col_indices(), A.values()
        key = ("csr", crow.data_ptr(), col.data_ptr(), v.data_ptr(), tuple(A.shape), v.numel(), crow.dtype, v.dtype,
               dtype, A.device.index)
        return key, (crow, col, v)
    if A.layout == torch.sparse_coo:
        idx, v = A._indices(), A._values()
        key = ("coo", idx.data_ptr(), v.data_ptr(), tuple(A.shape), v.numel(), v.dtype, dtype, A.device.index,
               A.is_coalesced())
        return key, (idx, v)
    key = ("dense", A.data_ptr(), tuple(A.shape), tuple(A.stride()), A.dtype, dtype, A.device.index)
    return key, (A.detach(),)


def _content_sum(parts) -> Optional[int]:
    if os.environ.get("BK_CACHE_VALIDATE", "1") == "0":
        return None
    acc = 0
    for i, t in enumerate(parts):
        if t.numel() == 0:
            continue
        if t.element_size() % 4 != 0:      # exotic dtypes: view through a 4-byte-aligned copy
            t = t.to(torch.float32)
        acc ^= (checksum(t) * (2 * i + 1)) & 0xFFFFFFFFFFFFFFFF
    return acc


def _prune_cache():
    orphans = [k for k, e in _CACHE.items() if e["src"]() is None]
    for k in orphans[:max(0, len(orphans) - _CACHE_MAX_ORPHANS)]:
        _CACHE.pop(k, None)
    while len(_CACHE) > _CACHE_MAX:
        _CACHE.popitem(last=False)


def register_matrix(A: torch.Tensor, dtype: torch.dtype = torch.float64) -> CsrMatrix:
    """Register a 2-D CUDA tensor with the library (cached per storage, validated by content — see above)."""
    if not A.is_cuda:
        raise NativeLibraryError("register_matrix expects a CUDA tensor")
    key, parts = _key_and_parts(A, dtype)
    hit = _CACHE.get(key)
    csum = _content_sum(parts)
    if hit is not None:
        if csum is None or hit["sum"] is None or hit["sum"] == csum:
            _CACHE.move_to_end(key)
            if hit["src"]() is None:
                try:
                    hit["src"] = weakref.ref(A)
                except TypeError:  # pragma: no cover
                    pass
            return hit["m"]
        _CACHE.pop(key)            # same storage, different content: the user updated the matrix in place
    m = _ingest_native(A, dtype)
    if m is None:
        with torch.no_grad():
            crow, col, val = _csr_components(A.detach())
            if val.dtype != dtype:
                val = val.to(dtype)
        m = CsrMatrix(Handle.get(A.device), crow, col, val, A.shape[0])
    try:
        src = weakref.ref(A)
    except TypeError:  # pragma: no cover
        src = (lambda: None)
    _CACHE[key] = {"m": m, "sum": csum, "src": src}
    _prune_cache()
    return m


def invalidate(A: Optional[torch.Tensor] = None):
    """Drop the cached registration(s) of `A` (all dtypes), or of every matrix when A is None.  Only needed with
    BK_CACHE_VALIDATE=0; with validation on, in-place updates of a registered matrix are detected by content."""
    if A is None:
        _CACHE.clear()
        return
    for dt in (torch.float64, torch.float32):
        _CACHE.pop(_key_and_parts(A, dt)[0], None)


def clear_cache():
    _CACHE.clear()


def solve_host(method: int, crow: torch.Tensor, col: torch.Tensor, val: torch.Tensor, b: torch.Tensor,
               x0: Optional[torch.Tensor], tol: float, atol: float, maxiter: Optional[int], restart: int = 20,
               gmres_method: int = BK_GMRES_BATCHED, device: Optional[int] = None) -> Tuple[torch.Tensor, dict]:
    """End-to-end solve from HOST buffers: H2D of matrix and b, the device loop, D2H of x (bk_solve_host)."""
    for t in (crow, col, val, b):
        if t.is_cuda:
            raise ValueError("solve_host takes CPU tensors")
    load_library()
    if not torch.cuda.is_available():
        raise NativeLibraryError("a CUDA device is required: module_a has no CPU fallback in this build")
    h = Handle.get(torch.device("cuda", torch.cuda.current_device() if device is None else device))
    crow, col, val, b = crow.contiguous(), col.contiguous(), val.contiguous(), b.contiguous()
    n = b.numel()
    # pinned inputs get a pinned result buffer (torch's caching host allocator recycles it between solves): the D2H
    # copy of x then runs at full PCIe speed instead of through pageable, never-touched memory
    pinned = b.is_pinned()
    if x0 is None:
        x = torch.empty(b.shape, dtype=b.dtype, pin_memory=pinned)
        has_x0 = 0
    else:
        x = torch.empty(b.shape, dtype=b.dtype, pin_memory=pinned)
        x.copy_(x0.to(b.dtype).reshape(b.shape))
        has_x0 = 1
    res = bk_result()
    _check(h.lib.bk_solve_host(h.ptr, int(method), n, val.numel(), crow.data_ptr(), col.data_ptr(),
                               32 if crow.dtype == torch.int32 else 64, val.data_ptr(), _dtype_code(val.dtype),
                               b.data_ptr(), x.data_ptr(), has_x0, float(tol), float(atol),
                               -1 if maxiter is None else int(maxiter), int(restart), int(gmres_method),
                               C.byref(res)), "bk_solve_host")
    return x, res.as_dict()
