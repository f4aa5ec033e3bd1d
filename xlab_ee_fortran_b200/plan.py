"""Batched device API (Part 2 of include/xee_b200.h) on torch CUDA tensors.

torch is plumbing only here: device memory and streams.  Every kernel is ours (csrc/*.cu),
reached through the C-ABI with raw device pointers.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib

F32, F64 = 0, 1
ARITH_STRICT, ARITH_FAST = 0, 1
JACOBI, CHEBYSHEV, LINE_JACOBI, LINE_CHEBYSHEV, LINE2_JACOBI, LINE2_CHEBYSHEV = 0, 1, 2, 3, 4, 5
LINE_BICGSTAB, LINE2_BICGSTAB, LINE2_MIXED = 6, 7, 8
METHODS = {"jacobi": JACOBI, "chebyshev": CHEBYSHEV, "line_jacobi": LINE_JACOBI, "line_chebyshev": LINE_CHEBYSHEV,
           "line2_jacobi": LINE2_JACOBI, "line2_chebyshev": LINE2_CHEBYSHEV, "line_bicgstab": LINE_BICGSTAB,
           "line2_bicgstab": LINE2_BICGSTAB, "line2_mixed": LINE2_MIXED}


class _PlanDesc(C.Structure):
    _fields_ = [("dtype", C.c_int), ("nx", C.c_int), ("ny", C.c_int), ("nbatch", C.c_int), ("shared_coe", C.c_int),
                ("arith", C.c_int), ("method", C.c_int), ("device", C.c_int), ("kernel", C.c_int)]


class _SolveParams(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("check_step", C.c_int), ("converge_time", C.c_int), ("lost_rate", C.c_int),
                ("r1", C.c_double), ("r2", C.c_double), ("alpha", C.c_double), ("r1_per_solve", C.c_void_p),
                ("rho_jacobi", C.c_double), ("detect_explode", C.c_int), ("sync_every", C.c_int), ("stall_checks", C.c_int)]


@dataclass
class SolveParams:
    """Arguments of solve_elliptic (elliptic_tools.f90:93-95) for a whole batch."""
    max_iter: int = 100000
    check_step: int = 100
    converge_time: int = 10
    lost_rate: int = 5
    r1: float = 0.0
    r2: float = 0.0
    alpha: float = 1.0
    r1_per_solve: object = None     # optional torch tensor [nbatch]
    rho_jacobi: float = 0.0
    detect_explode: bool = False
    sync_every: int = 1
    stall_checks: int = 0           # >0: stop with err bit 4 when the residual stops improving (not in the reference)


def _torch():
    import torch
    return torch


class Plan:
    """One operator geometry (nx, ny, dtype) and batch size; owns the planar operator and scratch."""

    def __init__(self, nx, ny, nbatch=1, dtype="f64", shared_coe=True, arith="strict", method="jacobi", device=None,
                 kernel=0):
        _lib.require_gpu()
        torch = _torch()
        self.torch_dtype = torch.float64 if dtype in ("f64", torch.float64, np.float64) else torch.float32
        self.dtype = F64 if self.torch_dtype == torch.float64 else F32
        self.nx, self.ny, self.nbatch, self.shared_coe = int(nx), int(ny), int(nbatch), bool(shared_coe)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        d = _PlanDesc(self.dtype, self.nx, self.ny, self.nbatch, int(self.shared_coe),
                      ARITH_STRICT if arith == "strict" else ARITH_FAST,
                      METHODS[method], self.device.index, int(kernel))
        self._h = C.c_void_p()
        L = _lib.lib()
        with torch.cuda.device(self.device):
            _lib.check(L.xee_plan_create(C.byref(d), C.byref(self._h)), "plan_create")

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.lib().xee_plan_destroy(self._h)
            self._h = None

    __del__ = close

    # ---- operator
    def _chk(self, t, shape=None):
        torch = _torch()
        assert t.is_cuda and t.dtype == self.torch_dtype and t.is_contiguous(), "contiguous CUDA tensor of the plan dtype required"
        if shape is not None:
            assert tuple(t.shape) == tuple(shape), (tuple(t.shape), shape)
        return C.c_void_p(t.data_ptr())

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def set_coe_aos(self, coe):
        """coe: the reference's coe(9,nx,ny) as (ny,nx,9) [or (nbatch,ny,nx,9)] numpy array or CUDA tensor."""
        torch = _torch()
        sets = () if self.shared_coe else (self.nbatch,)
        L = _lib.lib()
        if isinstance(coe, np.ndarray):
            npdt = np.float64 if self.dtype == F64 else np.float32
            coe = np.ascontiguousarray(coe, npdt)
            assert coe.shape == sets + (self.ny, self.nx, 9)
            _lib.check(L.xee_plan_set_coe_aos_host(self._h, coe.ctypes.data_as(C.c_void_p)), "set_coe_aos_host")
        else:
            torch.cuda.current_stream(self.device).synchronize()
            _lib.check(L.xee_plan_set_coe_aos_dev(self._h, self._chk(coe, sets + (self.ny, self.nx, 9))), "set_coe_aos_dev")

    def set_abc(self, a, b, c, dx, dy):
        """K1+K2 on device from the reference-shaped a (ny-2,nx-1), b (ny-1,nx-1), c (ny-1,nx-2) CUDA tensors."""
        torch = _torch()
        sets = () if self.shared_coe else (self.nbatch,)
        torch.cuda.current_stream(self.device).synchronize()
        _lib.check(_lib.lib().xee_plan_set_abc_dev(
            self._h, self._chk(a, sets + (self.ny - 2, self.nx - 1)), self._chk(b, sets + (self.ny - 1, self.nx - 1)),
            self._chk(c, sets + (self.ny - 1, self.nx - 2)), C.c_double(dx), C.c_double(dy)), "set_abc_dev")

    # ---- solves
    def _prm(self, p: SolveParams):
        q = _SolveParams(p.max_iter, p.check_step, p.converge_time, p.lost_rate, p.r1, p.r2, p.alpha, None,
                         p.rho_jacobi, int(p.detect_explode), p.sync_every, p.stall_checks)
        if p.r1_per_solve is not None:
            q.r1_per_solve = self._chk(p.r1_per_solve, (self.nbatch,)).value
        return q

    def solve(self, psi, f, p: SolveParams):
        """psi [nbatch,ny,nx] CUDA tensor in/out; returns dict(iters, r1, r2, err) numpy arrays."""
        nb = self.nbatch
        iters = np.zeros(nb, np.int32); err = np.zeros(nb, np.int32); r1 = np.zeros(nb); r2 = np.zeros(nb)
        q = self._prm(p)
        _lib.check(_lib.lib().xee_plan_solve_dev(
            self._h, self._chk(psi, (nb, self.ny, self.nx)), self._chk(f, (nb, self.ny, self.nx)), C.byref(q),
            iters.ctypes.data_as(C.c_void_p), r1.ctypes.data_as(C.c_void_p), r2.ctypes.data_as(C.c_void_p),
            err.ctypes.data_as(C.c_void_p), self._stream()), "solve_dev")
        return dict(iters=iters, r1=r1, r2=r2, err=err)

    def solve_host(self, psi, f, p: SolveParams):
        """Same with HOST numpy arrays (H2D + D2H inside the call): the end-to-end entry."""
        nb = self.nbatch
        npdt = np.float64 if self.dtype == F64 else np.float32
        assert psi.dtype == npdt and psi.flags.c_contiguous and psi.shape == (nb, self.ny, self.nx)
        f = np.ascontiguousarray(f, npdt)
        iters = np.zeros(nb, np.int32); err = np.zeros(nb, np.int32); r1 = np.zeros(nb); r2 = np.zeros(nb)
        q = self._prm(p)
        _lib.check(_lib.lib().xee_plan_solve_host(
            self._h, psi.ctypes.data_as(C.c_void_p), f.ctypes.data_as(C.c_void_p), C.byref(q),
            iters.ctypes.data_as(C.c_void_p), r1.ctypes.data_as(C.c_void_p), r2.ctypes.data_as(C.c_void_p),
            err.ctypes.data_as(C.c_void_p)), "solve_host")
        return dict(iters=iters, r1=r1, r2=r2, err=err)

    def sweeps(self, psi, f, alpha, sweeps, want_rms=False, check_step=100):
        """Exactly `sweeps` sweeps, no stop rule.  Returns the RMS residual of the last sweep per solve (or None).
        The BiCGStab methods run `sweeps` iterations with the residual replacements of a solve with `check_step` (the
        returned field is then that of a solve stopping at iters = sweeps) and return the true residual after them.
        line2_mixed runs `sweeps` fp32 sweeps in refinement steps of `check_step` (a partial last step is applied), the
        field and the residual are those of a solve stopping at iters = sweeps."""
        nb = self.nbatch
        rms = np.zeros(nb) if want_rms else None
        _lib.check(_lib.lib().xee_plan_sweeps_checked_dev(
            self._h, self._chk(psi, (nb, self.ny, self.nx)), self._chk(f, (nb, self.ny, self.nx)), C.c_double(alpha),
            C.c_int(sweeps), C.c_int(check_step), rms.ctypes.data_as(C.c_void_p) if want_rms else None, self._stream()),
            "sweeps_dev")
        return rms

    def apply(self, psi):
        """out = L psi on the interior, 0 on the boundary (do_elliptic for the whole batch)."""
        torch = _torch()
        out = torch.empty_like(psi)
        _lib.check(_lib.lib().xee_plan_apply_dev(self._h, self._chk(psi, (self.nbatch, self.ny, self.nx)),
                                                 C.c_void_p(out.data_ptr()), self._stream()), "apply_dev")
        return out

    def sweep_kernel_stats(self, reset=False):
        ms = C.c_double(0); n = C.c_longlong(0)
        _lib.lib().xee_sweep_kernel_stats(self._h, C.byref(ms), C.byref(n), C.c_int(int(reset)))
        return ms.value, n.value

    def kernel_info(self):
        """(variant 1..5, sweeps per kernel launch, kernel launches since the last stats reset) of the sweep kernel."""
        v = C.c_int(0); d = C.c_int(0); n = C.c_longlong(0)
        _lib.lib().xee_plan_kernel_info(self._h, C.byref(v), C.byref(d), C.byref(n))
        return v.value, d.value, n.value


    def cheb_params(self):
        """(rho, gamma) of the last accelerated call: spectral radius of I - gamma M^-1 L and the step length gamma."""
        r = C.c_double(0); g = C.c_double(0)
        _lib.lib().xee_plan_cheb_params(self._h, C.byref(r), C.byref(g))
        return r.value, g.value


def launch_count(reset=False) -> int:
    return int(_lib.lib().xee_launch_count(C.c_int(int(reset))))


def pool_stats():
    """(live_bytes, cached_bytes) of the library's device-memory pool: blocks held by live plans, maps and series, and
    freed blocks kept for reuse."""
    live = C.c_longlong(0); cached = C.c_longlong(0)
    _lib.check(_lib.lib().xee_pool_stats(C.byref(live), C.byref(cached)), "pool_stats")
    return live.value, cached.value
