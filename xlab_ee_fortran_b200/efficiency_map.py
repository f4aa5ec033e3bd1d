"""Efficiency map (Part 3 of include/xee_b200.h): one elliptic solve per heating location, sharded
across GPUs as independent batches and gathered to rank 0 with one collective.

Mirrors the heating -> circulation -> kinetic-energy-generation -> efficiency chain of the reference's
legacy driver (src/old-diagnose/diagnose.f90:383-461, 915-941, 1029-1127, 780-839); the adjoint check
is the current driver's eta field (src/diagnose/diagnose.f90:31-48).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .plan import ARITH_FAST, ARITH_STRICT, CHEBYSHEV, F32, F64, JACOBI, METHODS, SolveParams, _SolveParams

COLS = ("iters", "r1", "err", "sum_Q", "ke_gen", "efficiency", "sum_Qeta", "efficiency_eta")
ADJ_COLS = ("sum_Q", "ke_gen", "efficiency")     # rows of adjoint_eval
FIELDS = {"psi": 0, "f": 1, "theta": 2, "eta": 3, "chi": 4, "eta_discrete": 5, "lambda": 6}


class _MapDesc(C.Structure):
    _fields_ = [("dtype", C.c_int), ("nr", C.c_int), ("nz", C.c_int), ("nheat", C.c_int), ("density_mode", C.c_int),
                ("arith", C.c_int), ("method", C.c_int), ("device", C.c_int), ("adjoint_check", C.c_int),
                ("Lr", C.c_double * 2), ("Lz", C.c_double * 2), ("r1_rel_rms_f", C.c_double)]


def _prm(p: SolveParams):
    return _SolveParams(p.max_iter, p.check_step, p.converge_time, p.lost_rate, p.r1, p.r2, p.alpha, None,
                        p.rho_jacobi, int(p.detect_explode), p.sync_every, p.stall_checks)


class EfficiencyMap:
    """Holds the vortex operator on one GPU and solves `nheat` heating locations per run()."""

    def __init__(self, A, B, Cf, Lr, Lz, nheat, dtype="f64", density_mode=0, arith="fast", method="line_chebyshev",
                 adjoint_check=False, r1_rel=1e-12, device=-1):
        _lib.require_gpu()
        A = np.ascontiguousarray(A, np.float32); B = np.ascontiguousarray(B, np.float32); Cf = np.ascontiguousarray(Cf, np.float32)
        nz, nr = A.shape
        assert B.shape == (nz, nr) and Cf.shape == (nz, nr)
        self.nr, self.nz, self.nheat = nr, nz, int(nheat)
        self.np_dtype = np.float64 if dtype == "f64" else np.float32
        d = _MapDesc(F64 if dtype == "f64" else F32, nr, nz, self.nheat, density_mode,
                     ARITH_STRICT if arith == "strict" else ARITH_FAST, METHODS[method],
                     device, int(adjoint_check), (C.c_double * 2)(*Lr), (C.c_double * 2)(*Lz), float(r1_rel))
        self._h = C.c_void_p()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(_lib.lib().xee_map_create(C.byref(d), p(A), p(B), p(Cf), C.byref(self._h)), "map_create")

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.lib().xee_map_destroy(self._h)
            self._h = None

    __del__ = close

    def run(self, heat, p: SolveParams):
        """heat [nheat,5] host doubles -> table [nheat, 8] host doubles (columns COLS)."""
        heat = np.ascontiguousarray(heat, np.float64)
        assert heat.shape == (self.nheat, 5)
        table = np.zeros((self.nheat, len(COLS)))
        q = _prm(p)
        _lib.check(_lib.lib().xee_map_run_host(self._h, heat.ctypes.data_as(C.c_void_p), C.byref(q),
                                               table.ctypes.data_as(C.c_void_p)), "map_run_host")
        return table

    def run_dev(self, heat_t, table_t, p: SolveParams):
        """Device-resident variant: heat_t [nheat,5] and table_t [nheat,8] are CUDA float64 tensors."""
        import torch
        assert heat_t.is_cuda and heat_t.dtype == torch.float64 and heat_t.is_contiguous() and tuple(heat_t.shape) == (self.nheat, 5)
        assert table_t.is_cuda and table_t.dtype == torch.float64 and table_t.is_contiguous() and tuple(table_t.shape) == (self.nheat, len(COLS))
        q = _prm(p)
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.lib().xee_map_run_dev(self._h, C.c_void_p(heat_t.data_ptr()), C.byref(q),
                                              C.c_void_p(table_t.data_ptr()), s), "map_run_dev")
        return table_t

    def adjoint_solve(self, p: SolveParams):
        """Solves L^T lambda = g once (g: the gradient of ke_gen in psi) and forms mu = H^T lambda on the B cells, after which
        adjoint_eval gives the exact discrete efficiency of any heating.  Returns (iters, r1, err) of the solve."""
        q = _prm(p)
        it = C.c_int(0); r1 = C.c_double(0); err = C.c_int(0)
        _lib.check(_lib.lib().xee_map_adjoint_solve(self._h, C.byref(q), C.byref(it), C.byref(r1), C.byref(err)),
                   "map_adjoint_solve")
        return it.value, r1.value, err.value

    def adjoint_eval(self, heat):
        """heat [n,5] host doubles, any n >= 1 -> [n, 3] host doubles (columns ADJ_COLS) from the last adjoint_solve."""
        heat = np.ascontiguousarray(heat, np.float64)
        assert heat.ndim == 2 and heat.shape[1] == 5
        table = np.zeros((heat.shape[0], len(ADJ_COLS)))
        _lib.check(_lib.lib().xee_map_adjoint_eval_host(self._h, heat.ctypes.data_as(C.c_void_p), C.c_int(heat.shape[0]),
                                                        table.ctypes.data_as(C.c_void_p)), "map_adjoint_eval_host")
        return table

    def adjoint_timings(self):
        """Host wall time (ms) of the adjoint plan: setup (first solve only), spectral probes and sweep kernels."""
        v = [C.c_double(0) for _ in range(3)]
        _lib.check(_lib.lib().xee_map_adjoint_timings(self._h, *(C.byref(x) for x in v)), "map_adjoint_timings")
        return dict(setup_ms=v[0].value, probe_ms=v[1].value, sweep_ms=v[2].value)

    def field(self, which):
        """psi, f, theta, eta, chi as computed by run(); eta_discrete (eta_d on the B cells) and lambda by adjoint_solve()."""
        idx = FIELDS[which]
        shape = {0: (self.nheat, self.nz, self.nr), 1: (self.nheat, self.nz, self.nr), 2: (self.nz - 1, self.nr - 1),
                 3: (self.nz, self.nr - 1), 4: (self.nz, self.nr), 5: (self.nz - 1, self.nr - 1), 6: (self.nz, self.nr)}[idx]
        out = np.zeros(shape, self.np_dtype)
        _lib.check(_lib.lib().xee_map_get_field(self._h, idx, out.ctypes.data_as(C.c_void_p)), "map_get_field")
        return out

    def sweep_kernel_stats(self, reset=False):
        ms = C.c_double(0); n = C.c_longlong(0)
        _lib.lib().xee_map_sweep_kernel_stats(self._h, C.byref(ms), C.byref(n), C.c_int(int(reset)))
        return ms.value, n.value

    def kernel_info(self):
        """(variant 1..5, sweeps per kernel launch, kernel launches since the last stats reset) of the sweep kernel."""
        v = C.c_int(0); d = C.c_int(0); n = C.c_longlong(0)
        _lib.lib().xee_map_kernel_info(self._h, C.byref(v), C.byref(d), C.byref(n))
        return v.value, d.value, n.value


# ---------------------------------------------------------------------------------- sharding (SURVEY 8e)
def partition(n_items: int, world: int, rank: int):
    """Static contiguous chunks: item n goes to rank floor(n*world/n_items).  Returns (start, stop)."""
    start = (rank * n_items + world - 1) // world
    stop = ((rank + 1) * n_items + world - 1) // world
    return start, stop


def gather_rows(local_rows, n_items: int, group=None):
    """One collective: every rank contributes its [n_local, cols] rows; rank 0 gets [n_items, cols] (others None).

    Implemented as an all_gather of equal-size padded chunks (NCCL 2.27 has no gather primitive;
    the payload is KB-scale so there is nothing to overlap - SURVEY section 8e).
    """
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group); rank = dist.get_rank(group)
    cols = local_rows.shape[1]
    chunk = max(partition(n_items, world, r)[1] - partition(n_items, world, r)[0] for r in range(world))
    pad = torch.zeros((chunk, cols), dtype=local_rows.dtype, device=local_rows.device)
    pad[: local_rows.shape[0]] = local_rows
    out = torch.empty((world * chunk, cols), dtype=local_rows.dtype, device=local_rows.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    if rank != 0:
        return None
    parts = []
    for r in range(world):
        a, b = partition(n_items, world, r)
        parts.append(out[r * chunk: r * chunk + (b - a)])
    return torch.cat(parts, 0)
