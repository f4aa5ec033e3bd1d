"""Time-series diagnosis (Part 4 of include/xee_b200.h, BASELINE config 5): one operator per snapshot."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .efficiency_map import _prm
from .plan import ARITH_FAST, ARITH_STRICT, CHEBYSHEV, F32, F64, JACOBI, METHODS, SolveParams

COLS = ("iters", "r1", "err", "sum_Q", "ke_gen", "efficiency", "w_absmax", "u_absmax")
# TimeSeries.decompose: table columns (raw sums; an efficiency.txt line is "value , value / sum_Q"), the solves of the
# iters / err arrays, the fields of decomp_field and the baro modes
_TERMS = ("eta_bc", "eta_dB", "eta_B0", "bndconv", "bndconv2", "etaQ", "wtheta")
DECOMP_COLS = ("sum_Q", "sum_dtheta_dt", "local_heat_response") + tuple(f"{t}_0" for t in _TERMS) + tuple(f"{t}_B0dB" for t in _TERMS)
DECOMP_SOLVES = ("psi_before", "chi_0_0", "chi_B0dB_0", "chi_0_dB", "chi_B0dB_dB", "chi_0_B0", "chi_B0dB_B0", "psi_after_0",
                 "psi_after_B0dB")
DECOMP_FIELDS = ("dtheta_dt", "theta_after") + DECOMP_SOLVES
BARO = {"barotropic": 0, "baroclinic": 1, "all": 2}


class _SeriesDesc(C.Structure):
    _fields_ = [("dtype", C.c_int), ("nr", C.c_int), ("nz", C.c_int), ("nsnap", C.c_int), ("density_mode", C.c_int),
                ("arith", C.c_int), ("method", C.c_int), ("device", C.c_int), ("Lr", C.c_double * 2), ("Lz", C.c_double * 2),
                ("r1_rel_rms_f", C.c_double)]


class _DecompDesc(C.Structure):
    _fields_ = [("tendency", C.c_int), ("testing_dt", C.c_double), ("baro", C.c_int)]


class TimeSeries:
    def __init__(self, nr, nz, Lr, Lz, nsnap, dtype="f64", density_mode=0, arith="fast", method="line_chebyshev", r1_rel=1e-12,
                 device=-1):
        _lib.require_gpu()
        self.nr, self.nz, self.nsnap = int(nr), int(nz), int(nsnap)
        self.np_dtype = np.float64 if dtype == "f64" else np.float32
        d = _SeriesDesc(F64 if dtype == "f64" else F32, nr, nz, nsnap, density_mode,
                        ARITH_STRICT if arith == "strict" else ARITH_FAST, METHODS[method],
                        device, (C.c_double * 2)(*Lr), (C.c_double * 2)(*Lz), float(r1_rel))
        self._h = C.c_void_p()
        _lib.check(_lib.lib().xee_series_create(C.byref(d), C.byref(self._h)), "series_create")

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.lib().xee_series_destroy(self._h)
            self._h = None

    __del__ = close

    def run(self, params, p: SolveParams):
        params = np.ascontiguousarray(params, np.float64)
        assert params.shape == (self.nsnap, 21)
        table = np.zeros((self.nsnap, len(COLS)))
        q = _prm(p)
        _lib.check(_lib.lib().xee_series_run_host(self._h, params.ctypes.data_as(C.c_void_p), C.byref(q),
                                                  table.ctypes.data_as(C.c_void_p)), "series_run_host")
        return table

    def run_fields(self, A, B, Cf, Q, p: SolveParams, F=None, psi_bc=None):
        """The series on caller-supplied snapshots: A, B, C and psi_bc [nsnap, nz, nr] on the O grid, the heating Q and the
        momentum forcing F [nsnap, nz-1, nr-1] on the B cells, i (r) fastest.  F=None: no momentum term; psi_bc=None: a zero
        rim, else only its rim is read (Dirichlet values of r*psi).  Host arrays (numpy, CPU tensors) are converted to the
        plan dtype and go through the host entry.  CUDA tensors must all be of the plan dtype and on the series' device,
        and are read on the current stream; a mix of host and CUDA inputs is refused.  Returns the table
        [nsnap, 8] (columns COLS); a heating whose integral is 0 gives a non-finite efficiency."""
        arrs, ptrs, extra, dev = self._inputs("run_fields", dict(A=A, B=B, C=Cf, Q=Q, F=F, psi_bc=psi_bc))
        fn, what = (_lib.lib().xee_series_run_fields_dev, "series_run_fields_dev") if dev else \
            (_lib.lib().xee_series_run_fields_host, "series_run_fields_host")
        table = np.zeros((self.nsnap, len(COLS)))
        q = _prm(p)
        _lib.check(fn(self._h, *ptrs, C.byref(q), table.ctypes.data_as(C.c_void_p), *extra), what)
        return table

    def _inputs(self, what, given):
        """The caller's snapshot arrays checked and converted (host arrays to the plan dtype; CUDA tensors must all be of the
        plan dtype), which the caller keeps alive over the call, their pointers in the order of `given`, the trailing stream
        argument of the device entry and whether it is the device entry."""
        n, nz, nr = self.nsnap, self.nz, self.nr
        shapes = dict(A=(n, nz, nr), B=(n, nz, nr), C=(n, nz, nr), Q=(n, nz - 1, nr - 1), F=(n, nz - 1, nr - 1), psi_bc=(n, nz, nr),
                      chi_bc=(n, nz, nr))
        on_dev = any(getattr(v, "is_cuda", False) for v in given.values())
        if not on_dev:
            given = {k: None if v is None else np.asarray(v) for k, v in given.items()}
        for k, v in given.items():
            if v is not None and tuple(v.shape) != shapes[k]:
                raise ValueError(f"{what}: {k} has shape {tuple(v.shape)}, expected {shapes[k]}")
        if on_dev:
            import torch
            tdt = torch.float64 if self.np_dtype == np.float64 else torch.float32
            for k, v in given.items():
                if v is not None and not (isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == tdt):
                    raise TypeError(f"{what}: {k} must be a CUDA tensor of {tdt} like the other device inputs")
            arrs = {k: None if v is None else v.contiguous() for k, v in given.items()}
            ptr = lambda v: None if v is None else C.c_void_p(v.data_ptr())
            extra = (C.c_void_p(torch.cuda.current_stream(arrs["A"].device).cuda_stream),)
        else:
            arrs = {k: None if v is None else np.ascontiguousarray(v, self.np_dtype) for k, v in given.items()}
            ptr = lambda v: None if v is None else v.ctypes.data_as(C.c_void_p)
            extra = ()
        return arrs, [ptr(v) for v in arrs.values()], extra, on_dev

    def decompose(self, A, B, Cf, Q, p_psi: SolveParams, p_chi: SolveParams, F=None, psi_bc=None, chi_bc=None, testing_dt=None,
                  baro="all"):
        """The legacy efficiency decomposition (the terms of efficiency.txt) of every snapshot, on the inputs of run_fields plus
        chi_bc [nsnap, nz, nr] (only its rim is read; None: no boundary chi solves, no exchange conversion).  testing_dt=None
        is INSTANT mode, a number TENDENCY mode over that time step; baro "barotropic" (operator B = 0), "baroclinic"
        (B = B0 + dB) or "all" (also 0, 1, 2).  p_psi governs the psi solves, p_chi the chi solves.  Returns (table
        [nsnap, 17] with columns DECOMP_COLS, NaN where not computed; iters and err [nsnap, 9] in the order DECOMP_SOLVES,
        iters -1 for a solve not run)."""
        arrs, ptrs, extra, dev = self._inputs("decompose", dict(A=A, B=B, C=Cf, Q=Q, F=F, psi_bc=psi_bc, chi_bc=chi_bc))
        fn, what = (_lib.lib().xee_series_decompose_dev, "series_decompose_dev") if dev else \
            (_lib.lib().xee_series_decompose_host, "series_decompose_host")
        if isinstance(baro, str):
            if baro not in BARO:
                raise ValueError(f"decompose: baro must be one of {tuple(BARO)} or 0, 1, 2, not {baro!r}")
            baro = BARO[baro]
        desc = _DecompDesc(0 if testing_dt is None else 1, 0.0 if testing_dt is None else float(testing_dt), int(baro))
        table = np.zeros((self.nsnap, len(DECOMP_COLS)))
        iters = np.zeros((self.nsnap, len(DECOMP_SOLVES)), np.int32)
        err = np.zeros_like(iters)
        qp, qc = _prm(p_psi), _prm(p_chi)
        _lib.check(fn(self._h, C.byref(desc), *ptrs, C.byref(qp), C.byref(qc), table.ctypes.data_as(C.c_void_p),
                      iters.ctypes.data_as(C.c_void_p), err.ctypes.data_as(C.c_void_p), *extra), what)
        return table, iters, err

    def decomp_field(self, which):
        """A field of the last decompose: dtheta_dt, theta_after [nsnap, nz-1, nr-1] or the field of a solve of DECOMP_SOLVES
        [nsnap, nz, nr]; fails for a field it did not make."""
        idx = DECOMP_FIELDS.index(which)
        n, nz, nr = self.nsnap, self.nz, self.nr
        out = np.zeros((n, nz - 1, nr - 1) if idx < 2 else (n, nz, nr), self.np_dtype)
        _lib.check(_lib.lib().xee_series_get_decomp_field(self._h, idx, out.ctypes.data_as(C.c_void_p)), "series_get_decomp_field")
        return out

    def field(self, which):
        """psi, f, theta, u, w, A, B, C, m2, Q and F of the last run (F fails after a run_fields without F)."""
        nr, nz, n = self.nr, self.nz, self.nsnap
        idx, shape = {"psi": (0, (n, nz, nr)), "f": (1, (n, nz, nr)), "theta": (2, (n, nz - 1, nr - 1)), "u": (3, (n, nz - 1, nr)),
                      "w": (4, (n, nz, nr - 1)), "A": (5, (n, nz, nr)), "B": (6, (n, nz, nr)), "C": (7, (n, nz, nr)),
                      "m2": (8, (n, nz - 1, nr - 1)), "Q": (9, (n, nz - 1, nr - 1)), "F": (10, (n, nz - 1, nr - 1))}[which]
        out = np.zeros(shape, self.np_dtype)
        _lib.check(_lib.lib().xee_series_get_field(self._h, idx, out.ctypes.data_as(C.c_void_p)), "series_get_field")
        return out

    def sweep_kernel_stats(self, reset=False):
        ms = C.c_double(0); n = C.c_longlong(0)
        _lib.lib().xee_series_sweep_kernel_stats(self._h, C.byref(ms), C.byref(n), C.c_int(int(reset)))
        if reset:
            _lib.lib().xee_series_probe_stats(self._h, None, C.c_int(1))
        return ms.value, n.value

    def probe_ms(self):
        """Host wall time (ms) of the spectral-radius probes since the last stats reset."""
        ms = C.c_double(0)
        _lib.lib().xee_series_probe_stats(self._h, C.byref(ms), C.c_int(0))
        return ms.value

    def kernel_info(self):
        """(variant 1..5, sweeps per kernel launch, kernel launches since the last stats reset) of the sweep kernel."""
        v = C.c_int(0); d = C.c_int(0); n = C.c_longlong(0)
        _lib.lib().xee_series_kernel_info(self._h, C.byref(v), C.byref(d), C.byref(n))
        return v.value, d.value, n.value


def run_sharded(nr, nz, Lr, Lz, total, p: SolveParams, world=1, rank=0, device=-1, **kw):
    """BASELINE config 5 on `world` GPUs: snapshots [a, b) of a `total`-long series on this rank (static contiguous chunks,
    SURVEY section 8e: independent solves, nothing exchanged), parameters generated per rank from the snapshot index.
    Returns (a, b, table [b-a, 8]); gather the rows with efficiency_map.gather_rows (one collective)."""
    from . import workloads as W
    from .efficiency_map import partition
    a, b = partition(total, world, rank)
    ts = TimeSeries(nr, nz, Lr, Lz, b - a, device=device, **kw)
    try:
        return a, b, ts.run(W.series_params(b - a, total=total, first=a), p)
    finally:
        ts.close()


def run_fields_sharded(nr, nz, Lr, Lz, A, B, Cf, Q, p: SolveParams, F=None, psi_bc=None, world=1, rank=0, device=-1, **kw):
    """The field counterpart of run_sharded: snapshots [a, b) of the caller's whole series (static contiguous chunks of
    efficiency_map.partition) on this rank.  A, B, C, Q, F, psi_bc are the whole series' arrays as for TimeSeries.run_fields;
    only rows [a, b) are read.  Returns (a, b, table [b-a, 8])."""
    from .efficiency_map import partition
    a, b = partition(int(A.shape[0]), world, rank)
    ts = TimeSeries(nr, nz, Lr, Lz, b - a, device=device, **kw)
    try:
        rows = lambda x: None if x is None else x[a:b]
        return a, b, ts.run_fields(A[a:b], B[a:b], Cf[a:b], Q[a:b], p, F=rows(F), psi_bc=rows(psi_bc))
    finally:
        ts.close()


def decompose_sharded(nr, nz, Lr, Lz, A, B, Cf, Q, p_psi: SolveParams, p_chi: SolveParams, F=None, psi_bc=None, chi_bc=None,
                      testing_dt=None, baro="all", world=1, rank=0, device=-1, **kw):
    """TimeSeries.decompose of snapshots [a, b) of the caller's whole series on this rank (static contiguous chunks of
    efficiency_map.partition, as run_fields_sharded).  Returns (a, b, table, iters, err) of those rows."""
    from .efficiency_map import partition
    a, b = partition(int(A.shape[0]), world, rank)
    ts = TimeSeries(nr, nz, Lr, Lz, b - a, device=device, **kw)
    try:
        rows = lambda x: None if x is None else x[a:b]
        return (a, b, *ts.decompose(A[a:b], B[a:b], Cf[a:b], Q[a:b], p_psi, p_chi, F=rows(F), psi_bc=rows(psi_bc),
                                    chi_bc=rows(chi_bc), testing_dt=testing_dt, baro=baro))
    finally:
        ts.close()
