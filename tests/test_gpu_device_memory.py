"""Device-memory ownership: every pool block a plan, map or series allocates goes back to the pool when the object is
destroyed, also when its setup or a solve fails.  Each test compares the pool's live bytes (plan.pool_stats) after the
objects are gone with those before they were made."""
import ctypes as C
import gc

import numpy as np
import pytest

from oracle import oracle as O
from tests.test_gpu_parity import _rand_case
from tests.test_gpu_stop_rule import DNX, DNY, _divergent
from tests.test_gpu_twolevel import _aniso

pytestmark = pytest.mark.gpu
NX, NY = 64, 34


def _mods():
    import torch
    import xlab_ee_fortran_b200 as X
    return torch, X


def _live():
    from xlab_ee_fortran_b200.plan import pool_stats
    gc.collect()
    return pool_stats()[0]


def _coe(method, dt, nsets, nx=NX, ny=NY):
    """[nsets, ny, nx, 9] operators of the method's family."""
    coes = []
    for q in range(nsets):
        if method.startswith("line"):
            a, b, c = _aniso(nx, ny, seed=5 + q)
        else:
            a, b, c, _, _ = _rand_case(nx, ny, np.float64, seed=7 + q, bscale=0.02)
        coes.append(O.cal_coe(a.astype(dt), b.astype(dt), c.astype(dt), 1.0, 0.5, nx, ny)[0])
    return np.stack(coes)


def _layouts():
    """(method, dtype, shared operator) of every configuration plan.METHODS accepts."""
    from xlab_ee_fortran_b200.plan import METHODS
    for method in METHODS:
        for dt in ("f64",) if method.startswith("line2") else ("f32", "f64"):
            for shared in (True, False):
                yield method, dt, shared


def _plan_cycle(torch, X, method, dt, shared, arith, nb, kernel):
    """Create, set the operator from the host, solve on device and host buffers, sweep, apply, destroy."""
    npdt = np.float64 if dt == "f64" else np.float32
    coe = _coe(method, npdt, 1)[0] if shared else _coe(method, npdt, nb)
    rng = np.random.default_rng(nb)
    P = rng.standard_normal((nb, NY, NX)).astype(npdt); F = rng.standard_normal((nb, NY, NX)).astype(npdt)
    alpha = 0.45 if method == "line2_jacobi" else 1.0
    plan = X.Plan(NX, NY, nbatch=nb, dtype=dt, shared_coe=shared, arith=arith, method=method, kernel=kernel)
    plan.set_coe_aos(coe)
    prm = X.SolveParams(max_iter=60, check_step=10, r1=1e-30, r2=0.0, alpha=alpha, sync_every=2)
    psi = torch.from_numpy(P).cuda(); ft = torch.from_numpy(F).cuda()
    plan.solve(psi, ft, prm)
    plan.solve_host(P.copy(), F, prm)
    plan.sweeps(psi, ft, alpha, 15, want_rms=True)
    plan.apply(psi)
    torch.cuda.synchronize()
    plan.close()


@pytest.mark.parametrize("method,dt,shared", list(_layouts()))
def test_plan_returns_every_block(method, dt, shared):
    """nbatch 1 takes the resident solver (v3) where it applies; the point methods also run on the TMA (v2) and the
    temporal-blocking (v4) kernels, so that every resident and every lazily allocated buffer is reached."""
    torch, X = _mods()
    point = not method.startswith("line")
    for arith in ("strict", "fast") if point else ("fast",):
        for nb in (1, 5):
            kernels = [0, 2] + ([4] if shared else []) if point else [0]
            for kernel in kernels:
                base = _live()
                _plan_cycle(torch, X, method, dt, shared, arith, nb, kernel)
                assert _live() == base, (method, dt, shared, arith, nb, kernel, _live() - base)


def test_drop_ins_return_every_block():
    """The Fortran-facing entry points make and destroy a plan per call; legacy strategy 3 allocates the max-norm partials."""
    _, X = _mods()
    a, b, c, f, x0 = _rand_case(NX, NY, np.float64, seed=3, bscale=0.02)
    base = _live()
    coe = np.zeros((NY, NX, 9))
    assert X.cal_coe(a, b, c, coe, 1.0, 0.5, NX, NY) == 0
    X.do_elliptic(x0, coe, np.zeros_like(x0), NX, NY)
    dat = x0.copy(); wk = np.zeros_like(dat)
    X.solve_elliptic(300, 100, 10, 5, 1e-30, 0.0, 1.0, dat, coe, f, wk, NX, NY)
    dat = x0.copy(); st = C.c_int(3); sr = C.c_double(1e-30); err = C.c_int(0)
    p = lambda arr: arr.ctypes.data_as(C.c_void_p)
    X._lib.lib().xee_solve_elliptic_old_f64(C.byref(C.c_int(300)), C.byref(st), C.byref(sr), C.byref(C.c_double(1.0)), p(dat),
                                            p(coe), p(f), p(wk), C.byref(C.c_int(NX)), C.byref(C.c_int(NY)), C.byref(err),
                                            C.byref(C.c_int(0)))
    assert err.value & 1, err.value
    assert _live() == base, _live() - base


def _map_fields(nr, nz):
    from xlab_ee_fortran_b200 import workloads as W
    Lr, Lz = (0.0, 6.0e5), (0.0, 1.5e4)
    A, B, Cf = W.vortex_fields(nr, nz, Lr, Lz)
    heat = W.heating_lattice(2, 2, Lr, Lz, 3 * Lr[1] / (nr - 1), 3 * Lz[1] / (nz - 1), r_frac=(0.02, 0.5), z_frac=(0.15, 0.75))
    return A, B, Cf, Lr, Lz, heat


def test_map_and_series_return_every_block():
    """An efficiency map with the adjoint solve (its own plan and the r1 temporary of that solve), and a smooth time series
    (the subsampled spectral estimate runs on a plan of its own)."""
    _, X = _mods()
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    from xlab_ee_fortran_b200.time_series import TimeSeries
    A, B, Cf, Lr, Lz, heat = _map_fields(64, 48)
    prm = X.SolveParams(max_iter=400, check_step=5, converge_time=2, r1=1.0, r2=0.0)
    base = _live()
    m = EfficiencyMap(A, B, Cf, Lr, Lz, len(heat), "f64", method="line2_chebyshev", adjoint_check=True, r1_rel=1e-10)
    m.run(heat, prm)
    m.field("eta")
    m.close(); del m
    assert _live() == base, _live() - base
    ts = TimeSeries(64, 40, Lr, Lz, 32, "f64", method="line2_chebyshev", r1_rel=1e-10)
    ts.run(W.series_params(32, total=1024), prm)
    ts.close(); del ts
    assert _live() == base, _live() - base


def test_map_whose_coarse_grid_is_refused_returns_every_block():
    """1800 radial points give 112 coarse columns, whose band factorisation needs more shared memory than the kernel may
    take: the map's setup fails after it has allocated its own buffers and the staging temporaries."""
    _, X = _mods()
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    A, B, Cf, Lr, Lz, heat = _map_fields(1800, 20)
    base = _live()
    with pytest.raises(RuntimeError, match="coarse grid too wide"):
        EfficiencyMap(A, B, Cf, Lr, Lz, len(heat), "f64", method="line2_chebyshev")
    assert _live() == base, _live() - base


def test_plan_whose_setup_fails_returns_every_block():
    """line2_mixed refuses nx = 2 (mod 4) after the block-line and two-level buffers are allocated."""
    _, X = _mods()
    base = _live()
    with pytest.raises(RuntimeError, match="nx % 4 == 0"):
        X.Plan(66, NY, nbatch=3, dtype="f64", arith="fast", method="line2_mixed")
    assert _live() == base, _live() - base


def test_rejected_spectral_estimate_keeps_the_plan_memory():
    """The operator of the divergence tests has a stage-A ratio outside (0, 1): the estimate fails and its probe buffers go
    back; the plan then solves a valid operator."""
    torch, X = _mods()
    coe, f, x0 = _divergent(np.float64)
    P = np.stack([x0, 0.5 * x0]); F = np.stack([f, -f])
    plan = X.Plan(DNX, DNY, nbatch=2, dtype="f64", arith="fast", method="chebyshev")
    plan.set_coe_aos(coe)
    prm = lambda rho: X.SolveParams(max_iter=2000, check_step=20, converge_time=2, r1=1e-8, r2=0.0, rho_jacobi=rho)
    plan.solve(torch.from_numpy(P).cuda(), torch.from_numpy(F).cuda(), prm(0.99))   # an explicit radius: no estimate
    base = _live()
    with pytest.raises(RuntimeError, match="spectral-radius estimate outside"):
        plan.solve(torch.from_numpy(P).cuda(), torch.from_numpy(F).cuda(), prm(0.0))
    assert _live() == base, _live() - base
    plan.set_coe_aos(_coe("chebyshev", np.float64, 1, DNX, DNY)[0])
    out = plan.solve(torch.from_numpy(P).cuda(), torch.from_numpy(F).cuda(), prm(0.0))
    assert list(out["err"]) == [0, 0], out
    assert _live() == base, _live() - base
    plan.close()
