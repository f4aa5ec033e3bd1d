"""Discrete-adjoint efficiency maps (EfficiencyMap.adjoint_solve / adjoint_eval) against the exact discrete adjoint
(tests/adjoint_oracle.py: sparse LU of L^T) and against the map's own direct solves.

North-star tolerances as in test_gpu_bench_exact.py: fields within 1e-8 relative L2, efficiencies within 1e-6 relative.
An adjoint solved with L in place of L^T misses every operator used here by over 3e3 x that (test_adjoint_oracle.py).
"""
import gc
import os

import numpy as np
import pytest

from tests.adjoint_oracle import ExactAdjoint
from tests.exact_oracle import MapCase
from tests.util import rel_l2

pytestmark = pytest.mark.gpu
LR, LZ = (0.0, 1.0e6), (0.0, 1.5e4)


def _params(stall_checks=10, max_iter=2000000, check_step=5):
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=max_iter, check_step=check_step, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=stall_checks)


def _lattice(nr, nz, n_side=8, width=2.0):
    from xlab_ee_fortran_b200 import workloads as W
    return W.heating_lattice(n_side, n_side, LR, LZ, width * LR[1] / (nr - 1), width * LZ[1] / (nz - 1))


def _series_fields(nr, nz, first=900):
    from xlab_ee_fortran_b200 import workloads as W
    return W.series_fields_host(W.series_params(1, total=1024, first=first)[0], nr, nz, LR, LZ)[:3]


def _run_case(A, B, C, heat, dtype, method, arith, r1_rel, prm):
    """One map: run() on every heating row, then adjoint_solve and adjoint_eval of the same rows."""
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    m = EfficiencyMap(A, B, C, LR, LZ, len(heat), dtype, arith=arith, method=method, r1_rel=r1_rel)
    table = m.run(heat, prm)
    it, r1, err = m.adjoint_solve(prm)
    out = dict(table=table, iters=it, r1=r1, err=err, adj=m.adjoint_eval(heat), lam=m.field("lambda"),
               eta_d=m.field("eta_discrete"))
    return m, out


def _check_against_exact(name, A, B, C, heat, got, field_tol=1e-8, eff_tol=1e-6):
    ex = ExactAdjoint(MapCase(A, B, C, LR, LZ))
    ref = ex.rows(heat)
    e_lam, e_eta = rel_l2(got["lam"], ex.lam), rel_l2(got["eta_d"], ex.eta_d)
    e_exact = np.abs(got["adj"][:, 2] - ref[:, 2]) / np.abs(ref[:, 2])
    e_run = np.abs(got["adj"][:, 2] - got["table"][:, 5]) / np.abs(got["table"][:, 5])
    direct = got["table"][:, 0]
    print(f"{name}: adjoint {got['iters']} sweeps (err {got['err']}) against direct {int(direct.min())}-{int(direct.max())} "
          f"(median {int(np.median(direct))}); lambda {e_lam:.2e}, eta_d {e_eta:.2e} relative L2; efficiencies "
          f"{e_exact.max():.2e} from exact, {e_run.max():.2e} from run()")
    assert got["err"] in (0, 4), got["err"]
    assert np.all((got["table"][:, 2] == 0) | (got["table"][:, 2] == 4))
    assert e_lam < field_tol and e_eta < field_tol, (e_lam, e_eta)
    assert np.all(e_exact < eff_tol), [(int(n), e_exact[n]) for n in np.argsort(e_exact)[::-1][:8]]
    assert np.all(e_run < eff_tol), [(int(n), e_run[n]) for n in np.argsort(e_run)[::-1][:8]]
    # the preconditioned L^T has the spectrum of the preconditioned L: the adjoint takes as many sweeps as a direct solve
    assert 0.5 * np.median(direct) <= got["iters"] <= 2.0 * np.median(direct), (got["iters"], np.median(direct))
    return ex


# ------------------------------------------------------------------ 1. the bench shape
@pytest.fixture(scope="module")
def bench_case():
    import bench
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = bench.heat_rows(512)
    m, got = _run_case(A, B, C, heat, "f64", "line2_chebyshev", "fast", bench.R1_REL, _params())
    yield dict(A=A, B=B, C=C, heat=heat, m=m, got=got)
    m.close()


def test_bench_shape_against_exact_adjoint_and_direct_solves(bench_case):
    c = bench_case
    _check_against_exact("bench 512x256 line2_chebyshev", c["A"], c["B"], c["C"], c["heat"], c["got"])
    # sum_Q is computed cell for cell and summed in the order of the map's integrals kernel: the same bits
    assert np.array_equal(c["got"]["adj"][:, 0], c["got"]["table"][:, 3])
    assert np.all(c["got"]["lam"][0] == 0) and np.all(c["got"]["lam"][-1] == 0)
    assert np.all(c["got"]["lam"][:, 0] == 0) and np.all(c["got"]["lam"][:, -1] == 0)


# ------------------------------------------------------------------ 2. a strongly non-symmetric vortex
def test_late_series_snapshot_vortex():
    nr, nz = 128, 64
    A, B, C = _series_fields(nr, nz)
    heat = _lattice(nr, nz)
    m, got = _run_case(A, B, C, heat, "f64", "line2_chebyshev", "fast", 1e-12, _params(stall_checks=20))
    m.close()
    _check_against_exact("series snapshot 900, 128x64 line2_chebyshev", A, B, C, heat, got)


# ------------------------------------------------------------------ 3. the map's method and arithmetic: STRICT Jacobi
def test_strict_jacobi_small_grid():
    from xlab_ee_fortran_b200 import workloads as W
    nr, nz = 48, 40
    A, B, C = W.vortex_fields(nr, nz, LR, LZ)
    heat = _lattice(nr, nz, n_side=3, width=3.0)
    m, got = _run_case(A, B, C, heat, "f64", "jacobi", "strict", 1e-13, _params(stall_checks=40, check_step=100))
    m.close()
    _check_against_exact("48x40 STRICT jacobi", A, B, C, heat, got)


# ------------------------------------------------------------------ 4. an fp32 map
def test_fp32_map_is_as_close_to_exact_as_its_direct_solves():
    """No fp32 figure is known in advance: the adjoint's efficiencies may be at most 10 x as far from the exact (fp64)
    ones as the same map's direct solves are, on the same rows."""
    from xlab_ee_fortran_b200 import workloads as W
    nr, nz = 256, 128
    A, B, C = W.vortex_fields(nr, nz, LR, LZ)
    heat = _lattice(nr, nz)
    m, got = _run_case(A, B, C, heat, "f32", "line_chebyshev", "fast", 1e-6, _params(stall_checks=10, max_iter=200000))
    m.close()
    ref = ExactAdjoint(MapCase(A, B, C, LR, LZ)).rows(heat)[:, 2]
    e_dir = np.abs(got["table"][:, 5] - ref) / np.abs(ref)
    e_adj = np.abs(got["adj"][:, 2] - ref) / np.abs(ref)
    print(f"fp32 256x128 line_chebyshev: adjoint {got['iters']} sweeps (err {got['err']}), direct median "
          f"{int(np.median(got['table'][:, 0]))}; largest efficiency error from exact: adjoint {e_adj.max():.2e}, "
          f"direct {e_dir.max():.2e}")
    assert got["lam"].dtype == np.float32 and got["eta_d"].dtype == np.float32
    assert e_adj.max() <= 10 * e_dir.max(), (e_adj.max(), e_dir.max())


# ------------------------------------------------------------------ 5. rows do not depend on the call they share
def _cell_blobs(nr, nz, q0):
    """One narrow blob per B cell, centred on it: sigma = half a cell."""
    ra = np.linspace(LR[0], LR[1], nr); za = np.linspace(LZ[0], LZ[1], nz)
    rm, zm = (ra[:-1] + ra[1:]) / 2, (za[:-1] + za[1:]) / 2
    R, Z = np.meshgrid(rm, zm)
    n = R.size
    return np.stack([R.ravel(), Z.ravel(), np.full(n, 0.5 * (ra[1] - ra[0])), np.full(n, 0.5 * (za[1] - za[0])),
                     np.full(n, q0)], axis=1)


def test_rows_are_independent_of_the_row_count(bench_case):
    import bench
    m, heat = bench_case["m"], bench_case["heat"]
    many = m.adjoint_eval(heat)
    one = m.adjoint_eval(heat[7:8])
    assert np.array_equal(one[0], many[7])
    blobs = _cell_blobs(bench.NR, bench.NZ, heat[0, 4])
    assert len(blobs) == (bench.NR - 1) * (bench.NZ - 1) == 130305
    big = m.adjoint_eval(blobs)
    rng = np.random.default_rng(3)
    sample = np.sort(rng.choice(len(blobs), 256, replace=False))
    for q in sample:
        alone = m.adjoint_eval(blobs[q:q + 1])
        assert np.array_equal(alone[0], big[q]), (int(q), alone[0], big[q])
    # a blob half a cell wide is nearly all in its own cell: its efficiency is close to that cell's eta_d
    eta_d = bench_case["got"]["eta_d"].ravel()
    near = np.abs(big[:, 2] - eta_d) / np.abs(eta_d).max()
    print(f"130305 cell blobs: efficiency within {near.max():.2e} of max|eta_d| of the cell's eta_d")
    assert near.max() < 0.05


def test_skipping_cells_out_of_reach_gives_the_full_sums_bits(bench_case):
    """adjoint_eval visits only the cells where a blob's exponent can be above -800; XEE_ADJ_FULL_SUM=1 visits them all."""
    import bench
    m, heat = bench_case["m"], bench_case["heat"]
    blobs = _cell_blobs(bench.NR, bench.NZ, heat[0, 4])[::97]
    rows = np.concatenate([heat, blobs])
    windowed = m.adjoint_eval(rows)
    os.environ["XEE_ADJ_FULL_SUM"] = "1"
    try:
        full = m.adjoint_eval(rows)
    finally:
        del os.environ["XEE_ADJ_FULL_SUM"]
    assert np.array_equal(windowed, full)


# ------------------------------------------------------------------ 6. isolation and failures
def _live():
    from xlab_ee_fortran_b200.plan import pool_stats
    gc.collect()
    return pool_stats()[0]


def test_adjoint_leaves_run_and_memory_untouched():
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    nr, nz = 64, 48
    A, B, C = W.vortex_fields(nr, nz, LR, LZ)
    heat = _lattice(nr, nz, n_side=4)
    prm = _params()
    base = _live()
    plain = EfficiencyMap(A, B, C, LR, LZ, len(heat), "f64", method="line2_chebyshev", r1_rel=1e-12)
    t_plain = plain.run(heat, prm)
    with pytest.raises(RuntimeError, match="adjoint_solve"):
        plain.adjoint_eval(heat)
    with pytest.raises(RuntimeError, match="adjoint_solve"):
        plain.field("lambda")
    plain.close()
    m = EfficiencyMap(A, B, C, LR, LZ, len(heat), "f64", method="line2_chebyshev", r1_rel=1e-12)
    m.adjoint_solve(prm)
    m.adjoint_eval(heat)
    with pytest.raises(RuntimeError, match="n >= 1"):
        m.adjoint_eval(np.zeros((0, 5)))
    t1 = m.run(heat, prm)
    m.adjoint_solve(prm)
    t2 = m.run(heat, prm)
    m.close()
    assert np.array_equal(t_plain, t1) and np.array_equal(t_plain, t2)
    assert _live() == base
