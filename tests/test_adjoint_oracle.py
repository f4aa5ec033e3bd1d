"""CPU checks of the exact discrete adjoint (tests/adjoint_oracle.py) against the oracle's own routines: the functional g
against ke_gen, H^T against rhs_thermal, and the adjoint efficiencies against the direct ones of exact sparse-LU fields.
The last test is the guard of the GPU tests: an adjoint solved with L in place of L^T must miss by far more than they allow.
"""
import numpy as np
import pytest

from tests.adjoint_oracle import ExactAdjoint, asymmetry, heating_adjoint, ke_functional, rhs_thermal
from tests.exact_oracle import ExactSolver, MapCase, efficiency_row, ke_gen

LR, LZ = (0.0, 1.0e6), (0.0, 1.5e4)
GPU_EFF_TOL = 1e-6          # the efficiency tolerance of tests/test_gpu_adjoint.py


def vortex_case(nr, nz, Lr=LR, Lz=LZ):
    from xlab_ee_fortran_b200 import workloads as W
    return MapCase(*W.vortex_fields(nr, nz, Lr, Lz), Lr, Lz)


def series_case(nr, nz, first=900):
    """The vortex of a late snapshot of the 1024-long time series, where the operator is far from symmetric."""
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = W.series_fields_host(W.series_params(1, total=1024, first=first)[0], nr, nz, LR, LZ)[:3]
    return MapCase(A, B, C, LR, LZ)


def lattice(nr, nz, n_side=8, width=2.0, Lr=LR, Lz=LZ):
    from xlab_ee_fortran_b200 import workloads as W
    return W.heating_lattice(n_side, n_side, Lr, Lz, width * Lr[1] / (nr - 1), width * Lz[1] / (nz - 1))


# The operators of tests/test_gpu_adjoint.py
GPU_CASES = {
    "bench vortex 512x256": lambda: vortex_case(512, 256),
    "series snapshot 900, 128x64": lambda: series_case(128, 64),
    "vortex 64x48": lambda: vortex_case(64, 48),
    "vortex 256x128": lambda: vortex_case(256, 128),
}


@pytest.mark.parametrize("shape", [(40, 24), (64, 48)])
def test_functional_is_the_gradient_of_ke_gen(shape):
    case = vortex_case(*shape)
    g = ke_functional(case)
    rng = np.random.default_rng(1)
    for _ in range(4):
        psi = np.zeros(shape[::-1]); psi[1:-1, 1:-1] = rng.standard_normal((shape[1] - 2, shape[0] - 2))
        ke, ke_abs = ke_gen(psi, case.theta, case.d, case.k)
        assert abs(float((g * psi).sum()) - ke) <= 1e-13 * ke_abs, (float((g * psi).sum()), ke, ke_abs)
    assert np.all(g[0] == 0) and np.all(g[-1] == 0) and np.all(g[:, 0] == 0) and np.all(g[:, -1] == 0)


@pytest.mark.parametrize("shape", [(40, 24), (64, 48)])
def test_heating_adjoint_is_the_transpose_of_rhs_thermal(shape):
    case = vortex_case(*shape)
    nr, nz = shape
    rng = np.random.default_rng(2)
    for _ in range(4):
        lam = np.zeros((nz, nr)); lam[1:-1, 1:-1] = rng.standard_normal((nz - 2, nr - 2))
        Q = rng.standard_normal((nz - 1, nr - 1))
        lhs = float((heating_adjoint(lam, case) * Q).sum())
        f = rhs_thermal(Q, case)
        rhs = float((lam * f).sum())
        assert abs(lhs - rhs) <= 1e-13 * float(np.abs(lam * f).sum()), (lhs, rhs)


def test_adjoint_efficiencies_equal_the_direct_ones_at_bench_shape():
    """The direct efficiency of an exact field is summed twice: by the oracle's integrate_weight_B, sequentially, and with a
    correctly rounded sum (math.fsum) of the same cell terms.  The bench rows cancel hard (sum |w theta| is up to 5e5 x
    |ke_gen|), so the sequential sum alone is 1e-9 off for some of them: the adjoint is held to 1e-9 against the correctly
    rounded one and to the sequential sum's own rounding against efficiency_row."""
    import math
    import bench
    from oracle import oracle as O
    from tests.adjoint_oracle import cell_weight
    case = vortex_case(bench.NR, bench.NZ)
    heat = bench.heat_rows(64)
    adj = ExactAdjoint(case)
    rows = adj.rows(heat)
    psi = ExactSolver(case.coe).solve(np.stack([case.forcing(r) for r in heat]))
    s = float(case.k["g0"]) / float(case.k["theta0"])
    W = cell_weight(case.g)
    worst = worst_seq = 0.0
    for n, row in enumerate(heat):
        d = efficiency_row(psi[n], row, case)
        _, ke_abs = ke_gen(psi[n], case.theta, case.d, case.k)
        wth = O.cal_wtheta(O.cal_uw(psi[n], case.d)[1], case.theta, case.d)
        eff = math.fsum((wth * W).ravel()) * s / d["sum_Q"]
        assert rows[n, 0] == pytest.approx(d["sum_Q"], rel=1e-12)
        e = abs(rows[n, 2] - eff) / abs(eff)
        worst = max(worst, e)
        assert e < 1e-9, (n, e)
        e_seq = abs(rows[n, 2] - d["efficiency"]) * abs(d["sum_Q"]) / ke_abs
        worst_seq = max(worst_seq, e_seq)
        assert e_seq < 1e-13, (n, e_seq)
    print(f"exact adjoint against exact direct efficiencies, 64 bench rows: largest relative gap {worst:.2e} (correctly "
          f"rounded direct sums); {worst_seq:.2e} of sum |w theta| against efficiency_row")


def test_solving_with_L_instead_of_LT_misses_by_far_more_than_the_gpu_tolerance():
    """For each operator of the GPU tests: ||A - A^T|| / ||A||, and how far efficiencies from an adjoint solved with L
    itself land from the right ones.  The GPU tests can only catch a missing transpose on an operator where that miss is
    over 100 x their tolerance.  Every one of them is (the bench vortex, the most nearly symmetric, by 3e3 x)."""
    misses = {}
    for name, make in GPU_CASES.items():
        case = make()
        nz, nr = case.coe.shape[:2]
        heat = lattice(nr, nz)
        right = ExactAdjoint(case).rows(heat)[:, 2]
        wrong = ExactAdjoint(case, transpose=False).rows(heat)[:, 2]
        miss = float(np.max(np.abs(wrong - right) / np.abs(right)))
        misses[name] = miss
        print(f"{name}: ||A - A^T||_F / ||A||_F = {asymmetry(case.coe):.3e}; efficiencies with L for L^T miss by up to "
              f"{miss:.2e} ({miss / GPU_EFF_TOL:.1e} x the GPU tolerance)")
    assert all(m > 100 * GPU_EFF_TOL for m in misses.values()), misses
