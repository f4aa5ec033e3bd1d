"""The exact sparse-LU reference (tests/exact_oracle.py) checked against the oracle itself, on the CPU: its solutions
satisfy do_elliptic's equations to round-off, and the reference's own Jacobi iteration converges to them."""
import numpy as np
import pytest

from tests.exact_oracle import ExactSolver, MapCase, assemble, host_residual_rms, rms_interior


def _random_case(nx, ny, seed):
    """Diagonally dominant random operator (like the library's random test operators), random forcing and rim values."""
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    a = 1.0 + rng.random((ny - 2, nx - 1)); c = 1.0 + rng.random((ny - 1, nx - 2)); b = 0.05 * rng.standard_normal((ny - 1, nx - 1))
    coe, err = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    assert err == 0
    f = rng.standard_normal((ny, nx)); bc = rng.standard_normal((ny, nx))
    return coe, f, bc


@pytest.mark.parametrize("shape", [(48, 40), (67, 35)])
def test_lu_solution_satisfies_do_elliptic(shape):
    from oracle import oracle as O
    nx, ny = shape
    coe, f, bc = _random_case(nx, ny, seed=nx)
    ex = ExactSolver(coe)
    assert ex.A.shape == ((nx - 2) * (ny - 2),) * 2 and ex.A.nnz == 9 * (nx - 4) * (ny - 4) + 6 * 2 * ((nx - 4) + (ny - 4)) + 4 * 4
    psi = ex.solve(f, bc)
    rim = np.ones((ny, nx), bool); rim[1:-1, 1:-1] = False
    assert np.array_equal(psi[rim], bc[rim])                             # Dirichlet values are kept
    res = O.do_elliptic(psi, coe) - f
    assert rms_interior(res) <= 1e-13 * rms_interior(f), rms_interior(res) / rms_interior(f)
    assert host_residual_rms(psi, coe, f) <= 1e-13 * rms_interior(f)
    # the rim really enters: the same forcing without rim values gives a different field
    assert np.abs(ex.solve(f) - psi)[1:-1, 1:-1].max() > 1e-3 * np.abs(psi).max()
    # a batch of right-hand sides gives each single solution
    both = ex.solve(np.stack([f, 2.0 * f]), np.stack([bc, bc]))
    assert np.array_equal(both[0], psi) and rms_interior(O.do_elliptic(both[1], coe) - 2.0 * f) <= 1e-13 * rms_interior(2.0 * f)


def test_host_residual_is_the_nine_point_sum():
    """host_residual_rms agrees with do_elliptic's residual on a field that is not a solution."""
    from oracle import oracle as O
    coe, f, bc = _random_case(37, 29, seed=5)
    x = np.random.default_rng(1).standard_normal(f.shape)
    ref = rms_interior(O.do_elliptic(x, coe) - f)
    assert abs(host_residual_rms(x, coe, f) - ref) <= 1e-14 * ref


def test_reference_jacobi_converges_to_the_lu_solution():
    """Small, well-conditioned case: the oracle's STRICT Jacobi run to a tight tolerance lands on the LU solution within
    the error its own residual allows, |x - x*| <= |A^-1| |r|."""
    from oracle import oracle as O
    nx, ny = 20, 16
    coe, f, bc = _random_case(nx, ny, seed=3)
    ex = ExactSolver(coe)
    psi = ex.solve(f, bc)
    r1 = 1e-13 * rms_interior(f)
    it = O.solve_elliptic(400000, 50, 2, 5, r1, 0.0, 1.0, bc, coe, f)
    assert it["err"] == 0
    xj = it["dat"]
    r = (O.do_elliptic(xj, coe) - f)[1:-1, 1:-1].ravel()
    ainv = np.linalg.norm(np.linalg.inv(assemble(coe).toarray()), 2)
    err = np.linalg.norm((xj - psi)[1:-1, 1:-1])
    assert err <= 1.01 * ainv * np.linalg.norm(r) + 1e-14 * np.linalg.norm(psi), (err, ainv * np.linalg.norm(r))
    assert err <= 1e-11 * np.linalg.norm(psi)


def test_bench_operator_is_solved_to_round_off():
    """The benchmark's operator (vortex fields, 512 x 256) and four of its heating locations: residual and refinement
    change at round-off level (measured 2.5e-15 rms(f) and 1.8e-13)."""
    import bench
    from oracle import oracle as O
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    ex = ExactSolver(case.coe)
    rows = bench.heat_rows(4)
    F = np.stack([case.forcing(r) for r in rows])
    psi = ex.solve(F)
    print("refinement change", ex.last_refinement)
    assert np.all(ex.last_refinement <= 1e-12)
    for n in range(len(rows)):
        rf = rms_interior(F[n])
        res = rms_interior(O.do_elliptic(psi[n], case.coe) - F[n])
        assert res <= 1e-14 * rf, res / rf
        assert np.all(psi[n][0] == 0) and np.all(psi[n][-1] == 0) and np.all(psi[n][:, 0] == 0) and np.all(psi[n][:, -1] == 0)
