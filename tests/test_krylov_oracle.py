"""The numpy restatement of the BiCGStab methods (tests/krylov_oracle.py) against exact sparse-LU solutions
(tests/exact_oracle.py): random anisotropic operators, a late non-symmetric snapshot of the 1,024-long time series, and a
hand-built breakdown."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.exact_oracle import ExactSolver, rms_interior
from tests.krylov_oracle import Krylov, series_problem
from tests.test_gpu_twolevel import _aniso
from tests.util import rel_l2


def _converges(coe, f, x0, two_level, tol_rel=1e-12, max_iter=400, check_step=5):
    kr = Krylov(coe, two_level)
    exact = ExactSolver(coe).solve(f, x0)
    out = kr.run(x0, f, max_iter, check_step, stop_rms=tol_rel * rms_interior(f))
    res = out["checks"][-1]
    assert res < tol_rel * rms_interior(f), (out["iters"], res / rms_interior(f))
    # the error is L^-1 of the final residual: solve for it exactly and compare
    err = ExactSolver(coe).solve(kr.true_residual(out["x"], f))
    assert rel_l2(out["x"] - exact, -err) < 1e-3 + 1e-6 * np.linalg.norm(exact) / max(np.linalg.norm(err), 1e-300)
    assert rel_l2(out["x"], exact) < 1e-9, rel_l2(out["x"], exact)
    return out


@pytest.mark.parametrize("two_level", [False, True])
@pytest.mark.parametrize("seed", [3, 4])
def test_oracle_reaches_exact_solution_on_anisotropic_operators(two_level, seed):
    nx, ny = 128, 66
    a, b, c = _aniso(nx, ny, seed=seed)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    rng = np.random.default_rng(seed)
    f = rng.standard_normal((ny, nx))
    x0 = rng.standard_normal((ny, nx))
    out = _converges(coe, f, x0, two_level)
    print(f"aniso seed {seed} two_level {two_level}: {out['iters']} iterations, {out['restarts']} restarts")


@pytest.mark.parametrize("two_level", [False, True])
def test_oracle_reaches_exact_solution_on_late_series_snapshot(two_level):
    """Snapshot 1000 of 1,024 at 128 x 64: B varies strongly, the operator is several times further from symmetric than
    the first snapshot's."""
    def asymmetry(coe):
        A = ExactSolver(coe).A
        return abs(A - A.T).max() / abs(A).max()
    coe, f, x0 = series_problem(1000, 128, 64)
    asym = asymmetry(coe)
    assert asym > 5 * asymmetry(series_problem(0, 128, 64)[0]), asym
    out = _converges(coe, f, x0, two_level, max_iter=600)
    print(f"snapshot 1000 two_level {two_level}: {out['iters']} iterations, {out['restarts']} restarts, asymmetry {asym:.2e}")


@pytest.mark.parametrize("two_level", [False, True])
def test_breakdown_restarts_from_the_current_iterate(two_level):
    """A first guess that solves the problem exactly: r = 0, so rho = r0.r = 0 and alpha = 0/0 break down on every
    iteration.  Each restarts, the iterate stays exact and no NaN appears; the same plan object then solves a perturbed
    problem from there."""
    nx, ny = 64, 34
    a, b, c = _aniso(nx, ny, seed=7)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    rng = np.random.default_rng(7)
    x = rng.standard_normal((ny, nx))
    kr = Krylov(coe, two_level)
    f = np.zeros((ny, nx)); f[1:-1, 1:-1] = kr.L(x)[1:-1, 1:-1]
    assert not np.any(kr.true_residual(x, f))
    out = kr.run(x, f, 6, 3)
    assert out["restarts"] == 6 and out["checks"] == [0.0, 0.0]
    assert np.array_equal(out["x"], x)
    f2 = f + 1e-3 * rng.standard_normal((ny, nx))
    _converges(coe, f2, out["x"], two_level)
