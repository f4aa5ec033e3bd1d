"""CPU checks of the numpy restatement of line2_mixed (tests/mixed_oracle.py): it reaches the sparse-LU solution, one exact
refinement step with the operator rounded to fp32 contracts the bench operator's residual by 1e-6 or more, and refinement
steps far too short to converge still reduce the residual."""
import numpy as np

from tests.exact_oracle import ExactSolver, MapCase, assemble, rim_rhs, rms_interior
from tests.mixed_oracle import Mixed
from tests.test_twolevel_oracle import _operator
from tests.util import rel_l2


def _cheb(m, lmax=2.04):
    """(rho, gamma) as the library estimates them for the two-level methods: lmax = 1.02 * 2, lmin from the power iteration
    of I - M^-1 L / lmax, the real interval [1 - gamma lmax, 1 - gamma lmin]; 2 % margin on the gap."""
    rho0 = m.tl.spectral_radius(1.0 / lmax, iters=300)
    lmin = 0.98 * (1.0 - rho0) * lmax
    gamma = 2.0 / (lmax + lmin)
    return (lmax - lmin) / (lmax + lmin), gamma


def _case(nx=128, ny=66):
    coe = _operator(nx, ny)
    yy, xx = np.mgrid[0:ny, 0:nx]
    f = np.exp(-((xx - 40.0) / 9.0) ** 2 - ((yy - 30.0) / 6.0) ** 2)
    return coe, f


def test_restatement_reaches_the_exact_solution():
    coe, f = _case()
    m = Mixed(coe)
    rho, gamma = _cheb(m)
    out = m.run(np.zeros_like(f), f, rho, gamma, 80, 80 * 7)
    tol = 1e-12 * rms_interior(f)
    k = next(q for q, c in enumerate(out["checks"]) if c < tol)
    assert k <= 5, out["checks"]
    assert all(b < a for a, b in zip(out["checks"][:k], out["checks"][1:k + 1])), out["checks"]
    x = ExactSolver(coe).solve(f)
    assert rel_l2(out["psi"], x) < 1e-10, rel_l2(out["psi"], x)


def test_exact_fp32_operator_step_contracts_the_bench_residual():
    """x += A32^-1 (b - A64 x) with the bench map operator (512 x 256) rounded to fp32 and factored exactly: the inner solve
    is exact, so what is left is the cost of the rounded operator alone (scripts/prototypes/mixed_refine.py)."""
    import scipy.sparse.linalg as spla

    import bench
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    A64 = assemble(case.coe)
    lu32 = spla.splu(assemble(case.coe.astype(np.float32).astype(np.float64)))
    for row in bench.heat_rows(512)[::128]:
        b = rim_rhs(case.coe, case.forcing(row)).ravel()
        x = np.zeros_like(b)
        r0 = np.sqrt((b ** 2).mean())
        x += lu32.solve(b - A64 @ x)
        r1 = np.sqrt(((b - A64 @ x) ** 2).mean())
        assert r1 <= 1e-6 * r0, (row, r1 / r0)


def test_too_short_steps_still_reduce_the_residual():
    """Three sweeps per step, far from the ~80 a step needs here: the residual first grows (the block-line correction
    amplifies its rough part) but the steps keep reducing it and nothing diverges."""
    from tests.mixed_oracle import rms
    coe, f = _case()
    m = Mixed(coe)
    rho, gamma = _cheb(m)
    r0 = rms(m.residual(np.zeros_like(f), f))
    c = m.run(np.zeros_like(f), f, rho, gamma, 3, 3 * 30)["checks"]
    assert len(c) == 30 and np.all(np.isfinite(c))
    assert max(c) < 10 * r0 and c[-1] < 0.05 * r0, (r0, c)
    assert all(b < a for a, b in zip(c[::2], c[2::2])), c
