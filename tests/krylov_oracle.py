"""CPU restatement (numpy, fp64, test infrastructure only) of the BiCGStab methods of csrc/xee_krylov.cuh.

Right-preconditioned BiCGStab on A = L with K^-1 = M^-1 (line_bicgstab: tests/line_oracle.py's block-line correction) or
K^-1 = M^-1 + P Ac^-1 P^T (line2_bicgstab: tests/twolevel_oracle.py's two-level correction), step for step as the library
runs it: internally r = f - L x; on a check iteration (k % check_step == 0) the true residual replaces the recurrence
residual; a breakdown (|rho'| <= 1e-30 |r0| |r|, omega = 0, or a non-finite alpha, omega or beta) restarts from the current
iterate with r0 = p = r, and a bad alpha or omega counts as 0 for the rest of its iteration.
"""
import numpy as np

from tests import line_oracle as LO
from tests.twolevel_oracle import TwoLevel


def _dot(a, b):
    return np.float64(np.dot(a.ravel(), b.ravel()))   # IEEE division: 0/0 is NaN, not an exception


class Krylov:
    def __init__(self, coe, two_level):
        self.coe = np.asarray(coe, np.float64)
        ny, nx = self.coe.shape[:2]
        self.zero = np.zeros((ny, nx))
        if two_level:
            self.precond = TwoLevel(self.coe).correction
        else:
            fac = LO.factors(self.coe)
            self.precond = lambda v: LO.correction(v, self.coe, fac)

    def L(self, x):
        """L x on the interior, 0 on the rim."""
        return LO.residual(x, self.coe, self.zero)

    def true_residual(self, x, f):
        r = np.zeros_like(self.zero)
        r[1:-1, 1:-1] = (np.asarray(f, np.float64) - self.L(x))[1:-1, 1:-1]
        return r

    def run(self, x0, f, iters, check_step, stop_rms=None):
        """`iters` iterations from x0 (its rim is the Dirichlet data).  Returns dict(x, checks = RMS of the true residual at
        every check, restarts, iters).  stop_rms: stop at the first check whose residual is below it."""
        x = np.array(x0, np.float64, copy=True)
        r = self.true_residual(x, f)
        r0, p = r.copy(), r.copy()
        rho = r0n = _dot(r, r)
        checks, restarts = [], 0
        k = 0
        with np.errstate(all="ignore"):
            for k in range(1, iters + 1):
                ph = self.precond(p)
                v = self.L(ph)
                al = rho / _dot(r0, v)
                restart = not np.isfinite(al)
                if restart:
                    al = 0.0
                s = r - al * v
                x = x + al * ph
                sh = self.precond(s)
                t = self.L(sh)
                om = _dot(t, s) / _dot(t, t)
                if not np.isfinite(om) or om == 0.0:
                    om, restart = 0.0, True
                x = x + om * sh
                r = s - om * t
                if k % check_step == 0:
                    r = self.true_residual(x, f)
                    checks.append(float(np.sqrt((r[1:-1, 1:-1] ** 2).mean())))
                rn, rr = _dot(r0, r), _dot(r, r)
                bad = restart or not np.isfinite(rn) or not (abs(rn) > 1e-30 * np.sqrt(r0n) * np.sqrt(rr))
                beta = 0.0
                if not bad:
                    beta = (rn / rho) * (al / om)
                    bad = not np.isfinite(beta)
                if bad:
                    rho = r0n = rr
                    r0, p = r.copy(), r.copy()
                    restarts += 1
                else:
                    rho = rn
                    p = r + beta * (p - om * v)
                if stop_rms is not None and k % check_step == 0 and checks[-1] < stop_rms:
                    break
        return dict(x=x, checks=checks, restarts=restarts, iters=k)


def series_problem(q, nr, nz, total=1024):
    """Operator, forcing and first guess (pumping bottom row) of snapshot q of a `total`-long time series, in fp64, as
    tests/series_oracle.py composes them."""
    import bench
    from oracle import oracle as O
    from tests.map_oracle import heat_field
    from xlab_ee_fortran_b200 import workloads as W
    row = W.series_params(1, total=total, first=q)[0]
    d = O.Domain(bench.LR, bench.LZ, nr, nz, 0, 0)
    g = O.geometry(d, np.float64)
    A32, B32, C32, bottom, F = W.series_fields_host(row, nr, nz, bench.LR, bench.LZ)
    A, B, C = (x.astype(np.float64) for x in (A32, B32, C32))
    a, b, c = O.build_abc(A, B, C, d)
    coe, _ = O.cal_coe(a, b, c, g["dr"], g["dz"], nr, nz)
    _, f_thm = O.rhs_thermal(heat_field(row[14:19], g, np.float64), d)
    _, _, _, rhoC_C = O.stagger_averages(A, B, C, d)
    f = f_thm + O.rhs_momentum(O.angular_momentum_sq(rhoC_C, d), F.astype(np.float64), d)
    psi0 = np.zeros((nz, nr)); psi0[0, :] = bottom
    return coe, f, psi0
