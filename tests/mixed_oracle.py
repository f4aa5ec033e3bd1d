"""CPU restatement (numpy, test infrastructure only) of the mixed-precision two-level method of csrc/xee_mixed.cuh
(XEE_METHOD_LINE2_MIXED): fp64 iterative refinement around fp32 two-level block-line Chebyshev sweeps.

Outer loop, fp64: r = f - L psi (the nine-term sum on the fp64 operator), s a power of two, r32 = fp32(r / s), then
psi += s (e + P c).  Inner loop: check_step two-level Chebyshev sweeps on L32 e = r32 from e = 0, step by step as
tests/twolevel_oracle.py restates them but with the fields, the residual and the update in float32 on the operator rounded
to float32; the coarse vectors c, the Galerkin inverse (of the fp64 operator) and the Chebyshev parameters stay fp64, as in
the library.  The iterate is kept as the library keeps it: a float32 field y and a coarse vector c, e = y + P c.
"""
import math

import numpy as np

from tests import line_oracle as LO
from tests.twolevel_oracle import TwoLevel

f32 = np.float32


def cheb_omega(k, rho):
    """omega_k of csrc/xee_kernels.cuh::cheb_omega (fp64)."""
    if k <= 1:
        return 1.0
    sg = 1.0 / rho
    q = sg - math.sqrt(sg * sg - 1.0)
    q2k = q ** (2.0 * (k - 1))
    return (2.0 / rho) * q * (1.0 + q2k) / (1.0 + q2k * q * q)


def pow2_above(rms):
    """The power of two with rms in [s/2, s); 1 for a zero or non-finite rms (mixed_scale_kernel)."""
    if not (rms > 0.0 and math.isfinite(rms)):
        return 1.0
    return math.ldexp(1.0, math.frexp(rms)[1])


def rms(r):
    return float(np.sqrt((np.asarray(r, np.float64)[1:-1, 1:-1] ** 2).mean()))


class Mixed:
    def __init__(self, coe):
        self.coe = np.asarray(coe, np.float64)
        self.coe32 = self.coe.astype(f32)
        self.tl = TwoLevel(self.coe)                       # P, and Ac^-1 of the fp64 operator
        self.fac32 = LO.factors(self.coe32)                # block-line factors of the rounded operator
        self.zero = np.zeros(self.coe.shape[:2])

    def residual(self, psi, f):
        """r = f - L psi (fp64), 0 on the rim."""
        return -LO.residual(np.asarray(psi, np.float64), self.coe, np.asarray(f, np.float64))

    def inner(self, r32, rho, gamma, k):
        """k fp32 two-level Chebyshev sweeps on L32 e = r32 from e = 0 with Chebyshev radius rho and step gamma.
        Returns (y, c): e = y + P c."""
        ny, nx = r32.shape
        ncz, ncx = self.tl.shape
        y, ym = np.zeros((ny, nx), f32), np.zeros((ny, nx), f32)
        c, cm = np.zeros((ncz, ncx)), np.zeros((ncz, ncx))
        g32 = f32(gamma)
        for j in range(1, k + 1):
            om = f32(cheb_omega(j, rho))
            x = (y + self.tl.prolong(c).astype(f32)).astype(f32)
            xm = (ym + self.tl.prolong(cm).astype(f32)).astype(f32)
            res = LO.residual(x, self.coe32, r32).astype(f32)                 # L32 e - r32
            z = LO.correction(res.astype(np.float64), self.coe32, self.fac32).astype(f32)
            yn = (om * ((x - g32 * z).astype(f32) - xm) + xm).astype(f32)
            cn = -float(om) * gamma * (self.tl.Aci @ self.tl.restrict(res.astype(np.float64)).ravel()).reshape(self.tl.shape)
            y, ym, c, cm = yn, y, cn, c
        return y, c

    def run(self, psi0, f, rho, gamma, check_step, sweeps):
        """`sweeps` fp32 sweeps in refinement steps of check_step from psi0 (its rim is the Dirichlet data); a partial last
        step is applied.  Returns dict(psi, checks = RMS of the fp64 residual after every full step, corrections = the
        fp64 corrections s (e + P c) of every step)."""
        psi = np.array(psi0, np.float64)
        r = self.residual(psi, f)
        s = pow2_above(rms(r))
        r32 = (r / s).astype(f32)
        nxt = s
        checks, corr = [], []
        done = 0
        while done < sweeps:
            k = min(check_step, sweeps - done)
            y, c = self.inner(r32, rho, gamma, k)
            d = s * (y.astype(np.float64) + self.tl.prolong(c))
            d[0] = d[-1] = 0.0; d[:, 0] = d[:, -1] = 0.0
            psi = psi + d
            corr.append(d)
            done += k
            if k < check_step:
                break
            r = self.residual(psi, f)
            checks.append(rms(r))
            r32 = (r / nxt).astype(f32)
            s, nxt = nxt, pow2_above(checks[-1])
        return dict(psi=psi, checks=checks, corrections=corr)
