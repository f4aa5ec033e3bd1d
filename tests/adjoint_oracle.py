"""Exact discrete adjoint of the efficiency map (CPU, fp64, test infrastructure only).

ke_gen of a heating Q is <g, L^-1 H Q> = <H^T L^-T g, Q>: g is the gradient of (g0/theta0) I[w theta] in psi, L the interior
nine-point operator (tests/exact_oracle.assemble), H the map Q -> f of rhs_thermal.  This file writes g and H^T down from
the oracle's definitions of w, w theta, integrate_weight_B and rhs_thermal; tests/test_adjoint_oracle.py checks both against
those routines, so neither formula is taken on trust.
"""
import numpy as np
import scipy.sparse.linalg as spla

from oracle import oracle as O
from tests.exact_oracle import assemble


def cell_weight(g):
    """W_c = rho_ rcuv dr dz of integrate_weight_B on the (nz-1, nr-1) B cells."""
    ra, rc, rho, za = (np.asarray(g[k], np.float64) for k in ("ra", "rcuva", "rho", "za"))
    rcuv = ((rc[:-1] + rc[1:]) / 2)[None, :]
    dr = (ra[1:] - ra[:-1])[None, :]
    dz = (za[1:] - za[:-1])[:, None]
    rho_ = ((rho[1:] + rho[:-1]) / 2)[:, None]
    return rho_ * rcuv * dr * dz


def ke_functional(case):
    """g (nz, nr): ke_gen(psi) = <g, psi> for every psi with a zero rim.
    w(i,j) = (psi(i+1,j) - psi(i,j)) / (dr_i rbar_i rho_j) on the A grid, w theta = theta (w(.,j) + w(.,j+1)) / 2 on B."""
    g, k = case.g, case.k
    ra, rho = np.asarray(g["ra"], np.float64), np.asarray(g["rho"], np.float64)
    nz, nr = len(g["za"]), len(ra)
    s = float(k["g0"]) / float(k["theta0"])
    c = cell_weight(g) * case.theta / ((ra[1:] - ra[:-1]) * (ra[:-1] + ra[1:]) / 2)[None, :]     # (nz-1, nr-1)
    out = np.zeros((nz, nr))
    # interior point (I, J): + cells (I-1, J-1), (I-1, J); - cells (I, J-1), (I, J)
    cs = c[:-1, :] + c[1:, :]                                                                      # cj = J-1 and J, J = 1..nz-2
    out[1:-1, 1:-1] = s / (2 * rho[1:-1, None]) * (cs[:, :-1] - cs[:, 1:])
    return out


def heating_adjoint(lam, case):
    """mu = H^T lambda (nz-1, nr-1): <lambda, rhs_thermal(Q)> = <mu, Q> for every Q on the B cells."""
    g, k = case.g, case.k
    ra, ex = np.asarray(g["ra"], np.float64), np.asarray(g["exner"], np.float64)
    lam = np.asarray(lam, np.float64).copy()
    nz, nr = lam.shape
    lam[0] = lam[-1] = 0.0; lam[:, 0] = lam[:, -1] = 0.0
    d = np.zeros(nr); d[1:-1] = (ra[2:] - ra[:-2]) / 2
    L2 = lam[:-1, :] + lam[1:, :]                                 # lambda(., cj) + lambda(., cj+1), (nz-1, nr)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(d[None, :] > 0, L2 / np.where(d > 0, d, 1.0)[None, :], 0.0)
    s = float(k["g0"]) / float(k["theta0"])
    return s / (2 * float(k["Cp"]) * ex[:-1, None]) * (t[:, :-1] - t[:, 1:])


class ExactAdjoint:
    """splu of L^T: lambda, mu and the exact discrete efficiencies of a map case (tests/exact_oracle.MapCase)."""

    def __init__(self, case, transpose=True):
        self.case = case
        A = assemble(case.coe)
        self.A = A
        self.lu = spla.splu((A.T if transpose else A).tocsc())
        self.g = ke_functional(case)
        nz, nr = self.g.shape
        b = self.g[1:-1, 1:-1].ravel()
        At = A.T if transpose else A
        x = self.lu.solve(b)
        x += self.lu.solve(b - At @ x)                     # one step of iterative refinement, as ExactSolver
        self.lam = np.zeros((nz, nr))
        self.lam[1:-1, 1:-1] = x.reshape(nz - 2, nr - 2)
        self.mu = heating_adjoint(self.lam, case)
        self.W = cell_weight(case.g)
        self.eta_d = self.mu / self.W

    def rows(self, heat):
        """[n, 3]: sum_Q, ke_gen, efficiency of each heating row, from mu."""
        out = np.zeros((len(heat), 3))
        for n, row in enumerate(heat):
            Q = self.case.heat(row)
            sq = float((self.W * Q).sum()); ke = float((self.mu * Q).sum())
            out[n] = sq, ke, ke / sq
        return out


def asymmetry(coe):
    """||A - A^T||_F / ||A||_F of the interior operator."""
    A = assemble(coe)
    return float(spla.norm(A - A.T) / spla.norm(A))


def rhs_thermal(Q, case):
    return O.rhs_thermal(np.asarray(Q, np.float64), case.d)[1]
