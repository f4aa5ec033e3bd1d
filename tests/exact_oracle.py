"""Exact discrete reference (CPU, fp64, test infrastructure only): the interior nine-point operator of do_elliptic
(xtt-lib-fortran/elliptic_tools.f90:77-85) assembled as a sparse matrix and solved by sparse LU with one step of iterative
refinement.  Every iterative method of the library converges to this solution; comparing against it measures how far a
returned field is from the answer, not from another iteration.

The slot order is tests/line_oracle.py::_OFFS: slots 1-3 at j+1, 4-6 at j, 7-9 at j-1, each at (i-1, i, i+1).  Values on
the rim are Dirichlet data and move to the right-hand side (the time series pumps through its bottom row).
"""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import numpy_ref as N
from oracle import oracle as O
from tests.line_oracle import _OFFS
from tests.map_oracle import background_theta, heat_field


def _interior_index(ny, nx):
    return np.arange((ny - 2) * (nx - 2)).reshape(ny - 2, nx - 2)


def assemble(coe):
    """The interior operator of a (ny, nx, 9) coe array as a CSC matrix on the (ny-2)(nx-2) interior unknowns (row-major).
    Couplings to rim points are left out: they belong to the right-hand side (see rim_rhs)."""
    coe = np.asarray(coe, np.float64)
    ny, nx = coe.shape[:2]
    idx = _interior_index(ny, nx)
    J, I = np.mgrid[1:ny - 1, 1:nx - 1]
    rows, cols, vals = [], [], []
    for k, (di, dj) in enumerate(_OFFS):
        jj, ii = J + dj, I + di
        inner = (jj >= 1) & (jj <= ny - 2) & (ii >= 1) & (ii <= nx - 2)
        rows.append(idx[inner])
        cols.append(idx[jj[inner] - 1, ii[inner] - 1])
        vals.append(coe[1:-1, 1:-1, k][inner])
    n = idx.size
    return sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))


def rim_rhs(coe, f, bc=None):
    """Right-hand side of the interior system: f minus the couplings of every interior point to the rim values of `bc`."""
    f = np.asarray(f, np.float64)
    b = f[1:-1, 1:-1].copy()
    if bc is None:
        return b
    ny, nx = f.shape
    rim = np.array(bc, np.float64, copy=True)
    rim[1:-1, 1:-1] = 0.0
    for k, (di, dj) in enumerate(_OFFS):
        b -= coe[1:-1, 1:-1, k] * rim[1 + dj:ny - 1 + dj, 1 + di:nx - 1 + di]
    return b


class ExactSolver:
    """splu of one operator, reused for any number of right-hand sides."""

    def __init__(self, coe):
        self.coe = np.asarray(coe, np.float64)
        self.ny, self.nx = self.coe.shape[:2]
        self.A = assemble(self.coe)
        self.lu = spla.splu(self.A)
        self.last_refinement = None      # per field: |x_refined - x_lu| / |x_refined| of the last solve()

    def solve(self, f, bc=None, chunk=64):
        """f (ny, nx) or (n, ny, nx) -> psi of the same shape, with the rim of `bc` (0 if None) and the interior solving
        L psi = f exactly (LU, then one step of iterative refinement in fp64)."""
        f = np.asarray(f, np.float64)
        single = f.ndim == 2
        F = f[None] if single else f
        BC = None if bc is None else (np.asarray(bc, np.float64)[None] if single else np.asarray(bc, np.float64))
        n = F.shape[0]
        out = np.zeros((n, self.ny, self.nx))
        if BC is not None:
            out[:] = BC
            out[:, 1:-1, 1:-1] = 0.0
        ref = np.zeros(n)
        for a in range(0, n, chunk):
            ks = range(a, min(a + chunk, n))
            B = np.stack([rim_rhs(self.coe, F[k], None if BC is None else BC[k]).ravel() for k in ks], axis=1)
            X = self.lu.solve(B)
            dX = self.lu.solve(B - self.A @ X)
            X += dX
            ref[a:a + len(ks)] = np.sqrt((dX ** 2).sum(axis=0)) / np.maximum(np.sqrt((X ** 2).sum(axis=0)), 1e-300)
            for q, k in enumerate(ks):
                out[k, 1:-1, 1:-1] = X[:, q].reshape(self.ny - 2, self.nx - 2)
        self.last_refinement = ref
        return out[0] if single else out


def host_residual_rms(psi, coe, f):
    """rms over the interior of L psi - f, summed in long double on the host (not the library's apply kernel)."""
    ld = np.longdouble
    psi = np.asarray(psi, np.float64).astype(ld)
    coe = np.asarray(coe, np.float64)
    ny, nx = psi.shape
    acc = np.zeros((ny - 2, nx - 2), ld)
    for k, (di, dj) in enumerate(_OFFS):
        acc += coe[1:-1, 1:-1, k].astype(ld) * psi[1 + dj:ny - 1 + dj, 1 + di:nx - 1 + di]
    r = acc - np.asarray(f, np.float64)[1:-1, 1:-1].astype(ld)
    return float(np.sqrt((r * r).sum() / ld(r.size)))


def rms_interior(f):
    f = np.asarray(f, np.float64)
    return float(np.sqrt((f[1:-1, 1:-1] ** 2).mean()))


# ------------------------------------------------------------------ efficiency-map rows from a given field
class MapCase:
    """Host-side pieces of one efficiency map (vortex A, B, C as float32, like EfficiencyMap): domain, geometry, operator,
    background theta and the adjoint right-hand side, all in fp64 from the oracle's routines."""

    def __init__(self, A32, B32, C32, Lr, Lz, density_mode=0):
        nz, nr = A32.shape
        dt = np.float64
        self.d = O.Domain(Lr, Lz, nr, nz, density_mode, 0)
        self.g = O.geometry(self.d, dt)
        self.k = N.constants(dt)
        A, B, C = (np.asarray(x, np.float32).astype(dt) for x in (A32, B32, C32))
        a, b, c = O.build_abc(A, B, C, self.d)
        self.coe, _ = O.cal_coe(a, b, c, self.g["dr"], self.g["dz"], nr, nz)
        self.theta = background_theta(A, B, C, self.d, dt)
        _, _, rBB, _ = O.stagger_averages(A, B, C, self.d)
        self.fchi = O.rhs_from_B(rBB, self.d)

    def heat(self, row):
        return heat_field(row, self.g, np.float64)

    def forcing(self, row, dtype=np.float64):
        """f of one heating location: rhs_thermal of its heating field, evaluated in `dtype` (grid coordinates included)."""
        g = self.g if dtype == np.float64 else O.geometry(self.d, dtype)
        return O.rhs_thermal(heat_field(row, g, dtype), self.d)[1]

    def eta(self, chi):
        return O.cal_eta(np.asarray(chi, np.float64), self.d)


def ke_gen(psi, theta, d, k):
    """(g0/theta0) I[w theta] of a field psi and the integral of |w theta| (the scale of its rounding error)."""
    _, w = O.cal_uw(np.asarray(psi, np.float64), d)
    wth = O.cal_wtheta(w, theta, d)
    s = float(k["g0"]) / float(k["theta0"])
    return O.integrate_weight_B(wth, d) * s, O.integrate_weight_B(np.abs(wth), d) * s


def efficiency_row(psi, row, case, eta=None):
    """Table columns sum_Q, ke_gen, efficiency and efficiency_eta (None without eta) of the field psi at heating row."""
    Q = case.heat(row)
    sum_q = O.integrate_weight_B(Q, case.d)
    ke, _ = ke_gen(psi, case.theta, case.d, case.k)
    out = dict(sum_Q=sum_q, ke_gen=ke, efficiency=ke / sum_q, efficiency_eta=None)
    if eta is not None:
        out["efficiency_eta"] = O.cal_sum_Qeta(Q, np.asarray(eta, np.float64), case.d) / sum_q
    return out
