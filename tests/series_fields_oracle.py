"""Oracle-side restatement of the time series on caller-supplied fields (TimeSeries.run_fields) from the C++ oracle's
routines: per snapshot A, B, C on the O grid, the heating Q and the momentum forcing F on the B cells and the Dirichlet rim
of psi_bc, solved exactly by sparse LU (tests/exact_oracle.py) instead of iterated."""
import numpy as np

from oracle import numpy_ref as N
from oracle import oracle as O
from tests.exact_oracle import ExactSolver
from tests.map_oracle import background_theta


class FieldSnapshot:
    """Operator, theta, m2 and forcing f of one snapshot, all in fp64 from the oracle's routines."""

    def __init__(self, A, B, C, Q, F, Lr, Lz):
        dt = np.float64
        nz, nr = np.shape(A)
        self.d = O.Domain(Lr, Lz, nr, nz, 0, 0)
        self.g = O.geometry(self.d, dt)
        self.k = N.constants(dt)
        A, B, C = (np.asarray(x, dt) for x in (A, B, C))
        a, b, c = O.build_abc(A, B, C, self.d)
        self.coe, _ = O.cal_coe(a, b, c, self.g["dr"], self.g["dz"], nr, nz)
        self.theta = background_theta(A, B, C, self.d, dt)
        _, _, _, rhoC_C = O.stagger_averages(A, B, C, self.d)
        self.m2 = O.angular_momentum_sq(rhoC_C, self.d)
        self.Q = np.asarray(Q, dt)
        self.f = O.rhs_thermal(self.Q, self.d)[1]
        if F is not None:
            self.f = self.f + O.rhs_momentum(self.m2, np.asarray(F, dt), self.d)

    def diagnostics(self, psi):
        """u, w and the table columns sum_Q, ke_gen, efficiency, max|w|, max|u| of a field psi, plus the integral of |w theta|
        (the scale of ke_gen's rounding error)."""
        u, w = O.cal_uw(np.asarray(psi, np.float64), self.d)
        wth = O.cal_wtheta(w, self.theta, self.d)
        s = float(self.k["g0"]) / float(self.k["theta0"])
        sum_q = O.integrate_weight_B(self.Q, self.d)
        ke = O.integrate_weight_B(wth, self.d) * s
        with np.errstate(divide="ignore", invalid="ignore"):
            eff = ke / sum_q
        return dict(u=u, w=w, sum_Q=sum_q, ke_gen=ke, efficiency=eff, w_absmax=float(np.abs(w).max()),
                    u_absmax=float(np.abs(u).max()), abs_wtheta=O.integrate_weight_B(np.abs(wth), self.d) * s)


def series_fields_rows(A, B, C, Q, F, psi_bc, Lr, Lz):
    """A, B, C, psi_bc [n, nz, nr], Q, F [n, nz-1, nr-1] (F and psi_bc may be None).  Returns dict(table [n, 5] with columns
    sum_Q, ke_gen, efficiency, max|w|, max|u|, psi, f, theta, u, w, m2, abs_wtheta) with psi the exact solution of L psi = f
    whose rim is the rim of psi_bc."""
    out = {q: [] for q in ("table", "psi", "f", "theta", "u", "w", "m2", "abs_wtheta")}
    for n in range(np.shape(A)[0]):
        s = FieldSnapshot(A[n], B[n], C[n], Q[n], None if F is None else F[n], Lr, Lz)
        psi = ExactSolver(s.coe).solve(s.f, bc=None if psi_bc is None else psi_bc[n])
        r = s.diagnostics(psi)
        out["table"].append([r["sum_Q"], r["ke_gen"], r["efficiency"], r["w_absmax"], r["u_absmax"]])
        for q, v in (("psi", psi), ("f", s.f), ("theta", s.theta), ("u", r["u"]), ("w", r["w"]), ("m2", s.m2),
                     ("abs_wtheta", r["abs_wtheta"])):
            out[q].append(v)
    return {q: np.array(v) for q, v in out.items()}
