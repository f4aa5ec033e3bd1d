"""Oracle-side restatement of the time series' legacy efficiency decomposition (TimeSeries.decompose,
xee_series_decompose_*): the chain of tests/legacy_oracle.decompose (src/old-diagnose/diagnose.f90:238-841) with the
library's stated deviations, every solve exact by sparse LU (tests/exact_oracle.py) from its rim with a zero interior, and
the exchange conversion on the working-precision fields.  Arrays are [j][i]."""
import numpy as np

from oracle import numpy_ref as N
from oracle import oracle as O
from tests.exact_oracle import ExactSolver
from tests.legacy_oracle import exchange_conversion

TERMS = ("eta_bc", "eta_dB", "eta_B0", "bndconv", "bndconv2", "etaQ", "wtheta")
COLS = ("sum_Q", "sum_dtheta_dt", "local_heat_response") + tuple(f"{t}_0" for t in TERMS) + tuple(f"{t}_B0dB" for t in TERMS)
SOLVES = ("psi_before", "chi_0_0", "chi_B0dB_0", "chi_0_dB", "chi_B0dB_dB", "chi_0_B0", "chi_B0dB_B0", "psi_after_0",
          "psi_after_B0dB")


def _rim(x, shape):
    out = np.zeros(shape)
    if x is not None:
        out[[0, -1], :] = np.asarray(x, np.float64)[[0, -1], :]
        out[:, [0, -1]] = np.asarray(x, np.float64)[:, [0, -1]]
    return out


def decompose_exact(A, B, C, Q, F, psi_bc, chi_bc, Lr, Lz, testing_dt=None, baro=2):
    """One snapshot.  testing_dt None = INSTANT.  Returns (row [17] in COLS order with NaN where not computed,
    fields {name: array} with dtheta_dt, theta_after and the fields of SOLVES that were computed)."""
    dt = np.float64
    nz, nr = np.shape(A)
    d = O.Domain(Lr, Lz, nr, nz, 0, 0)
    g = O.geometry(d, dt)
    k = N.constants(dt)
    g0, th0 = k["g0"], k["theta0"]
    ra, za, rho = g["ra"], g["za"], g["rho"]
    A, B, C, Q = (np.asarray(x, dt) for x in (A, B, C, Q))
    intB = lambda w: O.integrate_weight_B(np.ascontiguousarray(w), d)
    a, b_basic_s, c = O.build_abc(A, B, C, d)
    rA, rBC, rBB, rCC = O.stagger_averages(A, B, C, d)
    b_basic = rBB.copy()
    J, f = O.rhs_thermal(Q, d)
    if F is not None:
        f = f + O.rhs_momentum(O.angular_momentum_sq(rCC, d), np.asarray(F, dt), d)
    coe_of = lambda bb: O.cal_coe(a, bb, c, g["dr"], g["dz"], nr, nz)[0]
    psi0 = _rim(psi_bc, (nz, nr))
    fields, row = {}, dict.fromkeys(COLS, np.nan)
    row["sum_Q"] = intB(Q)
    b_anom = np.zeros_like(rBB)
    if testing_dt is not None:
        rpsi = ExactSolver(coe_of(b_basic_s)).solve(f, bc=psi0)
        fields["psi_before"] = rpsi
        u, w = O.cal_uw(rpsi, d)
        th = J - th0 / g0 * (rA[:-1] * w[:-1] + rA[1:] * w[1:]) / 2.0 + th0 / g0 * (rBC[:, :-1] * u[:, :-1] + rBC[:, 1:] * u[:, 1:]) / 2.0
        fields["dtheta_dt"] = th.copy()
        row["sum_dtheta_dt"] = intB(th)
        row["local_heat_response"] = row["sum_dtheta_dt"] / row["sum_Q"]
        th = th * testing_dt
        dB = np.zeros_like(th)                                       # d_dr_B2B
        dB[:, 1:-1] = (th[:, :-2] - th[:, 2:]) / (ra[:-3] - ra[2:-1])[None, :]
        dB[:, 0] = (th[:, 0] - th[:, 1]) / (ra[0] - ra[1]); dB[:, -1] = (th[:, -2] - th[:, -1]) / (ra[-3] - ra[-2])
        b_anom = -g0 / th0 * dB
        rBB = rBB + b_anom
        dA = np.zeros((nz, nr - 1))                                   # d_dz_B2A on rows 2..nz-2, 0 elsewhere
        dA[1:nz - 2] = (th[1:nz - 2] - th[0:nz - 3]) / ((za[2:nz - 1] - za[0:nz - 3]) / 2.0)[:, None]
        rA = rA.copy(); rA[1:nz - 1] = rA[1:nz - 1] + g0 / th0 * dA[1:nz - 1]
    rBC = rBC.copy(); rBC[:, 1:-1] = (rBB[:, :-1] + rBB[:, 1:]) / 2.0
    theta = O.relative_theta(rA * (th0 / g0), rBC * (-th0 / g0), d)
    fields["theta_after"] = theta
    rs = ((ra[:-1] + ra[1:]) / 2.0)[None, :]; rr = ((rho[:-1] + rho[1:]) / 2.0)[:, None]
    rhs = dict(bc=np.zeros((nz, nr)), dB=O.rhs_from_B(b_anom, d), B0=O.rhs_from_B(b_basic, d))
    ops = dict(zip(("0", "B0dB"), (np.zeros_like(b_basic_s), b_basic_s + b_anom / rs / rr)))
    for t, tag in enumerate(("0", "B0dB")):
        if baro == 1 - t:                                             # baro 1 excludes tag 0, baro 0 excludes tag B0dB
            continue
        sol = ExactSolver(coe_of(ops[tag]))
        for kind in ("bc", "dB", "B0"):
            if kind == "bc" and chi_bc is None:
                continue
            chi = sol.solve(rhs[kind], bc=_rim(chi_bc, (nz, nr)) if kind == "bc" else None)
            fields[f"chi_{tag}_{kind.replace('bc', '0')}"] = chi
            row[f"eta_{kind}_{tag}"] = O.cal_sum_Qeta(Q, O.cal_eta(chi, d), d)
        rpsi = sol.solve(f, bc=psi0)
        fields[f"psi_after_{tag}"] = rpsi
        row[f"wtheta_{tag}"] = intB(O.cal_wtheta(O.cal_uw(rpsi, d)[1], theta, d)) * g0 / th0
        etaq = (0.0 if chi_bc is None else row[f"eta_bc_{tag}"]) + row[f"eta_dB_{tag}"] + row[f"eta_B0_{tag}"]
        if chi_bc is not None:
            chi3 = fields[f"chi_{tag}_0"] + fields[f"chi_{tag}_dB"] + fields[f"chi_{tag}_B0"]
            chi2 = fields[f"chi_{tag}_dB"] + fields[f"chi_{tag}_B0"]
            row[f"bndconv_{tag}"] = exchange_conversion(rpsi, chi3, C, g)[1]
            row[f"bndconv2_{tag}"] = exchange_conversion(rpsi, chi2, C, g)[1]
            etaq = etaq + row[f"bndconv_{tag}"]
        row[f"etaQ_{tag}"] = etaq
    return np.array([row[q] for q in COLS]), fields


def decompose_rows(A, B, C, Q, F, psi_bc, chi_bc, Lr, Lz, testing_dt=None, baro=2):
    """decompose_exact of every snapshot of [n, ...] arrays (F, psi_bc, chi_bc may be None).  Returns (table [n, 17],
    list of field dicts)."""
    rows, fields = [], []
    pick = lambda x, n: None if x is None else x[n]
    for n in range(np.shape(A)[0]):
        r, f = decompose_exact(A[n], B[n], C[n], Q[n], pick(F, n), pick(psi_bc, n), pick(chi_bc, n), Lr, Lz, testing_dt, baro)
        rows.append(r); fields.append(f)
    return np.array(rows), fields
