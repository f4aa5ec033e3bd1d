"""CPU check of tests/decompose_oracle.py, the exact restatement the GPU decomposition is tested against: on a small
vortex it gives every efficiency.txt term of the legacy chain (tests/legacy_oracle.decompose, the legacy loop run to a
tight tolerance, carried first guesses, float32 round trip before the exchange conversion)."""
import numpy as np
import pytest

from tests.decompose_oracle import COLS, decompose_exact
from tests.legacy_oracle import decompose
from tests.util import rel_l2

NR, NZ = 40, 30
LR, LZ = (0.0, 5.0e5), (0.0, 1.4e4)
PSI_SET, CHI_SET = (1, 1e-22, 4000000, 1.0), (1, 1e-19, 4000000, 1.0)


def _case(momentum):
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = (x.astype(np.float64) for x in W.vortex_fields(NR, NZ, LR, LZ))
    r = np.linspace(*LR, NR); z = np.linspace(*LZ, NZ)
    Rm, Zm = np.meshgrid(0.5 * (r[:-1] + r[1:]), 0.5 * (z[:-1] + z[1:]))
    Q = 0.116 * np.exp(-((Rm - 4.0e4) / 3.0e4) ** 2 - ((Zm - 5.0e3) / 2.5e3) ** 2)
    F = -2e-5 * np.exp(-Zm / 3e3) * np.sin(np.pi * Rm / LR[1]) if momentum else np.zeros_like(Q)
    s = np.sin(np.pi * r / LR[1])
    chi_bc = np.zeros((NZ, NR)); chi_bc[-1] = 2.0e11 * s * (r / LR[1]) ** 2
    psi_bc = np.zeros((NZ, NR)); psi_bc[0] = 4.0e6 * s * (r / LR[1]) ** 2
    return A, B, C, Q, F, psi_bc, chi_bc


def _legacy_row(ref):
    """The legacy composition's sums in the column order of the decomposition table."""
    row = dict(sum_Q=ref["sum_Q"], sum_dtheta_dt=ref.get("sum_dtheta_dt", np.nan))
    row["local_heat_response"] = row["sum_dtheta_dt"] / row["sum_Q"]
    for tag in ("0", "B0dB"):
        bc = f"sum_Qeta_{tag}_0" in ref
        row[f"eta_bc_{tag}"] = ref[f"sum_Qeta_{tag}_0"] if bc else np.nan
        row[f"eta_dB_{tag}"] = ref[f"sum_Qeta_{tag}_dB"]
        row[f"eta_B0_{tag}"] = ref[f"sum_Qeta_{tag}_B0"]
        row[f"bndconv_{tag}"] = ref[f"sum_bndconv_{tag}"] if bc else np.nan
        row[f"bndconv2_{tag}"] = ref[f"sum_bndconv2_{tag}"] if bc else np.nan
        tot = (ref[f"sum_Qeta_{tag}_0"] if bc else 0.0) + ref[f"sum_Qeta_{tag}_dB"] + ref[f"sum_Qeta_{tag}_B0"]
        row[f"etaQ_{tag}"] = tot + (ref[f"sum_bndconv_{tag}"] if bc else 0.0)
        row[f"wtheta_{tag}"] = ref[f"sum_wtheta_{tag}"]
    return np.array([row[q] for q in COLS])


CASES = [(True, False, False), (True, True, False), (False, False, False), (False, True, True)]   # tendency, chi_bc, momentum


@pytest.mark.parametrize("tendency,with_bc,momentum", CASES, ids=["tendency", "tendency-chi_bc", "instant", "instant-chi_bc-F"])
def test_exact_restatement_matches_the_legacy_chain(tendency, with_bc, momentum):
    A, B, C, Q, F, psi_bc, chi_bc = _case(momentum)
    dt = 3600.0 if tendency else None
    got, fields = decompose_exact(A, B, C, Q, F, psi_bc, chi_bc if with_bc else None, LR, LZ, testing_dt=dt, baro=2)
    ref = decompose(A, B, C, Q, F, LR, LZ, dt or 0.0, PSI_SET, CHI_SET, baro=2, rchi_bc=chi_bc if with_bc else None,
                    rpsi_bc=psi_bc, tendency=tendency)
    want = _legacy_row(ref)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    if not tendency:
        assert np.isnan(got[1]) and np.isnan(got[2])
        assert np.all(fields["chi_0_dB"] == 0) and np.all(fields["chi_B0dB_dB"] == 0)
    for q, g, w in zip(COLS, got, want):
        if np.isnan(w):
            continue
        tol = 1e-5 if q.startswith("bndconv") or q.startswith("etaQ") and with_bc else 1e-6
        assert abs(g - w) <= tol * abs(w), (q, g, w)
    if tendency:                           # from psi_before: exact against converged Jacobi
        assert rel_l2(fields["dtheta_dt"], ref["dtheta_dt"]) < 1e-8
        assert rel_l2(fields["theta_after"], ref["theta_after"]) < 1e-12
    else:                                  # the background state: the same routines on the same fields
        assert np.array_equal(fields["theta_after"], ref["theta_after"])


def test_decomposition_sum_matches_the_w_theta_integral():
    """Pure heating (F = 0, no boundary terms): the eta decomposition and the w theta integral measure the same generation,
    to first order in the grid spacing (the legacy driver's integral check)."""
    A, B, C, Q, F, psi_bc, _ = _case(False)
    for dt in (3600.0, None):
        got, _ = decompose_exact(A, B, C, Q, F, None, None, LR, LZ, testing_dt=dt, baro=2)
        for tag in ("0", "B0dB"):
            eq, wt = got[COLS.index(f"etaQ_{tag}")], got[COLS.index(f"wtheta_{tag}")]
            assert abs(eq - wt) <= 0.02 * abs(wt), (dt, tag, eq, wt)


def test_baro_selects_the_operators():
    A, B, C, Q, F, psi_bc, chi_bc = _case(True)
    full, _ = decompose_exact(A, B, C, Q, F, psi_bc, chi_bc, LR, LZ, testing_dt=1800.0, baro=2)
    for baro, keep in ((0, slice(3, 10)), (1, slice(10, 17))):
        got, fields = decompose_exact(A, B, C, Q, F, psi_bc, chi_bc, LR, LZ, testing_dt=1800.0, baro=baro)
        assert np.array_equal(got[:3], full[:3]) and np.array_equal(got[keep], full[keep])
        drop = slice(10, 17) if baro == 0 else slice(3, 10)
        assert np.all(np.isnan(got[drop]))
        assert ("psi_after_B0dB" in fields) == (baro == 1) and ("psi_after_0" in fields) == (baro == 0)
