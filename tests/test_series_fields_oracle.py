"""CPU check of tests/series_fields_oracle.py: on the fields the parametric series builds (workloads.series_fields_host),
the field restatement with sparse LU gives what the iterated parametric composition (tests/series_oracle.py) gives."""
import numpy as np

from oracle import oracle as O
from tests.map_oracle import heat_field
from tests.series_fields_oracle import series_fields_rows
from tests.series_oracle import series_rows
from tests.util import rel_l2
from xlab_ee_fortran_b200 import workloads as W


def _parametric_fields(params, nr, nz, Lr, Lz):
    g = O.geometry(O.Domain(Lr, Lz, nr, nz, 0, 0), np.float64)
    A, B, C, Q, F, bc = [], [], [], [], [], []
    for row in params:
        a, b, c, bottom, f = W.series_fields_host(row, nr, nz, Lr, Lz)
        A.append(a); B.append(b); C.append(c); F.append(f); Q.append(heat_field(row[14:19], g, np.float64))
        p = np.zeros((nz, nr)); p[0] = bottom; bc.append(p)
    return [np.array(x, np.float64) for x in (A, B, C, Q, F, bc)]


def test_field_restatement_matches_parametric_series():
    nr, nz = 40, 30
    Lr, Lz = (0.0, 6.0e5), (0.0, 1.5e4)
    params = np.concatenate([W.series_params(2, total=1024, first=0), W.series_params(1, total=1024, first=900)])
    ref = series_rows(params, nr, nz, Lr, Lz, np.float64, dict(max_iter=4000000, check_step=100, converge_time=2, r1_rel=1e-12))
    assert np.all(ref["table"][:, 2] == 0)
    A, B, C, Q, F, bc = _parametric_fields(params, nr, nz, Lr, Lz)
    got = series_fields_rows(A, B, C, Q, F, bc, Lr, Lz)
    for q in ("f", "theta", "m2"):
        assert np.array_equal(got[q], ref[q]), q                      # the same oracle routines on the same inputs
    for n in range(len(params)):
        assert np.array_equal(got["psi"][n][0], ref["psi"][n][0])      # the pumping rim is Dirichlet data
        assert rel_l2(got["psi"][n], ref["psi"][n]) < 1e-8, n          # exact against converged Jacobi
    assert np.array_equal(got["table"][:, 0], ref["table"][:, 3])      # sum_Q
    assert np.allclose(got["table"][:, 1:], ref["table"][:, 4:], rtol=1e-7, atol=0)


def test_field_restatement_without_momentum_and_rim():
    """F = None is the thermal forcing alone; psi_bc = None is a zero rim."""
    nr, nz = 24, 20
    Lr, Lz = (0.0, 6.0e5), (0.0, 1.5e4)
    A, B, C, Q, F, _ = _parametric_fields(W.series_params(1), nr, nz, Lr, Lz)
    a = series_fields_rows(A, B, C, Q, None, None, Lr, Lz)
    b = series_fields_rows(A, B, C, Q, np.zeros_like(F), np.zeros_like(A), Lr, Lz)
    d = O.Domain(Lr, Lz, nr, nz, 0, 0)
    assert np.array_equal(a["f"][0], O.rhs_thermal(Q[0], d)[1])
    assert np.array_equal(a["f"], b["f"]) and np.array_equal(a["psi"], b["psi"])
    assert np.all(a["psi"][0][[0, -1], :] == 0) and np.all(a["psi"][0][:, [0, -1]] == 0)
