"""The time series on caller-supplied snapshots (TimeSeries.run_fields, xee_series_run_fields_host/_dev): the parametric
series is one producer of the fields A, B, C, Q, F and the rim of psi, and feeding those fields back gives the same bits;
fields the parameters cannot express are checked against the oracle restatement with exact sparse-LU solutions."""
import ctypes as C

import numpy as np
import pytest

from tests.util import rel_l2

pytestmark = pytest.mark.gpu

LR, LZ = (0.0, 1.0e6), (0.0, 1.5e4)
FIRSTS = (0, 341, 700, 1023)      # spread over the 1,024-long series; the late snapshots are strongly non-symmetric
OUT_FIELDS = ("psi", "f", "theta", "u", "w", "m2")


def _prm(cs, max_iter=200000):
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=max_iter, check_step=cs, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=20)


def _spread_params(firsts=FIRSTS):
    from xlab_ee_fortran_b200 import workloads as W
    return np.concatenate([W.series_params(1, total=1024, first=q) for q in firsts])


def _read_back(ts):
    """A, B, C, Q, F and the rim of psi of the last run, as run_fields takes them."""
    A, B, Cf, Q, F, psi = (ts.field(q) for q in ("A", "B", "C", "Q", "F", "psi"))
    bc = np.zeros_like(psi)
    bc[:, [0, -1], :] = psi[:, [0, -1], :]
    bc[:, :, [0, -1]] = psi[:, :, [0, -1]]
    return A, B, Cf, Q, F, bc


def _outputs(ts, tab):
    return dict(table=tab, **{q: ts.field(q) for q in OUT_FIELDS})


def _assert_same_bits(a, b):
    for q in a:
        assert np.array_equal(a[q], b[q]), q


# ------------------------------------------------------------------ 1. round trip through the fields, bit for bit
ROUND_TRIP = [   # method, dtype, nr, nz, arith, check_step, r1_rel
    ("line2_chebyshev", "f64", 512, 256, "fast", 10, 1e-12),
    ("line2_bicgstab", "f64", 256, 128, "fast", 5, 1e-12),
    ("line2_mixed", "f64", 256, 128, "fast", 10, 1e-12),
    ("line_chebyshev", "f32", 256, 128, "fast", 25, 1e-5),
    ("chebyshev", "f64", 128, 64, "fast", 100, 1e-11),
    ("jacobi", "f64", 48, 36, "strict", 100, 1e-10),
]


@pytest.mark.parametrize("method,dtype,nr,nz,arith,cs,r1_rel", ROUND_TRIP, ids=[c[0] + "-" + c[1] for c in ROUND_TRIP])
def test_parametric_fields_round_trip(method, dtype, nr, nz, arith, cs, r1_rel):
    from xlab_ee_fortran_b200.time_series import TimeSeries
    params = _spread_params()
    prm = _prm(cs, max_iter=2000000 if method == "jacobi" else 200000)
    ts = TimeSeries(nr, nz, LR, LZ, len(params), dtype, arith=arith, method=method, r1_rel=r1_rel)
    tab = ts.run(params, prm)
    ref = _outputs(ts, tab)
    A, B, Cf, Q, F, bc = _read_back(ts)
    ts.close()
    ts = TimeSeries(nr, nz, LR, LZ, len(params), dtype, arith=arith, method=method, r1_rel=r1_rel)
    got = _outputs(ts, ts.run_fields(A, B, Cf, Q, prm, F=F, psi_bc=bc))
    assert np.array_equal(ts.field("Q"), Q) and np.array_equal(ts.field("F"), F)
    ts.close()
    print(f"{method} {dtype}: sweeps {tab[:, 0].tolist()}, err {tab[:, 2].tolist()}")
    if dtype == "f64":
        assert np.all((tab[:, 2] == 0) | (tab[:, 2] == 4)), tab[:, :3]
    _assert_same_bits(got, ref)


def test_round_trip_of_a_long_series_and_probe_policy(monkeypatch):
    """40 smooth snapshots: the parametric run with every operator probed equals the field run, which always probes every
    operator, also when it follows a parametric run with subsampled probes on the same object."""
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz, ns = 128, 64, 40
    params = W.series_params(ns, total=1024, first=100)
    prm = _prm(10)
    kw = dict(dtype="f64", arith="fast", method="line2_chebyshev", r1_rel=1e-11)
    monkeypatch.setenv("XEE_RHO_SUBSAMPLE", "0")
    ts = TimeSeries(nr, nz, LR, LZ, ns, **kw)
    ref = _outputs(ts, ts.run(params, prm))
    fields = _read_back(ts)
    monkeypatch.delenv("XEE_RHO_SUBSAMPLE")
    same_object = _outputs(ts, ts.run_fields(*fields[:4], prm, F=fields[4], psi_bc=fields[5]))
    ts.close()
    _assert_same_bits(same_object, ref)
    ts = TimeSeries(nr, nz, LR, LZ, ns, **kw)
    sub = ts.run(params, prm)                       # smooth and >= 32 snapshots: subsampled probes
    assert np.all(sub[:, 2] == 0)
    after = _outputs(ts, ts.run_fields(*fields[:4], prm, F=fields[4], psi_bc=fields[5]))
    ts.close()
    _assert_same_bits(after, ref)


# ------------------------------------------------------------------ 2. exact, on inputs the parameters cannot express
def _smooth(rng, nz, nr, modes=6):
    """A seeded smooth field on [0,1]^2 with max |.| = 1."""
    y, x = np.meshgrid(np.linspace(0.0, 1.0, nz), np.linspace(0.0, 1.0, nr), indexing="ij")
    s = np.zeros((nz, nr))
    for _ in range(modes):
        kx, ky = rng.integers(1, 5, 2); px, py = rng.random(2) * 2 * np.pi
        s += rng.standard_normal() * np.sin(np.pi * kx * x + px) * np.sin(np.pi * ky * y + py)
    return s / np.abs(s).max()


def _general_fields(ns, nr, nz, seed=7):
    """Vortex A, B, C (thermal-wind consistent) with smooth perturbations, Q = two blobs of opposite sign + a smooth field,
    a non-zero F and non-zero rim values on all four sides."""
    from xlab_ee_fortran_b200 import workloads as W
    rng = np.random.default_rng(seed)
    r = np.linspace(*LR, nr); z = np.linspace(*LZ, nz)
    rm = 0.5 * (r[:-1] + r[1:]); zm = 0.5 * (z[:-1] + z[1:])
    R, Z = np.meshgrid(rm, zm)
    q0 = 3.5 * 287.0 * 10.0 / 86400.0
    A, B, Cf, Q, F, bc = [], [], [], [], [], []
    for n in range(ns):
        a, b, c = (x.astype(np.float64) for x in W.vortex_fields(nr, nz, LR, LZ, f_arr=(1.0e-3 * (0.6 + 0.3 * n), 5e-5),
                                                                  radius_arr=(5.0e4 * (1.4 - 0.2 * n),), thermal_wind_consistent=True))
        a = a * (1.0 + 0.2 * _smooth(rng, nz, nr)); c = c * (1.0 + 0.2 * _smooth(rng, nz, nr))
        b = b * (1.0 + 0.2 * _smooth(rng, nz, nr))
        lim = np.sqrt(0.9 * a * c)
        b = np.clip(b, -lim, lim)
        assert np.all(a * c - b * b > 0)
        blob = lambda rc, zc, sr, sz: np.exp(-((R - rc) / sr) ** 2 - ((Z - zc) / sz) ** 2)
        q = q0 * (blob(4e4 + 1e4 * n, 5e3, 1e4, 2e3) - 0.6 * blob(1.5e5, 9e3, 3e4, 3e3) + 0.1 * _smooth(rng, nz - 1, nr - 1) * np.exp(-R / 2e5))
        f = 2e-4 * _smooth(rng, nz - 1, nr - 1) * np.exp(-Z / 8e3)
        p = np.zeros((nz, nr))
        p[0] = 5e7 * _smooth(rng, 1, nr)[0]; p[-1] = 1e7 * _smooth(rng, 1, nr)[0]
        p[:, 0] = 2e7 * _smooth(rng, nz, 1)[:, 0]; p[:, -1] = 3e7 * _smooth(rng, nz, 1)[:, 0]
        A.append(a); B.append(b); Cf.append(c); Q.append(q); F.append(f); bc.append(p)
    return [np.array(x) for x in (A, B, Cf, Q, F, bc)]


def test_general_fields_against_exact_solution():
    from oracle import oracle as O
    from tests.series_fields_oracle import series_fields_rows
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz, ns = 256, 128, 4
    A, B, Cf, Q, F, bc = _general_fields(ns, nr, nz)
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", arith="fast", method="line2_chebyshev", r1_rel=1e-12)
    tab = ts.run_fields(A, B, Cf, Q, _prm(10), F=F, psi_bc=bc)
    dev = {q: ts.field(q) for q in OUT_FIELDS}
    ts.close()
    ref = series_fields_rows(A, B, Cf, Q, F, bc, LR, LZ)
    print("sweeps", tab[:, 0].tolist(), "sum_Q", tab[:, 3].tolist(), "efficiency", tab[:, 5].tolist())
    assert np.all(tab[:, 2] == 0), tab[:, :3]
    for n in range(ns):
        assert rel_l2(dev["f"][n], ref["f"][n]) < 1e-12, n
        assert np.array_equal(dev["theta"][n], ref["theta"][n]), n
        u, w = O.cal_uw(dev["psi"][n], O.Domain(LR, LZ, nr, nz, 0, 0))
        assert np.array_equal(dev["u"][n], u) and np.array_equal(dev["w"][n], w), n
        assert rel_l2(dev["psi"][n], ref["psi"][n]) < 1e-8, (n, rel_l2(dev["psi"][n], ref["psi"][n]))
        assert np.array_equal(dev["psi"][n][[0, -1], :], bc[n][[0, -1], :]) and np.array_equal(dev["psi"][n][:, [0, -1]], bc[n][:, [0, -1]])
    sum_q, ke, eff = ref["table"][:, 0], ref["table"][:, 1], ref["table"][:, 2]
    assert np.all(np.abs(tab[:, 3] - sum_q) <= 1e-12 * np.abs(sum_q)), (tab[:, 3], sum_q)
    assert np.all(np.abs(tab[:, 4] - ke) <= 1e-6 * ref["abs_wtheta"]), (tab[:, 4], ke)
    assert np.all(np.abs(tab[:, 5] - eff) <= 1e-6 * np.abs(eff)), (tab[:, 5], eff)


# ------------------------------------------------------------------ 3. equivalences, bit for bit
def test_equivalent_inputs_give_the_same_bits():
    import torch
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz, ns = 128, 64, 3
    A, B, Cf, Q, F, bc = _general_fields(ns, nr, nz, seed=3)
    prm = _prm(10)
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", arith="fast", method="line2_chebyshev", r1_rel=1e-11)
    run = lambda **kw: _outputs(ts, ts.run_fields(A, B, Cf, Q, prm, **kw))
    no_f = run(F=None, psi_bc=bc)
    with pytest.raises(RuntimeError, match="no momentum forcing"):
        ts.field("F")
    _assert_same_bits(run(F=np.zeros_like(F), psi_bc=bc), no_f)
    assert np.array_equal(ts.field("F"), np.zeros_like(F))
    _assert_same_bits(run(F=F, psi_bc=np.zeros_like(bc)), run(F=F, psi_bc=None))
    noisy = bc + np.pad(np.random.default_rng(1).standard_normal((ns, nz - 2, nr - 2)), ((0, 0), (1, 1), (1, 1)))
    host = run(F=F, psi_bc=bc)
    _assert_same_bits(run(F=F, psi_bc=noisy), host)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    dev = _outputs(ts, ts.run_fields(t(A), t(B), t(Cf), t(Q), prm, F=t(F), psi_bc=t(noisy)))
    _assert_same_bits(dev, host)
    c = torch.from_numpy                                     # CPU tensors take the host entry
    _assert_same_bits(_outputs(ts, ts.run_fields(c(A), c(B), c(Cf), c(Q), prm, F=c(F), psi_bc=c(noisy))), host)
    with pytest.raises(TypeError, match="CUDA tensor"):      # host and device inputs mixed
        ts.run_fields(t(A), B, Cf, Q, prm)
    ts.close()


# ------------------------------------------------------------------ 4. sharding
def test_fields_sharded_equals_unsharded():
    import xlab_ee_fortran_b200 as X
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.time_series import TimeSeries, run_fields_sharded
    nr, nz, total = 64, 48, 7
    Lr, Lz = (0.0, 6.0e5), (0.0, 1.5e4)
    prm = X.SolveParams(max_iter=400000, check_step=25, converge_time=2, r1=1.0, r2=0.0, stall_checks=20)
    kw = dict(dtype="f64", arith="fast", method="line_chebyshev", r1_rel=1e-10)
    ts = TimeSeries(nr, nz, Lr, Lz, total, **kw)
    ts.run(W.series_params(total), prm)
    A, B, Cf, Q, F, bc = _read_back(ts)
    whole = ts.run_fields(A, B, Cf, Q, prm, F=F, psi_bc=bc)
    ts.close()
    parts = []
    for rank in range(3):
        a, b, tab = run_fields_sharded(nr, nz, Lr, Lz, A, B, Cf, Q, prm, F=F, psi_bc=bc, world=3, rank=rank, **kw)
        assert tab.shape == (b - a, 8)
        parts.append(tab)
    got = np.concatenate(parts)
    assert np.all(got[:, 2] == 0) and np.array_equal(got[:, 0], whole[:, 0])
    assert np.allclose(got[:, 3:], whole[:, 3:], rtol=1e-9, atol=0)


# ------------------------------------------------------------------ 5. loud failures and device memory
def test_loud_failures():
    from xlab_ee_fortran_b200 import _lib
    from xlab_ee_fortran_b200.efficiency_map import _prm as cprm
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz, ns = 32, 24, 2
    A, B, Cf, Q, F, bc = _general_fields(ns, nr, nz, seed=5)
    prm = _prm(10)
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", method="line2_chebyshev", r1_rel=1e-10)
    for bad in (dict(A=A[:, :-1]), dict(Q=np.zeros((ns, nz, nr))), dict(F=F[:1]), dict(psi_bc=bc[:, :, :-1])):
        args = {**dict(A=A, B=B, Cf=Cf, Q=Q, F=F, psi_bc=bc), **bad}
        with pytest.raises(ValueError, match="shape"):
            ts.run_fields(args["A"], args["B"], args["Cf"], args["Q"], prm, F=args["F"], psi_bc=args["psi_bc"])
    q = cprm(prm)
    table = np.zeros((ns, 8))
    p = lambda x: np.ascontiguousarray(x).ctypes.data_as(C.c_void_p)
    rc = _lib.lib().xee_series_run_fields_host(ts._h, p(A), p(B), p(Cf), None, p(F), p(bc), C.byref(q), p(table))
    assert rc != 0 and "NULL" in _lib.lib().xee_last_error().decode()
    rc = _lib.lib().xee_series_run_fields_dev(ts._h, p(A), p(B), p(Cf), p(Q), p(F), p(bc), C.byref(q), p(table), None)
    assert rc != 0 and "series' device" in _lib.lib().xee_last_error().decode()     # host memory through the device entry
    ts.run_fields(A, B, Cf, Q, prm)
    with pytest.raises(RuntimeError, match="no momentum forcing"):
        ts.field("F")
    ts.close()


def test_pool_returns_to_baseline_for_both_producers():
    from xlab_ee_fortran_b200.plan import pool_stats
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz, ns = 64, 40, 3
    A, B, Cf, Q, F, bc = _general_fields(ns, nr, nz, seed=9)
    prm = _prm(10, max_iter=400)
    base = pool_stats()[0]
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", method="line2_chebyshev", r1_rel=1e-10)
    ts.run(_spread_params(FIRSTS[:ns]), prm)
    ts.close(); del ts
    assert pool_stats()[0] == base
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", method="line2_chebyshev", r1_rel=1e-10)
    ts.run_fields(A, B, Cf, Q, prm, F=F, psi_bc=bc)
    ts.run_fields(A, B, Cf, Q, prm)
    ts.close(); del ts
    assert pool_stats()[0] == base


def test_device_entry_refuses_another_device():
    import torch
    from xlab_ee_fortran_b200.time_series import TimeSeries
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    nr, nz, ns = 32, 24, 1
    A, B, Cf, Q, F, bc = _general_fields(ns, nr, nz, seed=5)
    ts = TimeSeries(nr, nz, LR, LZ, ns, "f64", method="line2_chebyshev", r1_rel=1e-10, device=0)
    t = lambda x: torch.from_numpy(x).to("cuda:1")
    with pytest.raises(RuntimeError, match="series' device"):
        ts.run_fields(t(A), t(B), t(Cf), t(Q), _prm(10))
    ts.close()
