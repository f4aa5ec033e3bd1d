"""The legacy efficiency decomposition of the time series (TimeSeries.decompose, xee_series_decompose_host/_dev): every
snapshot's efficiency.txt terms from batched solves, against the exact restatement (tests/decompose_oracle.py), against
run_fields bit for bit where the chains coincide, and against the re-hosted legacy driver."""
import ctypes as C
import math
import subprocess

import numpy as np
import pytest

from tests.decompose_oracle import COLS, SOLVES, decompose_rows
from tests.util import rel_l2

pytestmark = pytest.mark.gpu

LR, LZ = (0.0, 1.0e6), (0.0, 1.5e4)
FIRSTS = (0, 341, 700, 1023)      # spread over the 1,024-long series; the late snapshots are strongly non-symmetric
DT = 3600.0
METHODS = (("line2_chebyshev", 10), ("line_chebyshev", 25), ("line2_bicgstab", 5))


def _prm(cs, max_iter=200000):
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=max_iter, check_step=cs, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=20)


def _snapshots(nr, nz, firsts=FIRSTS, Lr=LR, Lz=LZ):
    """A, B, C (float32 values, as files), Q, F, the pumping rim of psi and a chi rim on the top and outer boundaries of
    workloads.series_params snapshots, all float64 [n, ...]."""
    from oracle import oracle as O
    from tests.map_oracle import heat_field
    from xlab_ee_fortran_b200 import workloads as W
    params = np.concatenate([W.series_params(1, total=1024, first=q) for q in firsts])
    g = O.geometry(O.Domain(Lr, Lz, nr, nz, 0, 0), np.float64)
    r = np.linspace(*Lr, nr); z = np.linspace(*Lz, nz)
    out = {q: [] for q in ("A", "B", "C", "Q", "F", "psi_bc", "chi_bc")}
    for n, row in enumerate(params):
        a, b, c, bottom, f = W.series_fields_host(row, nr, nz, Lr, Lz)
        p = np.zeros((nz, nr)); p[0] = bottom
        x = np.zeros((nz, nr))
        x[-1] = 2.0e11 * (1 + 0.2 * n) * np.sin(np.pi * r / Lr[1]) * (r / Lr[1]) ** 2
        x[:, -1] = 5.0e10 * np.sin(np.pi * z / Lz[1])
        for q, v in zip(out, (a, b, c, heat_field(row[14:19], g, np.float64), f, p, x)):
            out[q].append(np.asarray(v, np.float64))
    return {q: np.array(v) for q, v in out.items()}


def _decompose(ts, s, p_psi, p_chi, tendency=True, bc=True, baro="all", **kw):
    return ts.decompose(s["A"], s["B"], s["C"], s["Q"], p_psi, p_chi, F=s["F"], psi_bc=s["psi_bc"],
                        chi_bc=s["chi_bc"] if bc else None, testing_dt=DT if tendency else None, baro=baro, **kw)


_BARO_KEEP = {0: np.r_[0:10], 1: np.r_[0:3, 10:17], 2: np.r_[0:17]}
_BARO_SOLVES = {0: [0, 1, 3, 5, 7], 1: [0, 2, 4, 6, 8], 2: list(range(9))}


# ------------------------------------------------------------------ 1. against the exact oracle
@pytest.mark.parametrize("nr,nz", [(128, 64), (256, 128)])
@pytest.mark.parametrize("tendency", [True, False], ids=["tendency", "instant"])
@pytest.mark.parametrize("bc", [True, False], ids=["chi_bc", "no_chi_bc"])
def test_against_exact_oracle(nr, nz, tendency, bc):
    from xlab_ee_fortran_b200.time_series import TimeSeries
    s = _snapshots(nr, nz)
    ref, ref_fields = decompose_rows(s["A"], s["B"], s["C"], s["Q"], s["F"], s["psi_bc"], s["chi_bc"] if bc else None, LR, LZ,
                                     testing_dt=DT if tendency else None, baro=2)
    for method, cs in METHODS:
        ts = TimeSeries(nr, nz, LR, LZ, len(FIRSTS), "f64", method=method, r1_rel=1e-12)
        for baro in (0, 1, 2):
            tab, it, err = _decompose(ts, s, _prm(cs), _prm(cs), tendency, bc, baro)
            print(method, baro, "sweeps", it.tolist(), "err", err.tolist())
            assert np.all((err == 0) | (err == 4)), (method, baro, err)
            ran = _BARO_SOLVES[baro] if tendency else _BARO_SOLVES[baro][1:]
            if not bc:
                ran = [k for k in ran if k not in (1, 2)]
            assert np.all(it[:, ran] >= 0) and np.all(np.delete(it, ran, axis=1) == -1), (method, baro, it)
            want = np.full_like(ref, np.nan)
            want[:, _BARO_KEEP[baro]] = ref[:, _BARO_KEEP[baro]]
            assert np.array_equal(np.isnan(tab), np.isnan(want)), (method, baro)
            fin = ~np.isnan(want)
            assert np.all(np.abs(tab[fin] - want[fin]) <= 1e-6 * np.abs(want[fin])), \
                (method, baro, [(COLS[j], tab[n, j], want[n, j]) for n, j in zip(*np.nonzero(fin & ~(np.abs(tab - want) <= 1e-6 * np.abs(want))))])
            for k in ran:
                got = ts.decomp_field(SOLVES[k])
                for n in range(len(FIRSTS)):
                    e = rel_l2(got[n], ref_fields[n][SOLVES[k]]) if np.any(ref_fields[n][SOLVES[k]]) else np.abs(got[n]).max()
                    assert e < 1e-8, (method, baro, SOLVES[k], n, e)
            if tendency:
                for name in ("dtheta_dt", "theta_after"):
                    got = ts.decomp_field(name)
                    for n in range(len(FIRSTS)):
                        assert rel_l2(got[n], ref_fields[n][name]) < 1e-8, (method, name, n)
        ts.close()


def test_f32_line_chebyshev_against_exact_oracle():
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz = 128, 64
    s = _snapshots(nr, nz)
    ref, _ = decompose_rows(s["A"], s["B"], s["C"], s["Q"], s["F"], s["psi_bc"], s["chi_bc"], LR, LZ, testing_dt=DT, baro=2)
    ts = TimeSeries(nr, nz, LR, LZ, len(FIRSTS), "f32", method="line_chebyshev", r1_rel=1e-5)
    tab, it, err = _decompose(ts, s, _prm(25), _prm(25))
    ts.close()
    print("f32 sweeps", it.tolist(), "err", err.tolist())
    assert np.all(it >= 0) and np.all((err == 0) | (err == 4))
    scale = np.abs(ref[:, 3:]).max(axis=1, keepdims=True)        # fp32 sums of cancelling terms: error relative to the row
    assert np.all(np.abs(tab[:, 3:] - ref[:, 3:]) <= 5e-3 * np.abs(ref[:, 3:]) + 1e-4 * scale), (tab, ref)
    assert np.allclose(tab[:, :3], ref[:, :3], rtol=5e-3, atol=0)


# ------------------------------------------------------------------ 2. bit for bit
def test_stage_one_and_instant_baroclinic_check_equal_run_fields():
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz = 128, 64
    s = _snapshots(nr, nz)
    prm = _prm(10)
    ts = TimeSeries(nr, nz, LR, LZ, len(FIRSTS), "f64", method="line2_chebyshev", r1_rel=1e-12)
    rf = ts.run_fields(s["A"], s["B"], s["C"], s["Q"], prm, F=s["F"], psi_bc=s["psi_bc"])
    psi = ts.field("psi")
    tab, it, _ = _decompose(ts, s, prm, prm, tendency=True, bc=True)
    assert np.array_equal(ts.decomp_field("psi_before"), psi) and np.array_equal(it[:, 0], rf[:, 0])
    assert np.array_equal(tab[:, 0], rf[:, 3])
    tab, it, _ = _decompose(ts, s, prm, prm, tendency=False, bc=False, baro="baroclinic")
    assert np.array_equal(ts.decomp_field("psi_after_B0dB"), psi) and np.array_equal(it[:, 8], rf[:, 0])
    assert np.array_equal(tab[:, 16], rf[:, 4]) and np.array_equal(tab[:, 0], rf[:, 3])
    with pytest.raises(RuntimeError, match="did not make"):
        ts.decomp_field("psi_before")
    ts.close()


def test_host_device_and_tensor_inputs_give_the_same_bits():
    import torch
    from xlab_ee_fortran_b200 import _lib
    from xlab_ee_fortran_b200.efficiency_map import _prm as cprm
    from xlab_ee_fortran_b200.time_series import TimeSeries, _DecompDesc
    nr, nz = 128, 64
    s = _snapshots(nr, nz, FIRSTS[:3])
    prm = _prm(10)
    ts = TimeSeries(nr, nz, LR, LZ, 3, "f64", method="line2_chebyshev", r1_rel=1e-11)
    host = _decompose(ts, s, prm, prm)
    fields = [ts.decomp_field(q) for q in ("dtheta_dt", "theta_after") + SOLVES]
    t = {q: torch.from_numpy(np.ascontiguousarray(v)).cuda() for q, v in s.items()}
    dev = _decompose(ts, t, prm, prm)
    for a, b in zip(host, dev):
        assert np.array_equal(a, b, equal_nan=True)
    for q, f in zip(("dtheta_dt", "theta_after") + SOLVES, fields):
        assert np.array_equal(ts.decomp_field(q), f), q
    # the raw C entries, iters/err NULL
    desc = _DecompDesc(1, DT, 2)
    tab = np.zeros((3, len(COLS)))
    qp = cprm(prm)
    p = lambda x: C.c_void_p(x.data_ptr())
    rc = _lib.lib().xee_series_decompose_dev(ts._h, C.byref(desc), p(t["A"]), p(t["B"]), p(t["C"]), p(t["Q"]), p(t["F"]),
                                             p(t["psi_bc"]), p(t["chi_bc"]), C.byref(qp), C.byref(qp),
                                             tab.ctypes.data_as(C.c_void_p), None, None, None)
    assert rc == 0 and np.array_equal(tab, host[0], equal_nan=True)
    ts.close()


def test_sharded_equals_single_run():
    from xlab_ee_fortran_b200.time_series import TimeSeries, decompose_sharded
    nr, nz = 64, 48
    s = _snapshots(nr, nz)
    prm = _prm(25, max_iter=400000)
    kw = dict(dtype="f64", method="line_chebyshev", r1_rel=1e-10)
    ts = TimeSeries(nr, nz, LR, LZ, len(FIRSTS), **kw)
    whole = _decompose(ts, s, prm, prm)
    ts.close()
    parts = []
    for rank in range(2):
        a, b, tab, it, err = decompose_sharded(nr, nz, LR, LZ, s["A"], s["B"], s["C"], s["Q"], prm, prm, F=s["F"],
                                               psi_bc=s["psi_bc"], chi_bc=s["chi_bc"], testing_dt=DT, world=2, rank=rank, **kw)
        assert tab.shape == (b - a, len(COLS))
        parts.append((tab, it, err))
    for q in range(3):
        assert np.array_equal(np.concatenate([x[q] for x in parts]), whole[q], equal_nan=True)


# ------------------------------------------------------------------ 3. against the re-hosted legacy driver
_LABELS = {   # efficiency.txt label -> table column
    "sum Q": 0, "sum dtheta_dt": 1, "Local heat response (sum Q / sum dtheta_dt)": 2,
    "eta [L(B=0)    = 0]      w/  boundary": 3, "eta [L(B=0)    = dB]     wo/ boundary": 4,
    "eta [L(B=0)    = B0]     wo/ boundary": 5, "bndconv [L(B=0) = B0dB]   w/ boundary": 6,
    "bndconv2 [L(B=0) = B0dB]   w/ boundary": 7, "etaQ [L(B=0)    = J F] w/  boundary": 8,
    "wtheta [L(B=0)    = J F] w/  boundary": 9,
    "eta [L(B=B0dB) = 0]      w/  boundary": 10, "eta [L(B=B0dB) = dB]     wo/ boundary": 11,
    "eta [L(B=B0dB) = B0]     wo/ boundary": 12, "bndconv [L(B=B0dB) = B0dB]w/ boundary": 13,
    "bndconv2 [L(B=B0dB) = B0dB]w/ boundary": 14, "etaQ [L(B=B0dB) = J F] w/  boundary": 15,
    "wtheta [L(B=B0dB) = J F] w/  boundary": 16,
}


def test_against_the_rehosted_legacy_driver(tmp_path):
    from xlab_ee_fortran_b200 import _lib
    from xlab_ee_fortran_b200.time_series import TimeSeries
    exe = _lib.build_old_diagnose()
    nr, nz = 40, 28
    Lr, Lz = (0.0, 5.0e5), (0.0, 1.4e4)
    s = _snapshots(nr, nz, (500,), Lr, Lz)
    s32 = {q: v.astype(np.float32) for q, v in s.items()}       # what the driver reads from its .bin files
    for q in ("A", "B", "C", "Q", "F", "psi_bc", "chi_bc"):
        s32[q][0].tofile(tmp_path / f"{q}.bin")
    cfg = ("CYLINDRICAL-TENDENCY-DENSITY_NORMAL-BARO_ALL // mode\n"
           f"{DT} // testing dt\n{Lr[0]} {Lr[1]} {Lz[0]} {Lz[1]} // domain\n{nr} {nz} // grid\n. // in\n. // out\n"
           "A.bin // A\nB.bin // B\nC.bin // C\nQ.bin // Q\nF.bin // F\n"
           "1 1e-21 4000000 1.0 // rpsi: strategy residue max_iter alpha\n"
           "1 1e-18 4000000 1.0 // rchi\nyes // rpsi bc\npsi_bc.bin\nyes // rchi bc\nchi_bc.bin\n")
    rr = subprocess.run([exe, "--r8"], input=cfg, capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert rr.returncode == 0, rr.stdout + rr.stderr
    vals = {}
    for line in (tmp_path / "efficiency.txt").read_text().splitlines():
        if ":" in line and not line.startswith(" #"):
            key, rest = line.split(":", 1)
            vals[key.strip()] = [float(x) for x in rest.split(",")]
    assert set(_LABELS) <= set(vals)
    ts = TimeSeries(nr, nz, Lr, Lz, 1, "f64", method="line2_chebyshev", r1_rel=1e-13)
    tab, it, err = _decompose(ts, {q: v.astype(np.float64) for q, v in s32.items()}, _prm(10), _prm(10))
    ts.close()
    assert np.all(err == 0), err
    for label, col in _LABELS.items():
        v = vals[label]
        assert v[0] == pytest.approx(tab[0, col], rel=1e-5), (label, v, tab[0, col])
        if len(v) > 1:
            assert v[1] == pytest.approx(tab[0, col] / tab[0, 0], rel=1e-5), label


# ------------------------------------------------------------------ 4. edge cases and failures
def test_instant_without_chi_bc_skips_the_zero_solves():
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz = 64, 48
    s = _snapshots(nr, nz)
    ts = TimeSeries(nr, nz, LR, LZ, len(FIRSTS), "f64", method="line2_chebyshev", r1_rel=1e-12)
    tab, it, err = _decompose(ts, s, _prm(10), _prm(10), tendency=False, bc=False)
    assert np.all(it[:, [3, 4]] == 0) and np.all(err[:, [3, 4]] == 0)
    assert np.all(it[:, [0, 1, 2]] == -1) and np.all(it[:, 5:] > 0)
    assert np.all(ts.decomp_field("chi_0_dB") == 0) and np.all(ts.decomp_field("chi_B0dB_dB") == 0)
    assert np.all(tab[:, [4, 11]] == 0) and np.all(np.isnan(tab[:, [1, 2, 3, 6, 7, 10, 13, 14]]))
    for name in ("dtheta_dt", "psi_before", "chi_0_0"):
        with pytest.raises(RuntimeError, match="did not make"):
            ts.decomp_field(name)
    ts.close()


def test_refused_inputs():
    from xlab_ee_fortran_b200 import _lib
    from xlab_ee_fortran_b200.efficiency_map import _prm as cprm
    from xlab_ee_fortran_b200.time_series import TimeSeries, _DecompDesc
    nr, nz = 32, 24
    s = _snapshots(nr, nz, FIRSTS[:2])
    prm = _prm(10)
    ts = TimeSeries(nr, nz, LR, LZ, 2, "f64", method="line2_chebyshev", r1_rel=1e-10)
    for baro in (3, -1):
        with pytest.raises(RuntimeError, match="baro"):
            _decompose(ts, s, prm, prm, baro=baro)
    with pytest.raises(ValueError, match="baro"):
        _decompose(ts, s, prm, prm, baro="both")
    for dt in (math.nan, math.inf):
        with pytest.raises(RuntimeError, match="testing_dt"):
            ts.decompose(s["A"], s["B"], s["C"], s["Q"], prm, prm, testing_dt=dt)
    with pytest.raises(ValueError, match="shape"):
        ts.decompose(s["A"], s["B"], s["C"], s["Q"], prm, prm, chi_bc=s["chi_bc"][:, 1:])
    q = cprm(prm)
    desc = _DecompDesc(1, DT, 2)
    tab = np.zeros((2, len(COLS)))
    p = lambda x: np.ascontiguousarray(x).ctypes.data_as(C.c_void_p)
    lib = _lib.lib()
    rc = lib.xee_series_decompose_host(ts._h, C.byref(desc), p(s["A"]), None, p(s["C"]), p(s["Q"]), None, None, None,
                                       C.byref(q), C.byref(q), p(tab), None, None)
    assert rc != 0 and "NULL" in lib.xee_last_error().decode()
    rc = lib.xee_series_decompose_dev(ts._h, C.byref(desc), p(s["A"]), p(s["B"]), p(s["C"]), p(s["Q"]), None, None,
                                      p(s["chi_bc"]), C.byref(q), C.byref(q), p(tab), None, None, None)
    assert rc != 0 and "series' device" in lib.xee_last_error().decode()
    with pytest.raises(RuntimeError, match="did not make"):      # nothing made by the refused calls
        ts.decomp_field("theta_after")
    ts.close()


def test_pool_baseline_and_run_fields_after_decompose():
    from xlab_ee_fortran_b200.plan import pool_stats
    from xlab_ee_fortran_b200.time_series import TimeSeries
    nr, nz = 64, 48
    s = _snapshots(nr, nz, FIRSTS[:3])
    prm = _prm(10)
    kw = dict(dtype="f64", method="line2_chebyshev", r1_rel=1e-11)
    base = pool_stats()[0]
    fresh = TimeSeries(nr, nz, LR, LZ, 3, **kw)
    want = fresh.run_fields(s["A"], s["B"], s["C"], s["Q"], prm, F=s["F"], psi_bc=s["psi_bc"])
    want_psi = fresh.field("psi")
    fresh.close(); del fresh
    ts = TimeSeries(nr, nz, LR, LZ, 3, **kw)
    before = pool_stats()[0]
    _decompose(ts, s, prm, prm)
    assert pool_stats()[0] > before                               # the decomposition's buffers, allocated on first use
    _decompose(ts, s, prm, prm, tendency=False, baro=1)
    got = ts.run_fields(s["A"], s["B"], s["C"], s["Q"], prm, F=s["F"], psi_bc=s["psi_bc"])
    assert np.array_equal(got, want) and np.array_equal(ts.field("psi"), want_psi)
    ts.close(); del ts
    assert pool_stats()[0] == base
