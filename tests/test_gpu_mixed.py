"""GPU tests of the mixed-precision two-level method (XEE_METHOD_LINE2_MIXED, csrc/xee_mixed.cuh).

1. The first two refinement steps against the numpy restatement (tests/mixed_oracle.py).
2. Converged fields against exact sparse-LU solutions: the bench map operator at every 16th benchmark location, and eight
   snapshots across the 1,024-long time series.
3. Stop decisions against the exact replay of the stop rule (tests/stop_rule.py), built like tests/test_gpu_stop_rule.py,
   with max_iter inside a refinement step; every field equals sweeps(iters); batch order changes no bits.
4. The power-of-two scale: a problem scaled by 2^-110 gives the scaled bits of the unscaled one.
5. solve_elliptic with XEE_METHOD=line2_mixed, and loud failures outside the supported configurations.
"""
from unittest import mock

import numpy as np
import pytest

import tests.test_gpu_stop_rule as SR
from oracle import oracle as O
from tests.exact_oracle import ExactSolver, MapCase, efficiency_row, host_residual_rms, rms_interior
from tests.mixed_oracle import Mixed
from tests.stop_rule import replay, same_bits
from tests.test_gpu_twolevel import _aniso
from tests.util import rel_l2

pytestmark = pytest.mark.gpu
METHOD = "line2_mixed"


def _mods():
    import torch
    import xlab_ee_fortran_b200 as X
    return torch, X


def _sweeps(torch, plan, P, F, k, check_step, want_rms=False):
    psi = torch.from_numpy(P).cuda(); ft = torch.from_numpy(F).cuda()
    rms = plan.sweeps(psi, ft, 1.0, k, want_rms=want_rms, check_step=check_step)
    return psi.cpu().numpy(), rms


# ------------------------------------------------------------------ 1. the first two steps against the restatement
@pytest.mark.parametrize("shared", [True, False])
def test_first_two_steps_match_numpy_restatement(shared):
    """Half a step, one step and two steps of 30 fp32 sweeps.  The device and the restatement differ in the rounding of the
    fp32 inner iteration (FMA, the fp32 factors of the rounded operator), so a step's correction s (e + P c) agrees to an
    fp32 tolerance; the second step starts from the device's own first iterate, so the fp64 iterate after it agrees to
    that tolerance times the size of the second correction."""
    torch, X = _mods()
    nx, ny, nb, cs = 128, 66, 3, 30
    coes = []
    for q in range(1 if shared else nb):
        a, b, c = _aniso(nx, ny, seed=21 + q)
        coes.append(O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)[0])
    rng = np.random.default_rng(5)
    F = rng.standard_normal((nb, ny, nx)); P = rng.standard_normal((nb, ny, nx))
    plan = X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=shared, arith="fast", method=METHOD)
    plan.set_coe_aos(coes[0] if shared else np.stack(coes))
    half, _ = _sweeps(torch, plan, P, F, cs // 2, cs)
    one, rms1 = _sweeps(torch, plan, P, F, cs, cs, want_rms=True)
    two, _ = _sweeps(torch, plan, P, F, 2 * cs, cs)
    rho, gamma = plan.cheb_params()
    assert plan.kernel_info()[0] == 5
    plan.close()
    # one operator per solve: cheb_params() reports solve 0's radius, so solve 0 is compared with the restatement and every
    # solve's steps must contract its own residual
    for n in range(nb) if shared else range(1):
        coe = coes[0 if shared else n]
        m = Mixed(coe)
        for k, got in ((cs // 2, half[n]), (cs, one[n])):
            d = m.run(P[n], F[n], rho, gamma, cs, k)["corrections"][0]
            e = rel_l2(got - P[n], d)
            print(f"shared={shared} n={n} {k} sweeps: correction error {e:.2e}")
            assert e < 1e-4, (n, k, e)
        assert abs(rms1[n] - host_residual_rms(one[n], coe, F[n])) <= 1e-9 * rms1[n]
        d2 = m.run(one[n], F[n], rho, gamma, cs, cs)["corrections"][0]
        e2 = np.linalg.norm(two[n] - (one[n] + d2)) / np.linalg.norm(d2)
        print(f"shared={shared} n={n} second step: correction error {e2:.2e}")
        assert e2 < 1e-4, (n, e2)
    for n in range(nb):
        coe = coes[0 if shared else n]
        r0 = host_residual_rms(P[n], coe, F[n])
        assert host_residual_rms(one[n], coe, F[n]) < 0.2 * r0
        assert host_residual_rms(two[n], coe, F[n]) < 0.2 * host_residual_rms(one[n], coe, F[n])


# ------------------------------------------------------------------ 2. converged fields against sparse LU
def _params(cs=100, stall=0):
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=200000, check_step=cs, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=stall)


def test_bench_map_against_exact_solution():
    """The bench map operator (512 x 256, fp64) at every 16th benchmark location, every solve to r1 = 1e-12 rms(f_n)."""
    import bench
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = bench.heat_rows(512)[::16]
    m = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method=METHOD, r1_rel=bench.R1_REL)
    tab = m.run(heat, _params())
    psi, f = m.field("psi"), m.field("f")
    assert m.kernel_info()[0] == 5
    m.close()
    assert np.all(tab[:, 2] == 0), np.unique(tab[:, 2])
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    exact = ExactSolver(case.coe).solve(f)
    fe = np.array([rel_l2(psi[n], exact[n]) for n in range(len(heat))])
    ee = np.array([abs(tab[n, 5] - efficiency_row(exact[n], row, case)["efficiency"]) / abs(tab[n, 5]) for n, row in enumerate(heat)])
    print(f"{METHOD} map: sweeps {int(tab[:, 0].min())}-{int(tab[:, 0].max())}, field error {fe.max():.2e}, "
          f"efficiency error {ee.max():.2e}")
    assert np.all(fe < 1e-8), fe
    assert np.all(ee < 1e-6), ee


def test_series_across_the_whole_series_against_exact_solution():
    """Eight snapshots spread over the 1,024-long series, the late non-symmetric ones included; one operator per solve."""
    import bench
    from tests.exact_oracle import ke_gen
    from tests.map_oracle import background_theta
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.time_series import TimeSeries
    NR, NZ, LR, LZ = bench.NR, bench.NZ, bench.LR, bench.LZ
    firsts = (0, 150, 341, 500, 700, 850, 950, 1023)
    params = np.concatenate([W.series_params(1, total=1024, first=q) for q in firsts])
    ts = TimeSeries(NR, NZ, LR, LZ, len(firsts), "f64", arith="fast", method=METHOD, r1_rel=bench.R1_REL)
    tab = ts.run(params, _params(stall=20))
    A, B, C, psi, f = (ts.field(q) for q in ("A", "B", "C", "psi", "f"))
    ts.close()
    assert np.all((tab[:, 2] == 0) | (tab[:, 2] == 4)), tab[:, :3]
    case = MapCase(A[0], B[0], C[0], LR, LZ)
    for n, q in enumerate(firsts):
        a, b, c = O.build_abc(A[n], B[n], C[n], case.d)
        coe, _ = O.cal_coe(a, b, c, case.g["dr"], case.g["dz"], NR, NZ)
        bc = np.zeros((NZ, NR)); bc[0] = psi[n][0]
        x = ExactSolver(coe).solve(f[n], bc)
        e = rel_l2(psi[n], x)
        ke_x, _ = ke_gen(x, background_theta(A[n], B[n], C[n], case.d, np.float64), case.d, case.k)
        ek = abs(tab[n, 4] - ke_x) / abs(ke_x)
        print(f"{METHOD} snapshot {q}: {int(tab[n, 0])} sweeps, err {int(tab[n, 2])}, field {e:.2e}, ke_gen {ek:.2e}")
        assert e < 1e-8, (q, e)
        assert ek < 1e-6, (q, ek)


# ------------------------------------------------------------------ 3. stop decisions
# method, arith, dtype, kernel, shared operator, nx, ny, nb, check_step, converge_time, lost_rate, r2, stall_checks
ROWS = {
    "mixed-shared": (METHOD, "fast", "f64", 0, True, 128, 72, 6, 12, 2, 1, 0.0, 0),
    "mixed-persolve": (METHOD, "fast", "f64", 0, False, 136, 70, 5, 10, 1, 5, 0.0, 0),
}


def _case(key):
    with mock.patch.dict(SR.ROWS, {key: ROWS[key]}):
        return SR.Case(key)


@pytest.mark.parametrize("key", list(ROWS))
def test_stop_decisions_match_replay(key):
    """max_iter = M check_step + 1 ends inside a refinement step: the solves that reach it apply one fp32 sweep's correction."""
    torch, X = _mods()
    case = _case(key)
    T = case.dt
    eps = float(np.finfo(T).eps)
    plan = case.plan(X)
    seq = SR._sequences(torch, X, case, plan)
    # a. the residual check m measured is that of the iterate after m refinement steps
    for m in sorted({1, 2, SR.M // 2, SR.M}):
        it, _ = _sweeps(torch, plan, case.P, case.F, m * case.cs, case.cs)
        for n in range(case.nb):
            host = host_residual_rms(it[n], case.coe_of(n), case.F[n])
            tol = 16 * eps * SR._magnitude(it[n], case.coe_of(n), case.F[n]) + 4 * eps * seq[n, m - 1]
            assert abs(seq[n, m - 1] - host) <= tol, (key, m, n, seq[n, m - 1], host, tol)
    # b. stop decisions, bit for bit, for sync_every 1, 2, 3; every field equals sweeps(iters[n])
    max_iter = SR.M * case.cs + 1
    stops = set()
    for shift in range(0, 5, case.nb):
        r1 = SR._thresholds(case, seq, shift).astype(T)
        want = [replay(seq[n], T, r1[n], case.r2, case.ct, case.lr, max_iter, case.cs, detect_explode=True,
                       stall_checks=case.stall) for n in range(case.nb)]
        stops |= {w[0] for w in want}
        r1_dev = torch.from_numpy(r1).cuda()
        runs = [SR._solve(torch, plan, case.P, case.F, case.params(X, max_iter=max_iter, r1_per_solve=r1_dev, sync_every=s))
                for s in (1, 2, 3)]
        got, out = runs[0]
        for n in range(case.nb):
            it, err, o1, o2 = want[n]
            assert (out["iters"][n], out["err"][n]) == (it, err), (key, n, out["iters"][n], out["err"][n], it, err)
            assert same_bits(out["r1"][n], o1) and same_bits(out["r2"][n], o2), (key, n)
        for g, o in runs[1:]:
            assert np.array_equal(g, got)
            for k in ("iters", "err", "r1", "r2"):
                assert np.array_equal(o[k], out[k], equal_nan=True), k
        for v in sorted(set(out["iters"].tolist())):
            ref, _ = _sweeps(torch, plan, case.P, case.F, v, case.cs)
            for n in np.nonzero(out["iters"] == v)[0]:
                assert np.array_equal(got[n], ref[n]), (key, n, v)
        # c. the reversed batch gives every solve the same bits (shared operator: the spectral estimate is common)
        if case.shared:
            g2, o2 = SR._solve(torch, plan, case.P[::-1].copy(), case.F[::-1].copy(),
                               case.params(X, max_iter=max_iter, r1_per_solve=torch.from_numpy(r1[::-1].copy()).cuda()))
            assert np.array_equal(g2[::-1], got)
            for k in ("iters", "err", "r1", "r2"):
                assert np.array_equal(o2[k][::-1], out[k], equal_nan=True), k
    assert len(stops) >= 4 and max_iter in stops, sorted(stops)
    if case.r2 == 0:
        assert min(stops) == case.ct * case.cs, sorted(stops)
    plan.close()


# ------------------------------------------------------------------ 4. the power-of-two scale
def test_scaled_problem_gives_scaled_bits():
    """f, the first guess and r1 scaled by 2^-110: the fp64 residual, the scale s and the stop rule scale exactly, and the
    fp32 right-hand side r / s is the same, so every solve returns exactly 2^-110 times the unscaled field with the same
    iters, err and ratio.  Without the scale the fp32 right-hand side would fall below fp32's normal range within a step
    (the residual reaches ~1e-41 after the first one)."""
    torch, X = _mods()
    nx, ny, nb = 128, 72, 3
    a, b, c = _aniso(nx, ny, seed=4)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    rng = np.random.default_rng(8)
    F = rng.standard_normal((nb, ny, nx)); P = rng.standard_normal((nb, ny, nx))
    plan = X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method=METHOD)
    plan.set_coe_aos(coe)
    sc = 2.0 ** -110
    prm = lambda r1: X.SolveParams(max_iter=2000, check_step=40, converge_time=2, r1=r1, r2=0.0)
    r1 = 1e-12 * rms_interior(F[0])
    g1, o1 = SR._solve(torch, plan, P, F, prm(r1))
    g2, o2 = SR._solve(torch, plan, P * sc, F * sc, prm(r1 * sc))
    plan.close()
    assert np.all(o1["err"] == 0), o1
    assert np.array_equal(g2, g1 * sc)
    assert np.array_equal(o2["iters"], o1["iters"]) and np.array_equal(o2["err"], o1["err"])
    assert np.array_equal(o2["r1"], o1["r1"] * sc) and np.array_equal(o2["r2"], o1["r2"])


# ------------------------------------------------------------------ 5. the Fortran-facing entry, loud failures
def test_solve_elliptic_with_xee_method(monkeypatch):
    """solve_elliptic with XEE_METHOD=line2_mixed XEE_ARITH=fast on reference case test1 (200 x 200, fp64)."""
    import xlab_ee_fortran_b200 as X
    from tests.util import ref_test1_inputs
    A, B, C, bc = ref_test1_inputs()
    d = O.Domain((0.0, 1.0), (0.0, 1.0), 200, 200, 0, 0)
    a, b, c = O.build_abc(A.astype(np.float64), B.astype(np.float64), C.astype(np.float64), d)
    g = O.geometry(d, np.float64)
    coe, _ = O.cal_coe(a, b, c, g["dr"], g["dz"], 200, 200)
    f = -B.astype(np.float64)
    r1 = 1e-11 * rms_interior(f)
    monkeypatch.setenv("XEE_METHOD", METHOD); monkeypatch.setenv("XEE_ARITH", "fast")
    dat = bc.astype(np.float64).copy(); wk = np.zeros_like(dat)
    it, r1o, r2o, err = X.solve_elliptic(200000, 100, 2, 5, r1, 0.0, 1.0, dat, coe, f, wk, 200, 200)
    assert err == 0 and r1o < r1, (it, r1o, err)
    assert np.array_equal(wk, dat)
    x = ExactSolver(coe).solve(f, bc.astype(np.float64))
    print(f"{METHOD} solve_elliptic: {it} sweeps, field error {rel_l2(dat, x):.2e}")
    assert rel_l2(dat, x) < 1e-8


@pytest.mark.parametrize("kw,msg", [
    (dict(dtype="f32"), "fp64 answers"),
    (dict(arith="strict"), "FAST"),
    (dict(kernel=1), "kernel 5"),
    (dict(nx=16, ny=16), "coarse node"),
    (dict(nx=130), "nx % 4"),
])
def test_unsupported_configurations_fail_loudly(kw, msg):
    _, X = _mods()
    base = dict(nx=128, ny=66, nbatch=2, dtype="f64", shared_coe=True, arith="fast", method=METHOD)
    base.update(kw)
    nx, ny = base.pop("nx"), base.pop("ny")
    with pytest.raises(RuntimeError, match=msg):
        X.Plan(nx, ny, **base)
