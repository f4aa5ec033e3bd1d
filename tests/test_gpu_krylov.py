"""GPU tests of the BiCGStab methods (XEE_METHOD_LINE_BICGSTAB, XEE_METHOD_LINE2_BICGSTAB, csrc/xee_krylov.cuh).

1. The first iterations against the numpy restatement (tests/krylov_oracle.py), fp64, small grids.
2. Converged fields against exact sparse-LU solutions: the bench map operator at a sample of the benchmark locations, and
   snapshots across the whole 1,024-long time series.
3. Stop decisions against the exact replay of the stop rule (tests/stop_rule.py), built like tests/test_gpu_stop_rule.py.
4. The efficiency map, the time series and the Fortran-facing solve_elliptic with the new methods.
5. Loud failures outside the supported configurations.
"""
from unittest import mock

import numpy as np
import pytest

import tests.test_gpu_stop_rule as SR
from oracle import oracle as O
from tests.exact_oracle import ExactSolver, MapCase, efficiency_row, host_residual_rms, rms_interior
from tests.krylov_oracle import Krylov
from tests.stop_rule import replay, same_bits
from tests.test_gpu_twolevel import _aniso
from tests.util import rel_l2

pytestmark = pytest.mark.gpu
METHODS = ("line_bicgstab", "line2_bicgstab")


def _mods():
    import torch
    import xlab_ee_fortran_b200 as X
    return torch, X


def _sweeps(torch, plan, P, F, k, check_step, want_rms=False):
    psi = torch.from_numpy(P).cuda(); ft = torch.from_numpy(F).cuda()
    rms = plan.sweeps(psi, ft, 1.0, k, want_rms=want_rms, check_step=check_step)
    return psi.cpu().numpy(), rms


# ------------------------------------------------------------------ 1. first iterations against the numpy restatement
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("shared", [True, False])
def test_first_iterations_match_numpy_restatement(method, shared):
    """Four iterations with a residual replacement after the second, fp64.  The device and the restatement differ only by
    rounding: FMA chains and the order of the tile sums in the dot products, a few ulp per operation.  Four iterations
    multiply such perturbations by at most the condition number of K^-1 L on this grid (~1e2 for the block-line and ~10
    for the two-level preconditioner, tests/twolevel_oracle.py) per iteration pair, far below the 1e-9 bound."""
    torch, X = _mods()
    nx, ny, nb = 128, 66, 3
    coes = []
    for q in range(1 if shared else nb):
        a, b, c = _aniso(nx, ny, seed=21 + q)
        coes.append(O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)[0])
    rng = np.random.default_rng(5)
    F = rng.standard_normal((nb, ny, nx)); P = rng.standard_normal((nb, ny, nx))
    plan = X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=shared, arith="fast", method=method)
    plan.set_coe_aos(coes[0] if shared else np.stack(coes))
    got, rms = _sweeps(torch, plan, P, F, 4, 2, want_rms=True)
    assert plan.kernel_info()[0] == 5 and plan.cheb_params() == (0.0, 1.0)
    plan.close()
    for n in range(nb):
        kr = Krylov(coes[0 if shared else n], method == "line2_bicgstab")
        ref = kr.run(P[n], F[n], 4, 2)["x"]
        e = rel_l2(got[n], ref)
        assert e < 1e-9, (n, e)
        host = host_residual_rms(got[n], coes[0 if shared else n], F[n])
        assert abs(rms[n] - host) <= 1e-9 * host, (n, rms[n], host)


# ------------------------------------------------------------------ 2. converged fields against sparse LU
def _bench_params(stall):
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=20000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=stall)


@pytest.mark.parametrize("method", METHODS)
def test_bench_map_against_exact_solution(method):
    """The bench map operator (512 x 256, fp64) at every 16th benchmark location, every solve to r1.
    No stall detector: the BiCGStab residual is not monotone, and with the block-line preconditioner alone it can sit on a
    plateau for more than 10 checks of 5 iterations far above its round-off floor (stall_checks = 10 stopped location 0 at a
    field error of 9e-6 on a B200).  r1 = 1e-12 rms(f_n) as in the benchmark for line2_bicgstab; line_bicgstab leaves the
    smooth error components largest, and at that tolerance location 0 was 3e-8 from the exact field, so it solves to 1e-13."""
    import bench
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = bench.heat_rows(512)[::16]
    r1_rel = bench.R1_REL if method == "line2_bicgstab" else 0.1 * bench.R1_REL
    m = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method=method, r1_rel=r1_rel)
    tab = m.run(heat, _bench_params(0))
    psi, f = m.field("psi"), m.field("f")
    assert m.kernel_info()[0] == 5
    m.close()
    assert np.all(tab[:, 2] == 0), np.unique(tab[:, 2])
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    exact = ExactSolver(case.coe).solve(f)
    fe = np.array([rel_l2(psi[n], exact[n]) for n in range(len(heat))])
    ee = np.array([abs(tab[n, 5] - efficiency_row(exact[n], row, case)["efficiency"]) / abs(tab[n, 5]) for n, row in enumerate(heat)])
    print(f"{method} map: iterations {int(tab[:, 0].min())}-{int(tab[:, 0].max())}, field error {fe.max():.2e}, "
          f"efficiency error {ee.max():.2e}")
    assert np.all(fe < 1e-8), fe
    assert np.all(ee < 1e-6), ee


@pytest.mark.parametrize("method", METHODS)
def test_series_across_the_whole_series_against_exact_solution(method):
    """Eight snapshots spread over the 1,024-long series, the late non-symmetric ones included; one operator per solve."""
    import bench
    import xlab_ee_fortran_b200 as X  # noqa: F401
    from tests.exact_oracle import ke_gen
    from tests.map_oracle import background_theta
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.time_series import TimeSeries
    NR, NZ, LR, LZ = bench.NR, bench.NZ, bench.LR, bench.LZ
    firsts = (0, 150, 341, 500, 700, 850, 950, 1023)
    params = np.concatenate([W.series_params(1, total=1024, first=q) for q in firsts])
    ts = TimeSeries(NR, NZ, LR, LZ, len(firsts), "f64", arith="fast", method=method, r1_rel=bench.R1_REL)
    tab = ts.run(params, _bench_params(20))
    assert ts.probe_ms() == 0.0
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
        print(f"{method} snapshot {q}: {int(tab[n, 0])} iterations, err {int(tab[n, 2])}, field {e:.2e}, ke_gen {ek:.2e}")
        assert e < 1e-8, (q, e)
        assert ek < 1e-6, (q, ek)


# ------------------------------------------------------------------ 3. stop decisions
# method, arith, dtype, kernel, shared operator, nx, ny, nb, check_step, converge_time, lost_rate, r2, stall_checks
ROWS = {
    "line_bicg-f32": ("line_bicgstab", "fast", "f32", 0, True, 128, 40, 12, 2, 2, 1, 0.0, 0),
    "line_bicg-persolve": ("line_bicgstab", "fast", "f64", 0, False, 136, 70, 5, 2, 1, 5, 0.0, 0),
    "line2_bicg-stall": ("line2_bicgstab", "fast", "f64", 0, True, 200, 56, 12, 3, 2, 1, 1.5, 10),
    "line2_bicg-persolve": ("line2_bicgstab", "fast", "f64", 0, False, 128, 72, 5, 3, 1, 5, 0.0, 0),
}


def _case(key):
    with mock.patch.dict(SR.ROWS, {key: ROWS[key]}):
        return SR.Case(key)


@pytest.mark.parametrize("key", list(ROWS))
def test_stop_decisions_match_replay(key):
    torch, X = _mods()
    case = _case(key)
    T = case.dt
    eps = float(np.finfo(T).eps)
    plan = case.plan(X)
    seq = SR._sequences(torch, X, case, plan)
    # a. the residual check m measured is that of the iterate after m * check_step iterations
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
        # c. the reversed batch gives every solve the same bits
        rev = plan if case.shared else case.plan(X, case.coe[::-1].copy())
        g2, o2 = SR._solve(torch, rev, case.P[::-1].copy(), case.F[::-1].copy(),
                           case.params(X, max_iter=max_iter, r1_per_solve=torch.from_numpy(r1[::-1].copy()).cuda()))
        assert np.array_equal(g2[::-1], got)
        for k in ("iters", "err", "r1", "r2"):
            assert np.array_equal(o2[k][::-1], out[k], equal_nan=True), k
        if rev is not plan:
            rev.close()
    assert len(stops) >= 4 and max_iter in stops, sorted(stops)
    if case.r2 == 0:
        assert min(stops) == case.ct * case.cs, sorted(stops)
    plan.close()


@pytest.mark.parametrize("method", METHODS)
def test_call_history_does_not_change_a_solve(method):
    """A solve after solves and sweeps with other check steps, sizes of max_iter and an explicit rho_jacobi (ignored)
    gives the bits of the first; cheb_params() stays (0, 1) and sweep_kernel_stats counts two sweeps per iteration."""
    torch, X = _mods()
    nx, ny, nb = 128, 72, 3
    a, b, c = _aniso(nx, ny, seed=3)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    rng = np.random.default_rng(5)
    F = rng.standard_normal((nb, ny, nx)); P = rng.standard_normal((nb, ny, nx))
    plan = X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method=method)
    plan.set_coe_aos(coe)
    prm = lambda **kw: X.SolveParams(**{**dict(max_iter=3000, check_step=4, converge_time=2, lost_rate=5, r1=1e-9, r2=0.0), **kw})
    gA, oA = SR._solve(torch, plan, P, F, prm())
    assert np.all(oA["err"] == 0), oA
    plan.sweep_kernel_stats(reset=True)
    SR._solve(torch, plan, P, F, prm(check_step=7, rho_jacobi=0.9, alpha=0.3))
    _sweeps(torch, plan, P, F, 13, 5)
    gC, oC = SR._solve(torch, plan, P, F, prm())
    assert np.array_equal(gC, gA)
    for k in ("iters", "err", "r1", "r2"):
        assert np.array_equal(oC[k], oA[k]), k
    assert plan.cheb_params() == (0.0, 1.0)
    _, sweeps = plan.sweep_kernel_stats()
    assert sweeps % 2 == 0 and sweeps >= 2 * (13 + int(oC["iters"].max()))
    plan.close()


@pytest.mark.parametrize("method", METHODS)
def test_exact_first_guess_breaks_down_and_stays_exact(method):
    """f = L psi from the library's own operator application: the residual is exactly 0, every iteration breaks down
    (rho = 0, alpha = 0/0) and restarts; the field comes back unchanged and the stop rule sees a zero residual."""
    torch, X = _mods()
    nx, ny, nb = 128, 66, 2
    a, b, c = _aniso(nx, ny, seed=9)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    P = np.random.default_rng(9).standard_normal((nb, ny, nx))
    plan = X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method=method)
    plan.set_coe_aos(coe)
    ft = plan.apply(torch.from_numpy(P).cuda())
    got, out = SR._solve(torch, plan, P, ft.cpu().numpy(), X.SolveParams(max_iter=50, check_step=3, converge_time=2, r1=1e-30))
    plan.close()
    assert np.array_equal(got, P)
    # check 1 (iteration 3) counts a converged check, check 2 stops on err_before == 0 (elliptic_tools.f90:206)
    assert np.all(out["r1"] == 0.0) and np.all(out["err"] == 0) and np.all(out["iters"] == 6), out


# ------------------------------------------------------------------ 4. the Fortran-facing entry
@pytest.mark.parametrize("method", METHODS)
def test_solve_elliptic_with_xee_method(method, monkeypatch):
    """solve_elliptic with XEE_METHOD=<method> XEE_ARITH=fast on reference case test1 (200 x 200, fp64)."""
    import xlab_ee_fortran_b200 as X
    from tests.util import ref_test1_inputs
    A, B, C, bc = ref_test1_inputs()
    d = O.Domain((0.0, 1.0), (0.0, 1.0), 200, 200, 0, 0)
    a, b, c = O.build_abc(A.astype(np.float64), B.astype(np.float64), C.astype(np.float64), d)
    g = O.geometry(d, np.float64)
    coe, _ = O.cal_coe(a, b, c, g["dr"], g["dz"], 200, 200)
    f = -B.astype(np.float64)
    r1 = 1e-11 * rms_interior(f)
    monkeypatch.setenv("XEE_METHOD", method); monkeypatch.setenv("XEE_ARITH", "fast")
    dat = bc.astype(np.float64).copy(); wk = np.zeros_like(dat)
    it, r1o, r2o, err = X.solve_elliptic(20000, 5, 2, 5, r1, 0.0, 1.0, dat, coe, f, wk, 200, 200)
    assert err == 0 and r1o < r1, (it, r1o, err)
    assert np.array_equal(wk, dat)
    x = ExactSolver(coe).solve(f, bc.astype(np.float64))
    print(f"{method} solve_elliptic: {it} iterations, field error {rel_l2(dat, x):.2e}")
    assert rel_l2(dat, x) < 1e-8


# ------------------------------------------------------------------ 5. loud failures
@pytest.mark.parametrize("kw,msg", [
    (dict(method="line2_bicgstab", dtype="f32"), "fp64"),
    (dict(method="line_bicgstab", arith="strict"), "FAST"),
    (dict(method="line2_bicgstab", arith="strict"), "FAST"),
    (dict(method="line_bicgstab", kernel=1), "kernel 5"),
    (dict(method="line2_bicgstab", kernel=4), "kernel 5"),
])
def test_unsupported_configurations_fail_loudly(kw, msg):
    _, X = _mods()
    base = dict(nbatch=2, dtype="f64", shared_coe=True, arith="fast")
    base.update(kw)
    with pytest.raises(RuntimeError, match=msg):
        X.Plan(128, 66, **base)
