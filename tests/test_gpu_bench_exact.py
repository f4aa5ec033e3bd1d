"""The benchmarked configuration against the exact discrete solution (tests/exact_oracle.py: sparse LU of the same
nine-point operator, fp64, one refinement step).

The efficiency map runs exactly as the value leg of bench.py: 512 x 256, bench.heat_rows(512), line2_chebyshev in FAST
arithmetic, r1 = 1e-12 rms(f_n), check_step 5, stall_checks 10, through run_dev.  Its forcing, integrals, returned fields
and efficiencies are checked against host references that share no code with the library; the adjoint path, the two-level
coarse solve at the benchmark's coarse size (465 coarse unknowns padded to 512) and the time series at the benchmark shape
likewise.  North_star tolerances: fields within 1e-8 relative L2, efficiencies within 1e-6 relative.
"""
import numpy as np
import pytest

from tests.exact_oracle import ExactSolver, MapCase, efficiency_row, host_residual_rms, ke_gen, rms_interior
from tests.util import rel_l2

pytestmark = pytest.mark.gpu


def _bench_params():
    import bench
    import xlab_ee_fortran_b200 as X
    return X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=10), bench


def _run_map(A, B, C, heat, adjoint=False):
    """bench.py's value leg: one untimed and one timed call of run_dev on device-resident inputs; returns the second."""
    import torch
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    prm, bench = _bench_params()
    m = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method="line2_chebyshev",
                      adjoint_check=adjoint, r1_rel=bench.R1_REL)
    heat_t = torch.from_numpy(np.ascontiguousarray(heat)).cuda()
    table_t = torch.zeros((len(heat), 8), dtype=torch.float64, device="cuda")
    for _ in range(2):
        m.run_dev(heat_t, table_t, prm)
    torch.cuda.synchronize()
    out = dict(table=table_t.cpu().numpy(), psi=m.field("psi"), f=m.field("f"))
    if adjoint:
        out["eta"] = m.field("eta"); out["chi"] = m.field("chi")
    m.close()
    return out


@pytest.fixture(scope="module")
def bench_map():
    import bench
    from xlab_ee_fortran_b200 import workloads as W
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = bench.heat_rows(512)
    run = _run_map(A, B, C, heat)
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    ex = ExactSolver(case.coe)
    exact = ex.solve(run["f"])                 # the device's own forcing: isolates the solve (the forcing is checked on its own)
    return dict(A=A, B=B, C=C, heat=heat, case=case, ex=ex, exact=exact, **run)


# ------------------------------------------------------------------ a. forcing (heating_rhs_kernel)
def _check_forcing(f_dev, heat, case, rel):
    """Largest |f_dev - f_ref| / max|f_ref| over the locations, the reference evaluated in the device's precision."""
    worst = 0.0
    for n, row in enumerate(heat):
        ref = case.forcing(row, f_dev.dtype.type).astype(np.float64)
        scale = np.abs(ref).max()
        e = np.abs(f_dev[n].astype(np.float64) - ref).max() / scale
        worst = max(worst, e)
        assert e <= rel, (n, row, e)
    return worst


def test_bench_forcing_matches_oracle(bench_map):
    """f of all 512 locations (8 block columns, 64 block rows of the forcing kernel) against rhs_thermal(heat_field)."""
    worst = _check_forcing(bench_map["f"], bench_map["heat"], bench_map["case"], 1e-13)
    print(f"forcing: largest error {worst:.2e} of max|f_n|")


@pytest.mark.parametrize("shape,dtype,method,rel", [((200, 37), "f64", "jacobi", 1e-13), ((300, 70), "f32", "jacobi", 1e-6)])
def test_forcing_on_ragged_and_f32_maps(shape, dtype, method, rel):
    """Partial blocks in both directions (200 = 3 x 64 + 8 columns, 37 = 9 x 4 + 1 rows), and an f32 map over five
    block columns; one sweep only, the forcing is what is checked.  The f32 map is compared with the oracle's f32 chain:
    against the fp64 chain it differs by 3e-5 of max|f_n| on this grid, the effect of float32 grid coordinates
    (r ~ 5e5 m to 0.06 m against blobs 6e3 m wide), which the reference's real(4) build shares."""
    import xlab_ee_fortran_b200 as X
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap
    nr, nz = shape
    Lr, Lz = (0.0, 6.0e5), (0.0, 1.5e4)
    A, B, C = W.vortex_fields(nr, nz, Lr, Lz)
    dr, dz = Lr[1] / (nr - 1), Lz[1] / (nz - 1)
    heat = W.heating_lattice(6, 4, Lr, Lz, 3 * dr, 3 * dz)
    m = EfficiencyMap(A, B, C, Lr, Lz, len(heat), dtype, arith="fast", method=method, r1_rel=1e-12)
    m.run(heat, X.SolveParams(max_iter=1, check_step=1, converge_time=1, r1=1.0, r2=0.0))
    f = m.field("f"); m.close()
    assert f.dtype == (np.float64 if dtype == "f64" else np.float32)
    assert np.all(f[:, 0] == 0) and np.all(f[:, -1] == 0) and np.all(f[:, :, 0] == 0) and np.all(f[:, :, -1] == 0)
    worst = _check_forcing(f, heat, MapCase(A, B, C, Lr, Lz), rel)
    print(f"forcing {shape} {dtype}: largest error {worst:.2e} of max|f_n|")


# ------------------------------------------------------------------ b. integrals (map_integrals_kernel) of the device's psi
def test_bench_integrals_of_the_returned_field(bench_map):
    case, tab = bench_map["case"], bench_map["table"]
    worst_q = worst_k = 0.0
    for n, row in enumerate(bench_map["heat"]):
        r = efficiency_row(bench_map["psi"][n], row, case)
        _, ke_abs = ke_gen(bench_map["psi"][n], case.theta, case.d, case.k)
        eq = abs(tab[n, 3] - r["sum_Q"]) / abs(r["sum_Q"])
        ek = abs(tab[n, 4] - r["ke_gen"]) / abs(r["ke_gen"])
        worst_q, worst_k = max(worst_q, eq), max(worst_k, ek)
        assert eq <= 1e-12, (n, eq)
        # a sum of terms of both signs: its rounding error is relative to the sum of their magnitudes
        assert abs(tab[n, 4] - r["ke_gen"]) <= 1e-12 * ke_abs, (n, ek, ke_abs / abs(r["ke_gen"]))
        assert tab[n, 5] == pytest.approx(tab[n, 4] / tab[n, 3], rel=1e-15)
    print(f"integrals: largest relative error sum_Q {worst_q:.2e}, ke_gen {worst_k:.2e}")


# ------------------------------------------------------------------ c. the returned field
def test_bench_returned_fields_solve_the_equations(bench_map):
    tab, psi, f, coe = bench_map["table"], bench_map["psi"], bench_map["f"], bench_map["case"].coe
    err = tab[:, 2]
    assert np.all((err == 0) | (err == 4)), np.unique(err)
    assert np.all(psi[:, 0] == 0) and np.all(psi[:, -1] == 0) and np.all(psi[:, :, 0] == 0) and np.all(psi[:, :, -1] == 0)
    ratios = []
    for n in range(len(psi)):
        rf = rms_interior(f[n])
        host = host_residual_rms(psi[n], coe, f[n])
        assert host <= 2e-12 * rf, (n, host / rf, err[n])
        if err[n] == 0:
            assert tab[n, 1] <= 1e-12 * rf, (n, tab[n, 1] / rf)
        # the stop test measured the iterate before the returned one: close to, not equal to, the returned residual
        ratios.append(host / tab[n, 1])
    ratios = np.array(ratios)
    print(f"residuals: host/reported in [{ratios.min():.3f}, {ratios.max():.3f}], largest factor "
          f"{max(ratios.max(), 1 / ratios.min()):.3f}; {int((err == 4).sum())} solves stopped on the round-off floor")
    assert np.all((ratios >= 0.5) & (ratios <= 2.0))


# ------------------------------------------------------------------ d. north_star against the exact answer
def test_bench_north_star_against_exact_solution(bench_map):
    psi, exact, tab, case = bench_map["psi"], bench_map["exact"], bench_map["table"], bench_map["case"]
    assert np.all(bench_map["ex"].last_refinement <= 1e-11)
    fe = np.array([rel_l2(psi[n], exact[n]) for n in range(len(psi))])
    ee = np.array([abs(tab[n, 5] - efficiency_row(exact[n], row, case)["efficiency"]) / abs(tab[n, 5])
                   for n, row in enumerate(bench_map["heat"])])
    k = int(fe.argmax())
    print(f"north_star: largest field error {fe.max():.2e} (location {k}, heat {bench_map['heat'][k]}), "
          f"largest efficiency error {ee.max():.2e} (location {int(ee.argmax())})")
    assert np.all(fe < 1e-8), [(int(n), fe[n]) for n in np.argsort(fe)[::-1][:8]]
    assert np.all(ee < 1e-6), [(int(n), ee[n]) for n in np.argsort(ee)[::-1][:8]]


# ------------------------------------------------------------------ e. adjoint path (single chi solve, fused coarse matvec)
def test_bench_adjoint_eta_against_exact_solution(bench_map):
    case = bench_map["case"]
    heat = bench_map["heat"][:64]
    run = _run_map(bench_map["A"], bench_map["B"], bench_map["C"], heat, adjoint=True)
    chi = bench_map["ex"].solve(case.fchi)
    eta = case.eta(chi)
    print(f"adjoint: chi {rel_l2(run['chi'], chi):.2e}, eta {rel_l2(run['eta'], eta):.2e} relative L2")
    assert rel_l2(run["chi"], chi) < 1e-8
    assert rel_l2(run["eta"], eta) < 1e-8
    worst = 0.0
    for n, row in enumerate(heat):
        ref = efficiency_row(bench_map["exact"][n], row, case, eta=eta)["efficiency_eta"]
        e = abs(run["table"][n, 7] - ref) / abs(ref)
        worst = max(worst, e)
        assert e < 1e-6, (n, e)
    print(f"adjoint: largest efficiency_eta error {worst:.2e}")


# ------------------------------------------------------------------ two-level coarse solve at the bench coarse size
@pytest.fixture(scope="module")
def coarse_cases():
    """Two shared 512 x 256 operators and their numpy restatements (tests/twolevel_oracle.py, 465 coarse unknowns)."""
    from oracle import oracle as O
    from tests.test_gpu_line import _batch
    from tests.test_gpu_twolevel import _aniso
    from tests.twolevel_oracle import TwoLevel
    nx, ny = 512, 256
    a, b, c, F, P = _batch(nx, ny, 37, np.float64, seed=2024)
    coe_r, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    a, b, c = _aniso(nx, ny)
    coe_a, _ = O.cal_coe(a, b, c, 1.0, 1.0, nx, ny)
    tl = TwoLevel(coe_r)
    assert tl.shape == (15, 31)
    return dict(rand=(coe_r, F, P, tl), aniso=(coe_a, TwoLevel(coe_a)))


def _checked(nb):
    return sorted({0, 1, nb - 1} | ({32, 33} if nb > 32 else set()))     # 32..36: the ragged second n-tile


@pytest.mark.parametrize("nb", [4, 5, 37])
def test_line2_jacobi_sweeps_at_bench_coarse_size(coarse_cases, nb):
    """nb = 4 takes the per-solve coarse matvec, nb = 5 and 37 the split-K DMMA GEMM (one, two n-tiles)."""
    import torch
    import xlab_ee_fortran_b200 as X
    coe, F, P, tl = coarse_cases["rand"]
    F, P = F[:nb], P[:nb]
    plan = X.Plan(512, 256, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method="line2_jacobi")
    plan.set_coe_aos(coe)
    psi = torch.from_numpy(P.copy()).cuda(); ft = torch.from_numpy(F).cuda()
    rms = plan.sweeps(psi, ft, 0.45, 3, want_rms=True)
    plan.close()
    got = psi.cpu().numpy()
    for k in _checked(nb):
        ref, rref = tl.jacobi(P[k], F[k], 0.45, 3)
        assert rel_l2(got[k], ref) < 1e-11, (k, rel_l2(got[k], ref))
        assert abs(rms[k] - rref) <= 1e-10 * rref, (k, rms[k], rref)


@pytest.mark.parametrize("nb", [4, 37])
def test_line2_chebyshev_sweeps_at_bench_coarse_size(coarse_cases, nb):
    import torch
    import xlab_ee_fortran_b200 as X
    coe, tl = coarse_cases["aniso"]
    rng = np.random.default_rng(nb)
    F = rng.standard_normal((nb, 256, 512)); P = np.zeros((nb, 256, 512))
    plan = X.Plan(512, 256, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method="line2_chebyshev")
    plan.set_coe_aos(coe)
    psi = torch.from_numpy(P.copy()).cuda(); ft = torch.from_numpy(F).cuda()
    plan.sweeps(psi, ft, 1.0, 6)
    rho, gamma = plan.cheb_params()
    plan.close()
    assert 0.5 < rho < 1.0 and 0.3 < gamma < 1.2, (rho, gamma)
    got = psi.cpu().numpy()
    for k in _checked(nb):
        ref = tl.chebyshev_sweeps(P[k], F[k], gamma, rho, 6)
        assert rel_l2(got[k], ref) < 1e-11, (k, rel_l2(got[k], ref))


# ------------------------------------------------------------------ time series at the bench shape
def test_series_at_bench_shape_against_exact_solution():
    """Four snapshots spread over the 1024-long series (700: the late, strongly non-symmetric regime), one operator per
    solve.  The exact reference is built from the device's A, B, C, forcing and pumping row, so it isolates the solver."""
    import bench
    import xlab_ee_fortran_b200 as X
    from oracle import oracle as O
    from tests.map_oracle import background_theta
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.time_series import TimeSeries
    NR, NZ, LR, LZ = bench.NR, bench.NZ, bench.LR, bench.LZ
    firsts = (0, 341, 700, 1023)
    params = np.concatenate([W.series_params(1, total=1024, first=q) for q in firsts])
    ts = TimeSeries(NR, NZ, LR, LZ, len(firsts), "f64", arith="fast", method="line2_chebyshev", r1_rel=bench.R1_REL)
    tab = ts.run(params, X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                                       stall_checks=20))
    A, B, C, psi, f = (ts.field(q) for q in ("A", "B", "C", "psi", "f"))
    ts.close()
    assert np.all((tab[:, 2] == 0) | (tab[:, 2] == 4)), tab[:, :3]
    case = MapCase(A[0], B[0], C[0], LR, LZ)                 # only its domain, geometry and constants are used
    d, g, k = case.d, case.g, case.k
    for n, q in enumerate(firsts):
        a, b, c = O.build_abc(A[n], B[n], C[n], d)
        coe, _ = O.cal_coe(a, b, c, g["dr"], g["dz"], NR, NZ)
        bottom = W.series_fields_host(params[n], NR, NZ, LR, LZ)[3]
        assert np.allclose(psi[n][0], bottom, rtol=1e-12, atol=1e-14 * 7e7)                 # the pumping row is kept
        assert np.all(psi[n][-1] == 0) and np.all(psi[n][:, 0] == 0) and np.all(psi[n][:, -1] == 0)
        bc = np.zeros((NZ, NR)); bc[0] = psi[n][0]
        ex = ExactSolver(coe)
        x = ex.solve(f[n], bc)
        e = rel_l2(psi[n], x)
        ke_x, _ = ke_gen(x, background_theta(A[n], B[n], C[n], d, np.float64), d, k)
        ek = abs(tab[n, 4] - ke_x) / abs(ke_x)
        print(f"series snapshot {q}: {int(tab[n, 0])} sweeps, err {int(tab[n, 2])}, field {e:.2e}, ke_gen {ek:.2e}, "
              f"host residual {host_residual_rms(psi[n], coe, f[n]) / rms_interior(f[n]):.2e} rms(f)")
        assert e < 1e-8, (q, e)
        assert ek < 1e-6, (q, ek)
