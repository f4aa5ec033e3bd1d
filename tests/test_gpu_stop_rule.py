"""Stop decisions of every sweep-kernel family against an exact replay of the stop rule (tests/stop_rule.py).

Fields converge whether or not a solve stops at the right check, so these tests look at what the field tests cannot: iters,
err, r1 and r2 of every solve, the field a solve returns (it must be the iterate of exactly `iters` sweeps), and that the
answers do not depend on sync_every, on the batch order or on the plan's call history.

a. Per-check sequences: solve() with max_iter = m * check_step stops at check m, so its r1 is the residual the device
   measured at check m.  Each value is compared with a long-double host residual of the iterate the check sweep read.
b. Stop decisions: per-solve thresholds between the sequence values; iters, err, r1 and r2 must equal the replay bit for
   bit, for sync_every 1, 2 and 3, and every field must equal the fixed-sweep iterate sweeps(iters[n]).
c. Batch order: the reversed batch gives every solve the same bits.
"""
import numpy as np
import pytest

from oracle import oracle as O
from tests.exact_oracle import host_residual_rms
from tests.line_oracle import _OFFS
from tests.stop_rule import ERR_EXPLODE, ERR_OVER_MAX_ITERATION, replay, same_bits
from tests.test_gpu_parity import _rand_case
from tests.test_gpu_twolevel import _aniso

pytestmark = pytest.mark.gpu
DTS = {"f32": np.float32, "f64": np.float64}
M = 20          # checks per sequence
LOST_ROWS = {"cheb-v4"}   # rows whose residual rises between checks: a converge count is gained and lost before the stop


def _mods():
    import torch
    import xlab_ee_fortran_b200 as X
    return torch, X


# method, arith, dtype, kernel (0 = auto), shared operator, nx, ny, nb, check_step, converge_time, lost_rate, r2, stall_checks
ROWS = {
    "jacobi-v1": ("jacobi", "strict", "f64", 1, True, 70, 45, 11, 4, 1, 5, 0.0, 0),
    "jacobi-v2-persolve-f32": ("jacobi", "strict", "f32", 2, False, 136, 70, 9, 3, 1, 5, 0.0, 0),
    "jacobi-v3": ("jacobi", "strict", "f64", 3, True, 140, 70, 2, 4, 1, 5, 0.0, 0),
    "jacobi-v4": ("jacobi", "fast", "f64", 4, True, 192, 100, 70, 4, 1, 5, 0.0, 0),
    "cheb-v1-persolve-f32": ("chebyshev", "fast", "f32", 1, False, 96, 64, 5, 3, 1, 5, 0.0, 0),
    "cheb-v2-ragged": ("chebyshev", "fast", "f64", 2, True, 260, 13, 37, 2, 2, 1, 0.5, 0),
    "cheb-v3": ("chebyshev", "fast", "f64", 3, True, 67, 35, 2, 3, 1, 5, 0.0, 0),
    "cheb-v4": ("chebyshev", "fast", "f64", 4, True, 256, 128, 40, 3, 2, 1, 0.0, 0),
    "line_jacobi-straddle": ("line_jacobi", "fast", "f64", 0, True, 136, 70, 40, 3, 1, 5, 0.0, 0),
    "line_cheb-f32": ("line_chebyshev", "fast", "f32", 0, True, 128, 40, 40, 2, 2, 1, 0.0, 0),
    "line_cheb-persolve": ("line_chebyshev", "fast", "f64", 0, False, 136, 70, 5, 2, 1, 5, 0.0, 0),
    "line2_jacobi-matvec": ("line2_jacobi", "fast", "f64", 0, True, 128, 72, 3, 3, 1, 5, 0.0, 0),
    "line2_cheb-bench": ("line2_chebyshev", "fast", "f64", 0, True, 200, 56, 40, 5, 2, 1, 1.5, 10),
    "line2_cheb-persolve": ("line2_chebyshev", "fast", "f64", 0, False, 128, 72, 5, 3, 1, 5, 0.0, 0),
}


class Case:
    def __init__(self, key):
        (self.method, self.arith, name, self.kernel, self.shared, self.nx, self.ny, self.nb, self.cs, self.ct, self.lr,
         self.r2, self.stall) = ROWS[key]
        self.dt = DTS[name]
        self.alpha = 0.45 if self.method == "line2_jacobi" else 1.0
        nx, ny, nb, dt = self.nx, self.ny, self.nb, self.dt
        rng = np.random.default_rng(nx * 7 + ny + nb)
        nsets = 1 if self.shared else nb
        coes = []
        for q in range(nsets):
            if self.method.startswith("line"):
                a, b, c = _aniso(nx, ny, seed=11 + q)
            else:
                a, b, c, _, _ = _rand_case(nx, ny, np.float64, seed=nx + q, bscale=0.02)
            coes.append(O.cal_coe(a.astype(dt), b.astype(dt), c.astype(dt), 1.0, 0.5, nx, ny)[0])
        self.coe = coes[0] if self.shared else np.stack(coes)
        self.F = rng.standard_normal((nb, ny, nx)).astype(dt)
        self.P = rng.standard_normal((nb, ny, nx)).astype(dt)

    def coe_of(self, n):
        return self.coe if self.shared else self.coe[n]

    def plan(self, X, coe=None):
        p = X.Plan(self.nx, self.ny, nbatch=self.nb, dtype="f64" if self.dt == np.float64 else "f32",
                   shared_coe=self.shared, arith=self.arith, method=self.method, kernel=self.kernel)
        p.set_coe_aos(self.coe if coe is None else coe)
        return p

    def params(self, X, **kw):
        base = dict(check_step=self.cs, converge_time=self.ct, lost_rate=self.lr, r2=self.r2, alpha=self.alpha,
                    stall_checks=self.stall)
        base.update(kw)
        return X.SolveParams(**base)


def _solve(torch, plan, P, F, prm):
    psi = torch.from_numpy(P).cuda(); ft = torch.from_numpy(F).cuda()
    out = plan.solve(psi, ft, prm)
    return psi.cpu().numpy(), out


def _sweeps(torch, plan, P, F, alpha, k):
    psi = torch.from_numpy(P).cuda(); ft = torch.from_numpy(F).cuda()
    plan.sweeps(psi, ft, alpha, k)
    return psi.cpu().numpy()


def _magnitude(psi, coe, f):
    """rms over the interior of sum_k |c_k p_k| + |f| (long double): the scale of the residual's rounding error."""
    ld = np.longdouble
    psi = np.asarray(psi, np.float64).astype(ld); coe = np.asarray(coe, np.float64)
    ny, nx = psi.shape
    acc = np.abs(np.asarray(f, np.float64)[1:-1, 1:-1]).astype(ld)
    for k, (di, dj) in enumerate(_OFFS):
        acc += np.abs(coe[1:-1, 1:-1, k].astype(ld) * psi[1 + dj:ny - 1 + dj, 1 + di:nx - 1 + di])
    return float(np.sqrt((acc * acc).sum() / ld(acc.size)))


def _sequences(torch, X, case, plan):
    """seq[n, m-1]: the residual the device measured for solve n at check m."""
    seq = np.zeros((case.nb, M))
    for m in range(1, M + 1):
        _, out = _solve(torch, plan, case.P, case.F, case.params(X, max_iter=m * case.cs, r1=1e-30, r2=0.0, stall_checks=0))
        assert list(out["iters"]) == [m * case.cs] * case.nb and list(out["err"]) == [ERR_OVER_MAX_ITERATION] * case.nb, out
        seq[:, m - 1] = out["r1"]
    return seq


def _thresholds(case, seq, shift):
    """Per-solve r1 between the sequence values, so that the solves stop at many different checks: r1 just above a new
    lowest residual makes that check the first one under r1.  One kind in five never converges and runs to max_iter, which
    is not a check sweep; another puts r1 across a rise of the sequence.  `shift` rotates the kinds over the batch."""
    r1 = np.zeros(case.nb)
    for n in range(case.nb):
        e = seq[n]
        kind = (n + shift) % 5
        if kind == 4:
            r1[n] = 1e-30
            continue
        if kind == 3:   # a rise in the sequence: first under r1, then over it (a lost converge count when ct >= 2)
            ups = [k for k in range(1, M - 3) if e[k] > e[k - 1]]
            if ups:
                k = ups[(n // 5) % len(ups)]
                r1[n] = 0.5 * (e[k - 1] + e[k])
                continue
        lows = [k for k in range(M) if k == 0 or e[k] < e[:k].min()]
        pick = [0, 1, len(lows) // 2 + (n // 5) % 3, len(lows) - 1][kind]
        k = lows[min(pick, len(lows) - 1)]
        r1[n] = 0.5 * (e[k] + e[:k].min()) if k > 0 else 2.0 * e[0]
    return r1


@pytest.mark.parametrize("key", list(ROWS))
def test_stop_decisions_match_replay(key):
    torch, X = _mods()
    case = Case(key)
    T = case.dt
    eps = float(np.finfo(T).eps)
    plan = case.plan(X)
    seq = _sequences(torch, X, case, plan)
    if case.kernel:
        assert plan.kernel_info()[0] == case.kernel
    # a. the residual each check measured is that of the iterate the check sweep read: sweeps(m * cs - 1)
    for m in sorted({1, 2, M // 2, M}):
        it = _sweeps(torch, plan, case.P, case.F, case.alpha, m * case.cs - 1)
        for n in sorted({0, case.nb // 2, case.nb - 1} | set(range(0, case.nb, max(1, case.nb // 4)))):
            host = host_residual_rms(it[n], case.coe_of(n), case.F[n])
            tol = 16 * eps * _magnitude(it[n], case.coe_of(n), case.F[n]) + 4 * eps * seq[n, m - 1]
            assert abs(seq[n, m - 1] - host) <= tol, (key, m, n, seq[n, m - 1], host, tol)
    # b. stop decisions (small batches: several threshold sets, so that the row sees every kind of stop)
    max_iter = M * case.cs + 1            # not a check sweep (check_step >= 2)
    stops, lost = set(), False
    for shift in range(0, 5, case.nb):
        r1 = _thresholds(case, seq, shift).astype(T)
        want = []
        for n in range(case.nb):
            log = []
            want.append(replay(seq[n], T, r1[n], case.r2, case.ct, case.lr, max_iter, case.cs,
                               detect_explode=case.method.endswith("chebyshev"), stall_checks=case.stall, log=log))
            lost = lost or any(b[1] < a[1] for a, b in zip(log, log[1:]))
        stops |= {w[0] for w in want}
        _check_stops(torch, X, case, plan, r1, want, max_iter, key)
    assert len(stops) >= 4 and max_iter in stops, sorted(stops)
    if case.r2 == 0:
        assert min(stops) == case.ct * case.cs, sorted(stops)
    if key in LOST_ROWS:
        assert lost, "no lost converge count in this row"
    plan.close()


def _check_stops(torch, X, case, plan, r1, want, max_iter, key):
    r1_dev = torch.from_numpy(r1).cuda()
    runs = []
    for sync in (1, 2, 3):
        runs.append(_solve(torch, plan, case.P, case.F, case.params(X, max_iter=max_iter, r1_per_solve=r1_dev, sync_every=sync)))
    got, out = runs[0]
    for n in range(case.nb):
        it, err, o1, o2 = want[n]
        assert (out["iters"][n], out["err"][n]) == (it, err), (key, n, (out["iters"][n], out["err"][n]), (it, err))
        assert same_bits(out["r1"][n], o1) and same_bits(out["r2"][n], o2), (key, n, out["r1"][n], o1, out["r2"][n], o2)
    for g, o in runs[1:]:
        assert np.array_equal(g, got)
        for k in ("iters", "err", "r1", "r2"):
            assert np.array_equal(o[k], out[k], equal_nan=True), k
    for v in sorted(set(out["iters"].tolist())):
        ref = _sweeps(torch, plan, case.P, case.F, case.alpha, v)
        for n in np.nonzero(out["iters"] == v)[0]:
            assert np.array_equal(got[n], ref[n]), (key, n, v)
    # c. batch order
    if not (case.method.endswith("chebyshev") and not case.shared):
        rev = plan if case.shared else case.plan(X, case.coe[::-1].copy())
        g2, o2 = _solve(torch, rev, case.P[::-1].copy(), case.F[::-1].copy(),
                        case.params(X, max_iter=max_iter, r1_per_solve=torch.from_numpy(r1[::-1].copy()).cuda()))
        assert np.array_equal(g2[::-1], got)
        for k in ("iters", "err", "r1", "r2"):
            assert np.array_equal(o2[k][::-1], out[k], equal_nan=True), k
        if rev is not plan:
            rev.close()


def test_line_chunk_straddles_solve_32():
    """The line_jacobi row's batch of 40 runs in units of ln_chunk solves; one unit holds solves 31 and 32, whose stop flags
    come from two words of the done mask (xee_sweep_line.cuh).  pick_chunk restated: 136 x 70 is 3 x 5 tiles of 64 x 16."""
    nt, nb, sms = 3 * 5, 40, 148
    best, chunk = None, 1
    for ch in range(min(32, nb), min(4, nb) - 1, -1):
        units = nt * -(-nb // ch)
        g = min(sms, units)
        cost = -(-units // g) * (ch + 1)
        if best is None or cost < best:
            best, chunk = cost, ch
    assert 31 // chunk == 32 // chunk, chunk            # the unit [31 // chunk * chunk, ...) contains both
    # ... and the thresholds give its solves different stops (kinds cycle with period 5 over the solve index)
    assert len({n % 5 for n in range(31 // chunk * chunk, min(nb, (31 // chunk + 1) * chunk))}) >= 2


# ---- divergence: a point-Jacobi-unstable operator under FAST Chebyshev must stop with the explode bit on every kernel
DNX, DNY, DCS, DMAX = 64, 34, 20, 2000


def _divergent(dt):
    a, b, c, f, x0 = _rand_case(DNX, DNY, np.float64, seed=1, bscale=5.0)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, DNX, DNY)
    return coe.astype(dt), f.astype(dt), x0.astype(dt)


def test_divergent_operator_on_the_reference():
    coe, f, x0 = _divergent(np.float64)
    r = O.solve_elliptic(200, 1, 10, 5, 1e-30, 0.0, 1.0, x0, coe, f, trace_cap=200)
    e = r["trace"]["err_now"]
    assert e[-1] > 1e6 * e[0]


@pytest.mark.parametrize("kernel", [1, 2, 3, 4])
@pytest.mark.parametrize("stall", [0, 10])
def test_divergent_chebyshev_explodes(kernel, stall):
    torch, X = _mods()
    coe, f, x0 = _divergent(np.float64)
    nb = 2
    P = np.stack([x0, 0.5 * x0]); F = np.stack([f, -f])
    plan = X.Plan(DNX, DNY, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method="chebyshev", kernel=kernel)
    plan.set_coe_aos(coe)
    prm = lambda mi, st: X.SolveParams(max_iter=mi, check_step=DCS, converge_time=10, lost_rate=5, r1=1e-30, r2=0.0,
                                       rho_jacobi=0.99, detect_explode=False, stall_checks=st)
    # the device's own per-check residuals, until a run stops before its max_iter
    seqs = [[] for _ in range(nb)]
    for m in range(1, DMAX // DCS + 1):
        _, out = _solve(torch, plan, P, F, prm(m * DCS, 0))
        assert plan.kernel_info()[0] == kernel
        for n in range(nb):
            if len(seqs[n]) == m - 1 and out["iters"][n] == m * DCS:
                seqs[n].append(out["r1"][n])
        if all(len(s) < m for s in seqs):
            break
    _, out = _solve(torch, plan, P, F, prm(DMAX, stall))
    for n in range(nb):
        want = replay(seqs[n], np.float64, 1e-30, 0.0, 10, 5, DMAX, DCS, detect_explode=True, stall_checks=stall)
        assert want[0] < DMAX and want[1] == ERR_EXPLODE, want
        assert (out["iters"][n], out["err"][n]) == want[:2], (kernel, stall, n, out, want)
        assert same_bits(out["r1"][n], want[2]) and same_bits(out["r2"][n], want[3])
    plan.close()


# ---- call history: an explicit rho_jacobi applies to its own call only
@pytest.mark.parametrize("method,kernel", [("chebyshev", 1), ("chebyshev", 3), ("chebyshev", 4), ("line_chebyshev", 0)])
def test_explicit_rho_does_not_stick_to_the_plan(method, kernel):
    torch, X = _mods()
    nx, ny, nb = 64, 34, 2
    if method == "line_chebyshev":
        a, b, c = _aniso(nx, ny, seed=3)
    else:
        a, b, c, _, _ = _rand_case(nx, ny, np.float64, seed=3, bscale=0.02)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    rng = np.random.default_rng(5)
    F = rng.standard_normal((nb, ny, nx)); P = rng.standard_normal((nb, ny, nx))
    mk = lambda: X.Plan(nx, ny, nbatch=nb, dtype="f64", shared_coe=True, arith="fast", method=method, kernel=kernel)
    prm = lambda rho: X.SolveParams(max_iter=3000, check_step=10, converge_time=2, lost_rate=5, r1=1e-9, r2=0.0, rho_jacobi=rho)
    plan = mk(); plan.set_coe_aos(coe)
    gA, oA = _solve(torch, plan, P, F, prm(0.0)); cA = plan.cheb_params()
    gB, oB = _solve(torch, plan, P, F, prm(0.9))
    assert plan.cheb_params()[0] == 0.9 and not np.array_equal(oB["iters"], oA["iters"])
    gC, oC = _solve(torch, plan, P, F, prm(0.0))
    assert plan.cheb_params() == cA
    assert np.array_equal(gC, gA)
    for k in ("iters", "err", "r1", "r2"):
        assert np.array_equal(oC[k], oA[k]), k
    _solve(torch, plan, P, F, prm(0.9))
    s1 = _sweeps(torch, plan, P, F, 1.0, 37)
    fresh = mk(); fresh.set_coe_aos(coe)
    s2 = _sweeps(torch, fresh, P, F, 1.0, 37)
    assert np.array_equal(s1, s2) and plan.cheb_params() == fresh.cheb_params() == cA
    plan.close(); fresh.close()
