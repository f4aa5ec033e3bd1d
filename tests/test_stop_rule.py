"""tests/stop_rule.py::replay against the reference's own stop decisions (the oracle, elliptic_tools.f90:93-265 restated),
and against hand-worked sequences for the extensions the reference lacks (explode and stall rules, include/xee_b200.h)."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.stop_rule import ERR_EXPLODE, ERR_OVER_MAX_ITERATION, ERR_STALLED, replay, same_bits

DTS = {"f32": np.float32, "f64": np.float64}


def _case(dt, nx=14, ny=11, seed=3):
    rng = np.random.default_rng(seed)
    a = (1.0 + rng.random((ny - 2, nx - 1))).astype(dt); c = (1.0 + rng.random((ny - 1, nx - 2))).astype(dt)
    b = (0.02 * rng.standard_normal((ny - 1, nx - 1))).astype(dt)
    f = rng.standard_normal((ny, nx)).astype(dt); x0 = rng.standard_normal((ny, nx)).astype(dt)
    coe, _ = O.cal_coe(a, b, c, 1.0, 0.5, nx, ny)
    return coe, f, x0


def _oracle(coe, f, x0, max_iter, cs, ct, lr, r1, r2, alpha=1.0):
    return O.solve_elliptic(max_iter, cs, ct, lr, r1, r2, alpha, x0, coe, f, trace_cap=max_iter // cs + 1)


def _check_against_oracle(dt, coe, f, x0, max_iter, cs, ct, lr, r1, r2):
    ref = _oracle(coe, f, x0, max_iter, cs, ct, lr, r1, r2)
    log = []
    it, err, o1, o2 = replay(ref["trace"]["err_now"], dt, r1, r2, ct, lr, max_iter, cs, log=log)
    assert (it, err) == (ref["max_iter"], ref["err"]), ((it, err), (ref["max_iter"], ref["err"]))
    assert type(o1) is dt and type(o2) is dt
    assert same_bits(o1, ref["r1"]) and same_bits(o2, ref["r2"]), ((o1, o2), (ref["r1"], ref["r2"]))
    return ref, log


def _decremented(log):
    return any(b[1] < a[1] for a, b in zip(log, log[1:]))


@pytest.mark.parametrize("name", ["f32", "f64"])
def test_replay_matches_oracle_stop_decisions(name):
    dt = DTS[name]
    coe, f, x0 = _case(dt)
    cs = 3
    base = _oracle(coe, f, x0, 60 * cs, cs, 10, 5, 1e-30, 0.0)
    e = base["trace"]["err_now"]; q = np.abs(base["trace"]["ratio"])
    assert len(e) == 60 and np.all(np.diff(e) < 0)
    # r1 alone decides (converge_time 3): first below r1 at check 9, stop at check 11
    ref, _ = _check_against_oracle(dt, coe, f, x0, 60 * cs, cs, 3, 2, float(e[7]), 0.0)
    assert ref["err"] == 0 and ref["max_iter"] == 11 * cs
    # r2 alone decides
    ref, _ = _check_against_oracle(dt, coe, f, x0, 60 * cs, cs, 2, 5, 0.0, float(q[10]))
    assert ref["err"] == 0 and ref["max_iter"] < 60 * cs
    # both decide: r2 holds from check 6 on, r1 only from check 14 on
    ref, _ = _check_against_oracle(dt, coe, f, x0, 60 * cs, cs, 2, 5, float(e[12]), float(q[5]))
    assert ref["err"] == 0 and ref["max_iter"] == 15 * cs
    # max_iter on a check sweep and on a non-check sweep (r1 tiny: never converges)
    ref, _ = _check_against_oracle(dt, coe, f, x0, 20 * cs, cs, 10, 5, 1e-30, 0.0)
    assert (ref["err"], ref["max_iter"]) == (ERR_OVER_MAX_ITERATION, 20 * cs)
    ref, _ = _check_against_oracle(dt, coe, f, x0, 20 * cs + 2, cs, 10, 5, 1e-30, 0.0)
    assert (ref["err"], ref["max_iter"]) == (ERR_OVER_MAX_ITERATION, 20 * cs + 2)
    ref, _ = _check_against_oracle(dt, coe, f, x0, cs - 1, cs, 10, 5, 1e-30, 0.0)    # no check at all: r1 = r2 = 0
    assert (ref["err"], ref["max_iter"], ref["r1"], ref["r2"]) == (ERR_OVER_MAX_ITERATION, cs - 1, 0.0, 0.0)


@pytest.mark.parametrize("name", ["f32", "f64"])
def test_replay_matches_oracle_lost_rate(name):
    """On the round-off floor the ratio wanders around zero: with a small r2 the converge count is gained and lost again.
    The case is searched for on the reference's own trace, then run once more with those settings."""
    dt = DTS[name]
    coe, f, x0 = _case(dt, seed=5)
    cs, n = 1, 4000 if dt == np.float64 else 800
    base = _oracle(coe, f, x0, n, cs, 10, 5, 1e-30, 0.0)
    q = np.abs(base["trace"]["ratio"])
    found = None
    for r2 in np.quantile(q[n // 2:], [0.3, 0.5, 0.7]):
        for ct, lr in ((3, 1), (3, 2), (4, 2), (2, 1)):
            log = []
            it, err, _, _ = replay(base["trace"]["err_now"], dt, 0.0, float(r2), ct, lr, n, cs, log=log)
            if err == 0 and _decremented(log):
                found = (float(r2), ct, lr)
                break
        if found:
            break
    assert found, "no converge-count decrement found on the round-off floor"
    r2, ct, lr = found
    ref, log = _check_against_oracle(dt, coe, f, x0, n, cs, ct, lr, 0.0, r2)
    assert ref["err"] == 0 and _decremented(log)


@pytest.mark.parametrize("name", ["f32", "f64"])
def test_replay_matches_oracle_zero_residual(name):
    """f = L psi0 in the reference's own arithmetic: the residual is exactly 0, the iterate never moves, and the
    err_before == 0 stop (:206) fires at the second check."""
    dt = DTS[name]
    coe, _, x0 = _case(dt, seed=7)
    f = O.do_elliptic(x0, coe)
    ref, _ = _check_against_oracle(dt, coe, f, x0, 100, 4, 10, 5, 1e-6, 0.0)
    assert ref["trace"]["err_now"][0] == 0.0
    assert (ref["err"], ref["max_iter"], ref["r1"]) == (0, 8, 0.0) and np.isnan(ref["r2"])   # ratio (0 - 0) / 0


# ---- extensions: expected results written out from include/xee_b200.h:146-148 and the 1e6 rule of the accelerated methods
@pytest.mark.parametrize("name", ["f32", "f64"])
def test_replay_stall_rule(name):
    dt = DTS[name]
    seq = [1.0, 0.5, 0.4996, 0.4996, 0.4996, 0.3, 0.2, 0.1]   # 0.4996 is not below 0.999 * 0.5
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 80, 10, stall_checks=3)[:2] == (50, ERR_STALLED)
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 80, 10, stall_checks=4)[:2] == (80, ERR_OVER_MAX_ITERATION)
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 80, 10, stall_checks=0)[:2] == (80, ERR_OVER_MAX_ITERATION)
    it, err, r1, r2 = replay(seq, dt, 1e-9, 0.0, 10, 5, 80, 10, stall_checks=3)
    assert r1 == dt(0.4996) and r2 == 0
    # a converging stop at the same check takes precedence (no stall bit)
    assert replay(seq, dt, 0.4997, 0.0, 1, 5, 80, 10, stall_checks=1)[:2] == (30, 0)


@pytest.mark.parametrize("name", ["f32", "f64"])
def test_replay_explode_rules(name):
    dt = DTS[name]
    for bad in (np.inf, np.nan):
        seq = [1.0, 0.5, bad, bad]
        assert replay(seq, dt, 1e-9, 0.0, 10, 5, 40, 10, detect_explode=True)[:2] == (30, ERR_EXPLODE)
        assert replay(seq, dt, 1e-9, 0.0, 10, 5, 40, 10, detect_explode=False)[:2] == (40, ERR_OVER_MAX_ITERATION)
        # a non-finite residual on the last check: both bits
        assert replay(seq, dt, 1e-9, 0.0, 10, 5, 30, 10, detect_explode=True)[:2] == (30, ERR_EXPLODE | ERR_OVER_MAX_ITERATION)
    # 10^6 above the best residual seen: explode, only with the stall detector on (it keeps the best residual)
    seq = [1.0, 1e-3, 0.5, 2e3, 1e30]
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 50, 10, detect_explode=True, stall_checks=10)[:2] == (40, ERR_EXPLODE)
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 50, 10, detect_explode=True, stall_checks=0)[:2] == (50, ERR_OVER_MAX_ITERATION)
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 50, 10, detect_explode=False, stall_checks=10)[:2] == (50, ERR_OVER_MAX_ITERATION)
    # a stall stop is not taken at an explode check
    seq = [1.0, 1.0, 1.0, 1e7]
    assert replay(seq, dt, 1e-9, 0.0, 10, 5, 50, 10, detect_explode=True, stall_checks=3)[:2] == (40, ERR_EXPLODE)
    # the first check compares with the initial best (HUGE): HUGE * 1e6 overflows to inf, so no first-check explode
    big = float(np.finfo(dt).max) / 2
    assert replay([big, big / 2], dt, 1e-9, 0.0, 10, 5, 20, 10, detect_explode=True, stall_checks=10)[:2] == (20, ERR_OVER_MAX_ITERATION)
