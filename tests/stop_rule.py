"""Exact host replay of the library's stop rule (test infrastructure only).

Restates finalize_check_kernel / stop_rule_check (csrc/xee_kernels.cuh) and finalize_maxiter_kernel operation by operation
in numpy scalars of the plan's dtype: the stop rule of solve_elliptic (elliptic_tools.f90:112-124, 160-164, 199-248) plus
the library's extensions, the explode rules (detect_explode) and the stall detector (stall_checks > 0).  The device does
each of these steps as one correctly rounded IEEE operation (Rn<T>), and so does numpy: given the per-check residuals
err_now the device measured, replay() predicts iters, err, r1 and r2 bit for bit.
"""
import numpy as np

ERR_OVER_MAX_ITERATION, ERR_EXPLODE, ERR_STALLED = 1, 2, 4


def replay(err_now_seq, dtype, r1, r2, converge_time, lost_rate, max_iter, check_step, detect_explode=False,
           stall_checks=0, log=None):
    """err_now_seq[m-1] = residual measured at check m (sweep m * check_step), at least up to the stop.
    Returns (iters, err, r1_out, r2_out) as solve() reports them; r1_out/r2_out are numpy scalars of `dtype`.
    `log` (a list) receives (cnt, converge_cnt, lose_cnt) after every check, to see which branches a case took."""
    T = np.dtype(dtype).type
    huge = T(np.finfo(T).max)
    check_step = check_step if check_step > 0 else 100          # :131-144
    converge_time = converge_time if converge_time > 0 else 10
    lost_rate = lost_rate if lost_rate > 0 else 5
    r1 = T(r1) if T(r1) > 0 else huge                           # :112-124
    r2 = T(r2) if T(r2) > 0 else huge
    err_before, best = huge, huge                               # :163
    ccnt = lcnt = errb = stall = 0
    err_now = ratio = T(0)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        for m in range(1, max_iter // check_step + 1):
            cnt = m * check_step
            err_now = T(err_now_seq[m - 1])
            ratio = np.abs(T(T(err_before - err_now) / err_before))   # :201, :205
            stop = False
            if err_before == 0:                                      # :206
                stop = True
            elif err_now < r1 and ratio < r2:                         # :211
                ccnt += 1; lcnt = 0
                stop = ccnt >= converge_time
            elif ccnt > 0:                                            # :221
                lcnt += 1
                if lcnt >= lost_rate:
                    ccnt -= 1; lcnt = 0
            if detect_explode and not (err_now == err_now and np.abs(err_now) <= huge):
                stop = True; errb |= ERR_EXPLODE
            if detect_explode and stall_checks > 0 and err_now > T(best * T(1e6)):
                stop = True; errb |= ERR_EXPLODE
            if stall_checks > 0 and not stop:
                if err_now < T(best * T(0.999)):
                    best = err_now; stall = 0
                else:
                    stall += 1
                    if stall >= stall_checks:
                        stop = True; errb |= ERR_STALLED
            err_before = err_now                                      # :233
            if log is not None:
                log.append((cnt, ccnt, lcnt))
            if cnt == max_iter:                                       # :242-244
                stop = True; errb |= ERR_OVER_MAX_ITERATION
            if stop:
                return cnt, errb, err_now, ratio
    # max_iter reached on a non-check sweep (finalize_maxiter_kernel)
    return max_iter, errb | ERR_OVER_MAX_ITERATION, err_now, ratio


def same_bits(a, b):
    """a and b are the same value (NaN equals NaN: a stop on a non-finite residual reports one)."""
    a, b = float(a), float(b)
    return a == b or (a != a and b != b)
