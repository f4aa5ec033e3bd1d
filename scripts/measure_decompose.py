"""The legacy efficiency decomposition of the time series (TimeSeries.decompose) against the field run it extends
(TimeSeries.run_fields), on the same inputs.

Snapshots 0-127 of the 1,024-long series at the benchmark's grid (512 x 256, fp64, line2_chebyshev, FAST arithmetic,
r1 = 1e-12 of the initial residual, check_step 5, stall detection after 20 checks, as bench.py --workload series).  One
parametric run produces the fields A, B, C, Q, F and the rim of psi; chi_bc adds a chi rim on the top and outer boundaries.
Both calls take CUDA tensors (the device entry).  decompose runs TENDENCY (testing_dt 3600 s), BARO_ALL, with chi_bc: nine
batched solves on three operator sets.  One untimed warm-up of each, then the two alternate for --runs timed calls each; a
timed call ends in a device synchronise.

Then one more decompose with XEE_TRACE=1, whose phase lines (host wall time around device-synchronised phases: stage I solve,
stage II kernels, each operator set, the chi solves and the check solve of each tag) are read from stderr; the probe time of
that call is reported beside them (it is inside the first solve after each operator set).  Last, xee_old_diagnose --r8 on
snapshot 0 written as .bin files, with --legacy-iters point-Jacobi sweeps per solve (the legacy loop always runs all of them),
timed end to end.  Writes one JSON document to --out and prints it; the card's name, power limit and max SM clock are part of it.

    python scripts/measure_decompose.py --runs 3 --out out/decompose.json
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import bench  # noqa: E402
import xlab_ee_fortran_b200 as X  # noqa: E402
from measure_krylov import card  # noqa: E402
from xlab_ee_fortran_b200 import _lib  # noqa: E402
from xlab_ee_fortran_b200 import workloads as W  # noqa: E402
from xlab_ee_fortran_b200.time_series import DECOMP_SOLVES, TimeSeries  # noqa: E402

NSNAP = 128
DT = 3600.0


def traced(fn):
    """fn() with XEE_TRACE=1; returns (result, the library's trace lines from stderr)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        os.environ["XEE_TRACE"] = "1"
        try:
            out = fn()
        finally:
            os.environ.pop("XEE_TRACE")
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        return out, [ln for ln in tmp.read().splitlines() if ln.startswith("xee trace:")]


def legacy_driver(A, B, C, Q, F, psi_bc, chi_bc, iters):
    exe = _lib.build_old_diagnose()
    nz, nr = A.shape
    with tempfile.TemporaryDirectory() as d:
        for name, arr in (("A", A), ("B", B), ("C", C), ("Q", Q), ("F", F), ("psi_bc", psi_bc), ("chi_bc", chi_bc)):
            arr.astype(np.float32).tofile(os.path.join(d, f"{name}.bin"))
        cfg = (f"CYLINDRICAL-TENDENCY-DENSITY_NORMAL-BARO_ALL\n{DT}\n{bench.LR[0]} {bench.LR[1]} {bench.LZ[0]} {bench.LZ[1]}\n"
               f"{nr} {nz}\n.\n.\nA.bin\nB.bin\nC.bin\nQ.bin\nF.bin\n1 1e-30 {iters} 1.0\n1 1e-30 {iters} 1.0\n"
               "yes\npsi_bc.bin\nyes\nchi_bc.bin\n")
        t0 = time.perf_counter()
        r = subprocess.run([exe, "--r8"], input=cfg, capture_output=True, text=True, cwd=d, timeout=3000)
        sec = time.perf_counter() - t0
    steps = [int(x) for x in re.findall(r"Relaxation uses\s+(\d+)\s+steps", r.stdout)]
    return dict(returncode=r.returncode, seconds=sec, solves=len(steps), sweeps_per_solve=steps)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--legacy-iters", type=int, default=20000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    prm = X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2, stall_checks=20)
    params = np.ascontiguousarray(W.series_params(NSNAP, total=1024, first=0))
    ts = TimeSeries(bench.NR, bench.NZ, bench.LR, bench.LZ, NSNAP, "f64", arith="fast", method="line2_chebyshev", r1_rel=bench.R1_REL)
    ts.run(params, prm)
    A, B, C, Q, F, psi = (ts.field(q) for q in ("A", "B", "C", "Q", "F", "psi"))
    bc = np.zeros_like(psi)
    bc[:, [0, -1], :] = psi[:, [0, -1], :]
    bc[:, :, [0, -1]] = psi[:, :, [0, -1]]
    r = np.linspace(*bench.LR, bench.NR); z = np.linspace(*bench.LZ, bench.NZ)
    chi = np.zeros_like(psi)
    chi[:, -1] = 2.0e11 * np.sin(np.pi * r / bench.LR[1]) * (r / bench.LR[1]) ** 2
    chi[:, :, -1] = 5.0e10 * np.sin(np.pi * z / bench.LZ[1])
    host = (A, B, C, Q, F, bc, chi)
    dev = tuple(torch.from_numpy(x).cuda() for x in host)
    torch.cuda.synchronize()
    calls = {
        "run_fields": lambda: ts.run_fields(*dev[:4], prm, F=dev[4], psi_bc=dev[5]),
        "decompose": lambda: ts.decompose(*dev[:4], prm, prm, F=dev[4], psi_bc=dev[5], chi_bc=dev[6], testing_dt=DT, baro="all"),
    }
    for call in calls.values():                # warm-up
        call()
    rows = {k: [] for k in calls}
    for _ in range(args.runs):
        for k, call in calls.items():
            ts.sweep_kernel_stats(reset=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = call()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            sweep_ms, _ = ts.sweep_kernel_stats()
            row = dict(ms=1e3 * dt, probe_ms=ts.probe_ms(), sweep_kernel_ms=sweep_ms)
            if k == "run_fields":
                row.update(sweeps_per_solve=float(out[:, 0].mean()), err=sorted(set(int(e) for e in out[:, 2])))
            else:
                tab, it, err = out
                row.update(sweeps_per_solve={s: float(it[:, j].mean()) for j, s in enumerate(DECOMP_SOLVES)},
                           err=sorted(set(int(e) for e in err.ravel())), nan_columns=int(np.isnan(tab).any(axis=0).sum()))
            rows[k].append(row)
    ts.sweep_kernel_stats(reset=True)
    _, lines = traced(calls["decompose"])
    phases = {}
    for ln in lines:
        m = re.match(r"xee trace:\s+(.*?)\s+([0-9.]+) ms", ln)
        if m:
            phases.setdefault(m.group(1).strip(), []).append(float(m.group(2)))
    traced_probe_ms = ts.probe_ms()
    ts.close()
    legacy = legacy_driver(A[0], B[0], C[0], Q[0], F[0], bc[0], chi[0], args.legacy_iters)
    result = dict(card=card(), runs=args.runs, nsnap=NSNAP, grid=[bench.NR, bench.NZ], method="line2_chebyshev", check_step=5,
                  configs=rows, traced_decompose=dict(phases_ms=phases, probe_ms=traced_probe_ms),
                  legacy_driver_one_snapshot=dict(max_iter_per_solve=args.legacy_iters, **legacy))
    for k, r in rows.items():
        print(f"{k:10s} ms {' '.join(f'{x['ms']:8.1f}' for x in r)}  probe ms {' '.join(f'{x['probe_ms']:7.1f}' for x in r)}", flush=True)
    print("traced decompose phases (ms):", {k: [round(x, 1) for x in v] for k, v in phases.items()}, "probe ms", round(traced_probe_ms, 1))
    print("legacy driver, one snapshot:", legacy)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
