"""line2_chebyshev against line2_bicgstab on the benchmark's workloads (fp64, 512 x 256, FAST arithmetic, r1 = 1e-12 rms).

Workloads: the 512-location efficiency-map shard, and 128-snapshot time-series shards at the start, the middle and the end
of the 1,024-snapshot series (the end is the non-symmetric regime).  Each configuration gets one untimed warm-up call, then
the two methods alternate for --runs timed calls each; a timed call ends in a device synchronise.  The spectral probes of
Chebyshev are inside the timed call (one operator per solve: they run on every run()).  Writes one JSON document to --out
and prints it; the card's name and power limit are part of it.

    python scripts/measure_krylov.py --runs 3 --out out/krylov.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import bench  # noqa: E402
import xlab_ee_fortran_b200 as X  # noqa: E402
from xlab_ee_fortran_b200 import workloads as W  # noqa: E402
from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap  # noqa: E402
from xlab_ee_fortran_b200.time_series import TimeSeries  # noqa: E402

METHODS = ("line2_chebyshev", "line2_bicgstab")


def params():
    return X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                         stall_checks=20)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def make(workload, method):
    if workload == "map":
        A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
        heat = bench.heat_rows(512)
        obj = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method=method, r1_rel=bench.R1_REL)
        return obj, (lambda: obj.run(heat, params())), len(heat)
    first = {"series-start": 0, "series-middle": 448, "series-end": 896}[workload]
    prm = np.ascontiguousarray(W.series_params(128, total=1024, first=first))
    obj = TimeSeries(bench.NR, bench.NZ, bench.LR, bench.LZ, 128, "f64", arith="fast", method=method, r1_rel=bench.R1_REL)
    return obj, (lambda: obj.run(prm, params())), 128


def timed(obj, call):
    import torch
    obj.sweep_kernel_stats(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tab = call()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    _, sweeps = obj.sweep_kernel_stats()
    probe = obj.probe_ms() if hasattr(obj, "probe_ms") else 0.0
    return dt, tab, sweeps, probe


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--workloads", default="map,series-start,series-middle,series-end")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    result = dict(card=card(), runs=args.runs, workloads={})
    for wl in args.workloads.split(","):
        objs = {m: make(wl, m) for m in METHODS}
        for m in METHODS:                     # warm-up: module loads, operator setup, tensor maps
            objs[m][1]()
        rows = {m: [] for m in METHODS}
        for _ in range(args.runs):
            for m in METHODS:
                obj, call, n = objs[m]
                dt, tab, sweeps, probe = timed(obj, call)
                rows[m].append(dict(seconds=dt, solves_per_s=n / dt, probe_ms=probe, sweeps=int(sweeps),
                                    iters_mean=float(tab[:, 0].mean()), iters_max=int(tab[:, 0].max()),
                                    err=sorted(set(int(e) for e in tab[:, 2]))))
        for m in METHODS:
            objs[m][0].close()
        result["workloads"][wl] = rows
        for m in METHODS:
            r = rows[m]
            print(f"{wl:14s} {m:16s} solves/s {' '.join(f'{x['solves_per_s']:8.1f}' for x in r)}  iters mean {r[-1]['iters_mean']:.1f} "
                  f"max {r[-1]['iters_max']}  sweeps {r[-1]['sweeps']}  probe ms {r[-1]['probe_ms']:.1f}  err {r[-1]['err']}", flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
