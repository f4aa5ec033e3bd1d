"""line2_chebyshev against line2_mixed on the benchmark's workloads (fp64, 512 x 256, FAST arithmetic, r1 = 1e-12 rms).

Workloads: the 512-location efficiency-map shard, and the 128-snapshot time-series shards 0-127 and 896-1023 (the end is
the non-symmetric regime).  line2_chebyshev runs with the benchmark's settings (check_step 5); line2_mixed with
check_step 80, 100 and 130, i.e. fp32 sweeps per refinement step.  Both at converge_time 2 (the benchmark's) and 1; stall
detection as in the benchmark (10 checks for the map, 20 for the series).  Each configuration gets one untimed warm-up
call, then the configurations alternate for --runs timed calls each; a timed call ends in a device synchronise, and the
spectral probes are inside it for the series (one operator per solve).  Reported per configuration: solves/s, sweeps per
solve (fp32 sweeps for line2_mixed) and refinement steps per solve (mean), and microseconds per batch-wide sweep (the
event-timed sweep loop, coarse solves and, for line2_mixed, the fold and residual passes included, over the sweep count).
Writes one JSON document to --out and prints it; the card's name and power limit are part of it.

    python scripts/measure_mixed.py --runs 3 --out out/mixed.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import bench  # noqa: E402
import xlab_ee_fortran_b200 as X  # noqa: E402
from measure_krylov import card  # noqa: E402
from xlab_ee_fortran_b200 import workloads as W  # noqa: E402
from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap  # noqa: E402
from xlab_ee_fortran_b200.time_series import TimeSeries  # noqa: E402

CONFIGS = (("line2_chebyshev", 5), ("line2_mixed", 80), ("line2_mixed", 100), ("line2_mixed", 130))


def make(workload, method):
    if workload == "map":
        A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
        heat = bench.heat_rows(512)
        obj = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method=method, r1_rel=bench.R1_REL)
        return obj, (lambda p: obj.run(heat, p)), len(heat)
    first = {"series-0": 0, "series-896": 896}[workload]
    prm = np.ascontiguousarray(W.series_params(128, total=1024, first=first))
    obj = TimeSeries(bench.NR, bench.NZ, bench.LR, bench.LZ, 128, "f64", arith="fast", method=method, r1_rel=bench.R1_REL)
    return obj, (lambda p: obj.run(prm, p)), 128


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--workloads", default="map,series-0,series-896")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    result = dict(card=card(), runs=args.runs, workloads={})
    for wl in args.workloads.split(","):
        objs = {m: make(wl, m) for m in ("line2_chebyshev", "line2_mixed")}
        stall = 10 if wl == "map" else 20
        keys = [(m, cs, ct) for ct in (2, 1) for m, cs in CONFIGS]
        prm = {k: X.SolveParams(max_iter=2000000, check_step=k[1], converge_time=k[2], r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                                stall_checks=stall) for k in keys}
        for k in keys:                        # warm-up: module loads, operator setup, spectral estimate, tensor maps
            objs[k[0]][1](prm[k])
        rows = {k: [] for k in keys}
        for _ in range(args.runs):
            for k in keys:
                obj, call, n = objs[k[0]]
                obj.sweep_kernel_stats(reset=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                tab = call(prm[k])
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                ms, sweeps = obj.sweep_kernel_stats()
                it = tab[:, 0]
                rows[k].append(dict(seconds=dt, solves_per_s=n / dt, sweeps_per_solve=float(it.mean()), sweeps_max=int(it.max()),
                                    steps_per_solve=float(np.ceil(it / k[1]).mean()), us_per_sweep=1e3 * ms / max(sweeps, 1),
                                    probe_ms=obj.probe_ms() if hasattr(obj, "probe_ms") else 0.0,
                                    err=sorted(set(int(e) for e in tab[:, 2]))))
        for o in objs.values():
            o[0].close()
        result["workloads"][wl] = {f"{m} cs={cs} ct={ct}": r for (m, cs, ct), r in rows.items()}
        for (m, cs, ct), r in rows.items():
            last = r[-1]
            print(f"{wl:11s} {m:16s} cs {cs:3d} ct {ct}  solves/s {' '.join(f'{x['solves_per_s']:8.1f}' for x in r)}  sweeps/solve "
                  f"{last['sweeps_per_solve']:7.1f} (max {last['sweeps_max']})  steps/solve {last['steps_per_solve']:5.2f}  "
                  f"us/sweep {last['us_per_sweep']:7.1f}  probe ms {last['probe_ms']:.1f}  err {last['err']}", flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
