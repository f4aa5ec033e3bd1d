"""Direct efficiency map against the discrete adjoint on the benchmark's vortex (fp64, 512 x 256, line2_chebyshev, FAST
arithmetic, r1 = 1e-12 rms of the forcing, resp. of g, check_step 5, stall detection 10 checks).

Timed, each call ending in a device synchronise:
  - run() on the benchmark's 512 heating locations (one solve per location);
  - adjoint_solve() + adjoint_eval() of the same 512 locations;
  - adjoint_eval() alone on 130,305 locations, one narrow blob (half a cell wide) per B cell of the grid.
The first adjoint_solve() of the map is timed on its own and split into setup (the L^T plan: operator, line factors, coarse
operator), spectral probe and the rest (sweeps, mu and eta_d); later solves reuse all of it.  After one untimed call of each
kind, the three calls alternate for --runs rounds.  The efficiencies of both routes are compared.  Writes one JSON document,
with the card's name, power limit and max SM clock read in the same run, to --out-dir/adjoint.json and prints it.

    python scripts/measure_adjoint.py --runs 5 --out-dir out
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


def cell_blobs(q0):
    ra = np.linspace(bench.LR[0], bench.LR[1], bench.NR); za = np.linspace(bench.LZ[0], bench.LZ[1], bench.NZ)
    R, Z = np.meshgrid((ra[:-1] + ra[1:]) / 2, (za[:-1] + za[1:]) / 2)
    n = R.size
    return np.stack([R.ravel(), Z.ravel(), np.full(n, 0.5 * (ra[1] - ra[0])), np.full(n, 0.5 * (za[1] - za[0])),
                     np.full(n, q0)], axis=1)


def timed(call):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = call()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out-dir", default=None)
    args = ap.parse_args()
    X._lib.require_gpu()
    gpu = card()
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = bench.heat_rows(512)
    blobs = cell_blobs(heat[0, 4])
    prm = X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2, stall_checks=10)
    m = EfficiencyMap(A, B, C, bench.LR, bench.LZ, len(heat), "f64", arith="fast", method="line2_chebyshev", r1_rel=bench.R1_REL)
    t_run0, table = timed(lambda: m.run(heat, prm))
    t_first, (it, r1, err) = timed(lambda: m.adjoint_solve(prm))
    tm = m.adjoint_timings()
    first = dict(seconds=t_first, setup_ms=tm["setup_ms"], probe_ms=tm["probe_ms"],
                 rest_ms=1e3 * t_first - tm["setup_ms"] - tm["probe_ms"], iters=it, r1=r1, err=err)
    adj = m.adjoint_eval(heat)
    m.adjoint_eval(blobs)
    rows = dict(run_512=[], adjoint_solve_eval_512=[], adjoint_eval_130305=[])
    for _ in range(args.runs):
        dt, table = timed(lambda: m.run(heat, prm))
        rows["run_512"].append(dt)
        dt, (it, _, _) = timed(lambda: (m.adjoint_solve(prm), m.adjoint_eval(heat))[0])
        rows["adjoint_solve_eval_512"].append(dt)
        dt, big = timed(lambda: m.adjoint_eval(blobs))
        rows["adjoint_eval_130305"].append(dt)
    adj = m.adjoint_eval(heat)
    gap = np.abs(adj[:, 2] - table[:, 5]) / np.abs(table[:, 5])
    direct_sweeps = table[:, 0]
    m.close()
    result = dict(
        card=gpu, runs=args.runs, untimed_first_run_s=t_run0, first_adjoint_solve=first,
        seconds={k: v for k, v in rows.items()},
        median_ms={k: 1e3 * float(np.median(v)) for k, v in rows.items()},
        locations_per_s=dict(run_512=512 / float(np.median(rows["run_512"])),
                             adjoint_solve_eval_512=512 / float(np.median(rows["adjoint_solve_eval_512"])),
                             adjoint_eval_130305=130305 / float(np.median(rows["adjoint_eval_130305"]))),
        adjoint_sweeps=it, direct_sweeps=dict(min=int(direct_sweeps.min()), median=float(np.median(direct_sweeps)),
                                              max=int(direct_sweeps.max())),
        efficiency_gap_adjoint_vs_run=dict(max=float(gap.max()), median=float(np.median(gap))))
    text = json.dumps(result, indent=1)
    if args.out_dir:
        os.makedirs(args.out_dir, exist_ok=True)
        with open(os.path.join(args.out_dir, "adjoint.json"), "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
