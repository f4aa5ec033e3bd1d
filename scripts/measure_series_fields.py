"""The time series on its parameters against the same series on caller-supplied fields (TimeSeries.run_fields).

Snapshots 0-127 of the 1,024-long series at the benchmark's grid (512 x 256, fp64, line2_chebyshev, FAST arithmetic,
r1 = 1e-12 of the initial residual, check_step 5, stall detection after 20 checks, as bench.py --workload series).  One
parametric run produces the fields A, B, C, Q, F and the rim of psi; the same fields then go through the host entry (numpy)
and the device entry (CUDA tensors already on the device).  Each configuration gets one untimed warm-up call, then the
three alternate for --runs timed calls each; a timed call ends in a device synchronise and includes the spectral probes.

Reported per configuration: snapshots/s, sweeps per snapshot, probe ms (host wall time of the spectral probes); for the host
entry also the upload time, measured as the same six arrays copied from pageable numpy memory to the device by torch,
timed alone.  Then the largest table and psi differences of each field run against the parametric run: the parametric run
probes every 8th operator of this smooth series and interpolates, the field runs probe every operator, so differences come
from the different Chebyshev weights only.  Writes one JSON document to --out and prints it; the card's name and power limit
are part of it.

    python scripts/measure_series_fields.py --runs 3 --out out/series_fields.json
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
from xlab_ee_fortran_b200.time_series import TimeSeries  # noqa: E402

NSNAP = 128


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
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
    host = (A, B, C, Q, F, bc)
    dev = tuple(torch.from_numpy(x).cuda() for x in host)
    torch.cuda.synchronize()
    calls = {
        "parametric": lambda: ts.run(params, prm),
        "fields_host": lambda: ts.run_fields(A, B, C, Q, prm, F=F, psi_bc=bc),
        "fields_dev": lambda: ts.run_fields(*dev[:4], prm, F=dev[4], psi_bc=dev[5]),
    }
    for call in calls.values():                # warm-up
        call()
    rows = {k: [] for k in calls}
    out = {}
    upload = []
    for _ in range(args.runs):
        for k, call in calls.items():
            ts.sweep_kernel_stats(reset=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tab = call()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            rows[k].append(dict(seconds=dt, snapshots_per_s=NSNAP / dt, sweeps_per_snapshot=float(tab[:, 0].mean()),
                                sweeps_max=int(tab[:, 0].max()), probe_ms=ts.probe_ms(), err=sorted(set(int(e) for e in tab[:, 2]))))
            out[k] = (tab, ts.field("psi"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tmp = [torch.from_numpy(x).cuda() for x in host]
        torch.cuda.synchronize()
        upload.append(time.perf_counter() - t0)
        del tmp
    ts.close()
    ref_tab, ref_psi = out["parametric"]
    diffs = {}
    for k in ("fields_host", "fields_dev"):
        tab, p = out[k]
        rel = np.abs(tab - ref_tab) / np.maximum(np.abs(ref_tab), 1e-300)
        diffs[k] = dict(table_max_rel={c: float(rel[:, i].max()) for i, c in enumerate(("iters", "r1", "err", "sum_Q", "ke_gen",
                                                                                            "efficiency", "w_absmax", "u_absmax"))},
                        psi_max_rel_l2=float(max(np.linalg.norm(p[n] - ref_psi[n]) / np.linalg.norm(ref_psi[n]) for n in range(NSNAP))),
                        bit_identical=bool(np.array_equal(tab, ref_tab) and np.array_equal(p, ref_psi)))
    diffs["host_vs_dev_bit_identical"] = bool(np.array_equal(out["fields_host"][0], out["fields_dev"][0])
                                              and np.array_equal(out["fields_host"][1], out["fields_dev"][1]))
    mib = sum(x.nbytes for x in host) / 2 ** 20
    result = dict(card=card(), runs=args.runs, nsnap=NSNAP, grid=[bench.NR, bench.NZ], method="line2_chebyshev", check_step=5,
                  configs=rows, upload=dict(mib=mib, seconds=upload), differences=diffs)
    for k, r in rows.items():
        print(f"{k:12s} snapshots/s {' '.join(f'{x['snapshots_per_s']:7.1f}' for x in r)}  sweeps/snapshot "
              f"{r[-1]['sweeps_per_snapshot']:6.1f} (max {r[-1]['sweeps_max']})  probe ms {' '.join(f'{x['probe_ms']:6.1f}' for x in r)}  "
              f"err {r[-1]['err']}", flush=True)
    print(f"host upload of {mib:.0f} MiB: {' '.join(f'{1e3 * s:.1f}' for s in upload)} ms", flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
