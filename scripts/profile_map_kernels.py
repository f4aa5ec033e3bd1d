"""Per-kernel GPU time of the benchmark's default workload (efficiency map, 512 heating locations, 512 x 256, fp64,
line2_chebyshev, check_step 5) from torch.profiler with CUDA activities.  One untimed run, then --steps profiled runs;
prints one JSON document: the card (name, power limit, max SM clock, read in the same run) and, per kernel name, the
launch count, total and mean time.  Profile in a run of its own: tracing slows the host, so take end-to-end numbers from
bench.py.  XEE_SO selects the library build, as for every other script.

    python scripts/profile_map_kernels.py --steps 2
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import bench  # noqa: E402
import xlab_ee_fortran_b200 as X  # noqa: E402
from measure_krylov import card  # noqa: E402
from xlab_ee_fortran_b200 import workloads as W  # noqa: E402
from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--method", default="line2_chebyshev")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    X._lib.require_gpu()
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    heat = torch.from_numpy(bench.heat_rows(512)).cuda()
    table = torch.zeros((512, 8), dtype=torch.float64, device="cuda")
    m = EfficiencyMap(A, B, C, bench.LR, bench.LZ, 512, "f64", arith="fast", method=args.method, r1_rel=bench.R1_REL)
    prm = X.SolveParams(max_iter=2000000, check_step=5, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2, stall_checks=10)
    m.run_dev(heat, table, prm)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            m.run_dev(heat, table, prm)
        torch.cuda.synchronize()
    sweeps = table[:, 0].cpu().numpy()
    kernels = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and e.count > 0:
            us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            kernels[e.key] = {"count": e.count, "total_us": us, "mean_us": us / e.count}
    m.close()
    doc = {"card": card(), "method": args.method, "steps": args.steps, "sweeps_per_solve": [float(sweeps.min()), float(sweeps.max())],
           "kernels": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["total_us"]))}
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
