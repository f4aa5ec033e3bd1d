"""Checks what `bench.py --dump-outputs DIR` wrote against the exact discrete solution (tests/exact_oracle.py: sparse LU of
the benchmark's operator, fp64), not against another build.   check_bench_outputs.py DIR

The efficiency-map workload only.  Its inputs are rebuilt from the number of rows of table.npy with bench.heat_rows (the
sampled solves in psi.npy are rank 0's rows, which start at location 0); each sampled location is solved exactly and its
field (relative L2) and efficiency (relative) errors are printed.  Exit 0 = every sampled location is within the
north_star tolerances (fields 1e-8, efficiencies 1e-6), 1 = one is not, 2 = not an efficiency-map dump."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FIELD_TOL, EFF_TOL = 1e-8, 1e-6


def main(path):
    import bench
    from tests.exact_oracle import ExactSolver, MapCase, efficiency_row
    from tests.util import rel_l2
    from xlab_ee_fortran_b200 import workloads as W
    table = np.load(os.path.join(path, "table.npy"))
    psi = np.load(os.path.join(path, "psi.npy"))
    pick = np.load(os.path.join(path, "psi_solves.npy")).astype(np.int64)
    # the map's last two columns (adjoint route) are 0 in the benchmark; the series writes max|w|, max|u| there
    if table.ndim != 2 or table.shape[1] != 8 or psi.shape[1:] != (bench.NZ, bench.NR) or np.any(table[:, 6:] != 0):
        print(f"{path}: not an efficiency-map dump of the {bench.NR}x{bench.NZ} benchmark; this checker handles the map workload only")
        return 2
    heat = bench.heat_rows(table.shape[0])
    A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
    case = MapCase(A, B, C, bench.LR, bench.LZ)
    exact = ExactSolver(case.coe).solve(np.stack([case.forcing(heat[n]) for n in pick]))
    ok = True
    print(f"{'row':>5} {'iters':>6} {'err':>3} {'field rel L2':>13} {'efficiency rel':>15}")
    for q, n in enumerate(pick):
        fe = rel_l2(psi[q], exact[q])
        eff = efficiency_row(exact[q], heat[n], case)["efficiency"]
        ee = abs(table[n, 5] - eff) / abs(eff)
        bad = not (fe < FIELD_TOL and ee < EFF_TOL)
        ok &= not bad
        print(f"{n:>5d} {int(table[n, 0]):>6d} {int(table[n, 2]):>3d} {fe:>13.2e} {ee:>15.2e}{'  FAIL' if bad else ''}")
    print(f"{len(pick)} locations of {table.shape[0]}: {'within' if ok else 'NOT within'} the north_star tolerances "
          f"(fields {FIELD_TOL:g} relative L2, efficiencies {EFF_TOL:g} relative)")
    return 0 if ok else 1


if __name__ == "__main__":
    if len(sys.argv) != 2:
        print(__doc__)
        sys.exit(2)
    sys.exit(main(sys.argv[1]))
