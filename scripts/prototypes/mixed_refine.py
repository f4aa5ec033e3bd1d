"""Prototype (CPU, scipy): fp64 iterative refinement with the bench operator rounded to fp32 and factored exactly.
x += A32^-1 (b - A64 x) for heating rows 0, 128, 256, 384 of bench.heat_rows(512); prints the relative RMS residual after
every step.  The inner solve is exact, so the numbers show what rounding the operator to fp32 costs by itself.
python scripts/prototypes/mixed_refine.py [steps]"""
import os
import sys

import numpy as np
import scipy.sparse.linalg as spla

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from tests.exact_oracle import MapCase, assemble, rim_rhs  # noqa: E402
from xlab_ee_fortran_b200 import workloads as W  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
A, B, C = W.vortex_fields(bench.NR, bench.NZ, bench.LR, bench.LZ)
case = MapCase(A, B, C, bench.LR, bench.LZ)
A64 = assemble(case.coe)
c32 = case.coe.astype(np.float32).astype(np.float64)
print("largest relative change of a coefficient: %.2e" % np.max(np.abs(c32 - case.coe) / np.maximum(np.abs(case.coe), 1e-300)))
lu32 = spla.splu(assemble(c32))
for q, row in zip(range(0, 512, 128), bench.heat_rows(512)[::128]):
    b = rim_rhs(case.coe, case.forcing(row)).ravel()
    x = np.zeros_like(b)
    r0 = np.sqrt((b ** 2).mean())
    res = []
    for _ in range(steps):
        x += lu32.solve(b - A64 @ x)
        res.append(np.sqrt(((b - A64 @ x) ** 2).mean()) / r0)
    print("row %3d: " % q + "  ".join("%.1e" % v for v in res))
