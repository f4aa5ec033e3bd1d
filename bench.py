#!/usr/bin/env python
"""bench.py - headline benchmark of the B200-native elliptic-solve hot path.

Metric (BASELINE.json): elliptic solves/sec and GB/s vs HBM peak on the 512x256 r-z grid.
Workload: one shard of the efficiency map (BASELINE config 4): `--nheat` heating locations per GPU
(default 512; 8 GPUs = 4096 locations) on a 512x256 grid, fp64, one balanced vortex shared by all
solves, every solve iterated to r1 = 1e-12 * rms(f_n).  A "step" is one complete pass: heating RHS
built on the device, all solves to tolerance, energy integrals, efficiency table (+ the gather at N>1).

  python bench.py --gpus N --steps K --warmup W          # ours (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W  # the reference algorithm on the host cores

Method (`--method`, default line2_chebyshev): Chebyshev-accelerated TWO-LEVEL block-line relaxation (v5 kernel: 32-point radial
blocks solved inside the sweep, plus a Galerkin coarse-grid correction on a 16 x 16-spaced bilinear space whose prolongation
is fused into the sweep kernel; same residual, tolerance and stop rule as solve_elliptic); `line_chebyshev` = the one-level
block-line method (the pure streaming kernel, last round's default); `chebyshev` = accelerated point
Jacobi on the temporally blocked kernel (v4); `jacobi` = the reference iteration.  Results of all four agree within the
north_star tolerances (tests/test_gpu_map.py, tests/test_gpu_line.py, tests/test_gpu_twolevel.py).

Workloads (`--workload`): `map` (default, above) and `series` = BASELINE config 5: `--nsnap` snapshots per GPU (default 128;
8 GPUs = the 1024-snapshot series) with ONE OPERATOR PER SOLVE (varying wind profile / Ekman pumping), thermal + dynamical
source term, built on the device from 21 parameters per snapshot.  `--total T` fixes the TOTAL number of locations /
snapshots (strong scaling: `--total 4096` is BASELINE config 4 as written at every N).

`value`  : whole-job solves/s with the operator and heating parameters resident in HBM.
`e2e`    : the same metric through the host-facing call (HOST A,B,C + heating table in, efficiency
           table out; H2D/D2H and operator assembly inside the timed region).
`roofline`: dominant kernel = the sweep kernel; achieved = algorithmic bytes / CUDA-event time.
`roofline_streaming_kernel`: the same for the one-level variant of the kernel (pure HBM streaming), one extra pass (N=1).
`cpu_baseline`: the oracle's literal restatement of the reference algorithm on the host cores, three variants
           (`ref_O3` = reference loop order at -O3, `ref_O0` = the same at -O0 like make-diagnosis.sh:10-11, `fair` = fused,
           contiguous loop order), each a bounded sample of Jacobi sweeps; solves/s EXTRAPOLATED linearly to the Jacobi sweep
           count of profiles/workload_constants.json (measured with the bit-identical GPU Jacobi path).
`like_for_like`: the same algorithm on both sides, nothing extrapolated: reference Jacobi point-sweeps/s, GPU (STRICT
           arithmetic, iterates bit-identical to the oracle) over CPU (ref_O3).  The headline `value`/`e2e` use a DIFFERENT
           iteration (`same_config: false`): their ratio to the reference arm = algorithmic factor x hardware factor.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NR, NZ = 512, 256
LR, LZ = (0.0, 1.0e6), (0.0, 1.5e4)
R1_REL = 1e-12
CONSTANTS = os.path.join(ROOT, "profiles", "workload_constants.json")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload_constants():
    return json.load(open(CONSTANTS)) if os.path.exists(CONSTANTS) else {}


def heat_rows(total):
    """The first `total` locations of BASELINE config 4's 64x64 = 4096 heating-location lattice, taken in a fixed
    scrambled order (odd-stride permutation) so that every prefix samples the whole r-z plane: N GPUs x 512
    locations is the same kind of work for every N, and N = 8 is exactly the full 4096-location map."""
    from xlab_ee_fortran_b200 import workloads as W
    dr, dz = LR[1] / (NR - 1), LZ[1] / (NZ - 1)
    lattice = W.heating_lattice(64, 64, LR, LZ, 2 * dr, 2 * dz)
    perm = (np.arange(4096, dtype=np.int64) * 2053) % 4096
    reps = (total + 4095) // 4096
    return np.concatenate([lattice[perm]] * reps)[:total]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


_CPU_CASE = {}


def cpu_case(threads, workload="map"):
    """Inputs of the CPU legs (built once per process): `threads` independent 512x256 fp64 solves of the bench workload."""
    key = (threads, workload)
    if key in _CPU_CASE:
        return _CPU_CASE[key]
    from oracle import oracle as O
    from xlab_ee_fortran_b200 import workloads as W
    from tests.map_oracle import heat_field
    dt = np.float64
    d = O.Domain(LR, LZ, NR, NZ, 0, 0)
    g = O.geometry(d, dt)
    if workload == "map":
        A, B, C = W.vortex_fields(NR, NZ, LR, LZ)
        a, b, c = O.build_abc(A.astype(dt), B.astype(dt), C.astype(dt), d)
        coe, _ = O.cal_coe(a, b, c, g["dr"], g["dz"], NR, NZ)
        rows = heat_rows(threads)
        F = np.stack([O.rhs_thermal(heat_field(r, g, dt), d)[1] for r in rows])
        P = np.zeros_like(F)
    else:   # series: one operator per solve, snapshots spread over the 1024-long series; thermal source term + pumping boundary row
        prm = np.concatenate([W.series_params(1, total=1024, first=int(q)) for q in np.linspace(0, 1023, threads).astype(int)])
        coes, F, P = [], [], []
        for row in prm:
            A, B, C, bottom, _ = W.series_fields_host(row, NR, NZ, LR, LZ)
            a, b, c = O.build_abc(A.astype(dt), B.astype(dt), C.astype(dt), d)
            coes.append(O.cal_coe(a, b, c, g["dr"], g["dz"], NR, NZ)[0])
            F.append(O.rhs_thermal(heat_field(row[14:19], g, dt), d)[1])
            p0 = np.zeros((NZ, NR)); p0[0] = bottom; P.append(p0)
        coe, F, P = np.stack(coes), np.stack(F), np.stack(P)
    _CPU_CASE[key] = (coe, F, P)
    return _CPU_CASE[key]


def cpu_sample(sweeps, threads, method_sweeps, variant="ref_O3", workload="map"):
    """The reference algorithm (oracle literal restatement: 4 passes per sweep, reference loop order) on the host
    cores: `threads` independent 512x256 fp64 solves of this workload, `sweeps` Jacobi sweeps each, one per thread.
    variant: ref_O3 | ref_O0 (same code at -O0, what make-diagnosis.sh builds) | fair (fused passes, contiguous loop order).
    solves/s is extrapolated linearly to `method_sweeps` (the Jacobi sweep count to the bench tolerance)."""
    from oracle import oracle as O
    coe, F, P = cpu_case(threads, workload)
    if variant == "fair":
        planar = np.ascontiguousarray(np.moveaxis(coe, -1, -3))          # (.., ny, nx, 9) -> (.., 9, ny, nx)
        sec = O.fair_batch(P, planar, F, 1.0, sweeps, threads=threads)["seconds"]
    else:
        sec = O.solve_batch(sweeps, 100, 10, 5, 1e-300, 0.0, 1.0, P, coe, F, threads=threads, variant="O0" if variant == "ref_O0" else "O3")["seconds"]
    sweeps_per_s = threads * sweeps / sec                 # aggregate over the cores
    return dict(seconds=sec, sweeps=sweeps, sweeps_per_s=sweeps_per_s, solves_per_s=sweeps_per_s / method_sweeps,
                point_sweeps_per_s=sweeps_per_s * (NR - 2) * (NZ - 2))


def jacobi_sweeps_constant(workload):
    k = workload_constants()
    key = "jacobi_sweeps_to_tol" if workload == "map" else "jacobi_sweeps_to_tol_series"
    return (float(k.get(key, 0)) or None), key


def run_reference(args):
    args.check_step = 100      # the Jacobi sweep count of profiles/workload_constants.json was measured with check_step 100
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    js, js_key = jacobi_sweeps_constant(args.workload)
    cores = O.max_threads()
    vals = []
    sweeps = args.ref_sweeps
    for s in range(args.warmup + args.steps):
        r = cpu_sample(sweeps, cores, js or 1.0, "ref_O3", args.workload)
        if s >= args.warmup:
            vals.append(r)
    v = float(np.mean([r["solves_per_s"] for r in vals])) if js else None
    ms = float(np.mean([r["seconds"] for r in vals])) * 1e3
    sample = (f"{cores} independent 512x256 fp64 solves (one per host thread), {sweeps} reference Jacobi sweeps each per step; "
              f"solves/s extrapolated linearly to the {js:.0f} sweeps Jacobi needs for r1=1e-12*rms(f) on this workload "
              f"(measured with the bit-identical GPU Jacobi path, profiles/workload_constants.json:{js_key})" if js else "no sweep-count constant")
    line = {"impl": "reference", "metric": "elliptic_solves_per_sec", "value": v, "unit": "solves/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, "jacobi (reference algorithm, elliptic_tools.f90:93-265)"),
            "cpu_baseline": {"value": v, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample,
                             "point_sweeps_per_s": float(np.mean([r["point_sweeps_per_s"] for r in vals]))},
            "e2e": {"value": v, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            # what this number is: NOT a run to tolerance.  A bounded sample of sweeps is timed and scaled by a sweep count
            # measured elsewhere; and it does not grow with --gpus (one host, all its cores, whatever N is), so the ratio of
            # the GPU arm to this line grows with N by construction.
            "extrapolated": True, "sweeps_timed_per_solve": sweeps, "sweeps_to_tolerance": js,
            "sweeps_to_tolerance_source": f"profiles/workload_constants.json:{js_key} (GPU STRICT Jacobi, bit-identical iterates)",
            "flat_in_n_gpus": True, "reference_is": "C++ restatement of the Fortran (no Fortran compiler in the image), -O3, reference loop order"}
    print(json.dumps(line), flush=True)


def workload_config(args, method):
    per = args.per_gpu
    if args.workload == "series":
        wl = (f"time-series diagnosis (BASELINE config 5): {per} snapshots per GPU of the 1024-snapshot series (varying wind profile / "
              f"Ekman pumping) on a {NR}x{NZ} r-z grid, ONE OPERATOR PER SOLVE, thermal + dynamical source term, every solve to "
              f"r1=1e-12*rms(initial residual)")
        cfg = {"workload": wl, "grid": [NR, NZ], "nsnap_per_gpu": per}
    else:
        wl = (f"efficiency-map shard (BASELINE config 4): {per} heating locations per GPU on a {NR}x{NZ} r-z grid, "
              f"shared vortex operator, every solve to r1=1e-12*rms(f)")
        cfg = {"workload": wl, "grid": [NR, NZ], "nheat_per_gpu": per}
    if args.total > 0:
        cfg["total"] = args.total
        cfg["workload"] += f"; STRONG scaling: {args.total} in total, split over the GPUs"
    cfg.update({"method": method, "tolerance": f"r1 = 1e-12 * rms(f_n) at 2 consecutive checks, {args.check_step} sweeps apart; r2 off",
                "l2_policy": "inputs larger than L2 (psi+psi'+f = %.2f GiB per GPU vs 126 MB L2)" % (3 * per * NR * NZ * 8 / 2 ** 30)})
    return cfg


def dump_outputs(path, table, field, n_local):
    """Writes what the last timed step computed as <path>/<name>.npy: `table` (float64), the result table the timed call
    returns (one row per solve, columns COLS of efficiency_map / time_series), and `psi` (float64), the solution fields
    of a fixed, seeded sample of at most 16 of this process's solves (1 MiB each on the bench grid), with their row
    numbers in `psi_solves`.  The inputs depend on the arguments only, so two builds can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "table.npy"), np.asarray(table, np.float64))
    pick = np.sort(np.random.default_rng(0).choice(n_local, size=min(16, n_local), replace=False))
    np.save(os.path.join(path, "psi_solves.npy"), pick.astype(np.float64))
    np.save(os.path.join(path, "psi.npy"), np.ascontiguousarray(field("psi")[pick], np.float64))


KERNEL_NAMES = {1: "sweep_direct_kernel (v1)", 2: "sweep_tma_kernel (v2)", 3: "solve_resident_kernel (v3)",
                4: "sweep_tb_kernel (v4, temporal blocking)", 5: "sweep_line_kernel (v5, block-line relaxation, TMA loads + TMA stores)"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import xlab_ee_fortran_b200 as X
    from xlab_ee_fortran_b200 import plan as P
    from xlab_ee_fortran_b200 import workloads as W
    from xlab_ee_fortran_b200.efficiency_map import EfficiencyMap, gather_rows, partition
    from xlab_ee_fortran_b200.time_series import TimeSeries

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        # stdout carries exactly ONE JSON line: NCCL prints "NCCL version ..." there when NCCL_DEBUG is WARN/VERSION, so the
        # communicator is created (first collective) with stdout pointed at stderr
        sys.stdout.flush()
        saved = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier(); torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1); os.close(saved)
    series = args.workload == "series"
    total = args.total if args.total > 0 else args.per_gpu * world
    a, b = partition(total, world, rank)
    nloc = b - a
    args.per_gpu = max(partition(total, world, r)[1] - partition(total, world, r)[0] for r in range(world))
    # stall_checks: 3 of the 4096 lattice locations (next to the vortex ring, where C jumps) sit on a round-off floor
    # of ~1.2e-12*rms(f) and can never reach 1e-12; they stop as "converged to the floor" (err bit 4) instead of
    # running to max_iter.  Any other error bit fails the run.
    prm = X.SolveParams(max_iter=args.max_iter, check_step=args.check_step, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2,
                        stall_checks=10 if not series else 20)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ value leg (inputs resident in HBM)
    if series:
        my = np.ascontiguousarray(W.series_params(nloc, total=max(total, 1024), first=a))
        m = TimeSeries(NR, NZ, LR, LZ, nloc, "f64", arith=args.arith, method=args.method, r1_rel=R1_REL, device=local)

        def step():
            t = m.run(my, prm)                       # 21 parameters per snapshot in, 8 result columns out (KB-scale, host)
            return (gather_rows(torch.from_numpy(t).cuda(), total) if world > 1 else t), t
    else:
        A, B, C = W.vortex_fields(NR, NZ, LR, LZ)
        my = np.ascontiguousarray(heat_rows(total)[a:b])
        m = EfficiencyMap(A, B, C, LR, LZ, nloc, "f64", arith=args.arith, method=args.method, r1_rel=R1_REL, device=local)
        heat_t = torch.from_numpy(my).cuda(); table_t = torch.zeros((nloc, 8), dtype=torch.float64, device="cuda")

        def step():
            m.run_dev(heat_t, table_t, prm)
            return (gather_rows(table_t, total) if world > 1 else table_t), table_t

    for _ in range(args.warmup):
        out, loc = step()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler: sampler.start()
    barrier()
    m.sweep_kernel_stats(reset=True); P.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out, loc = step()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = P.launch_count()
    sweep_ms, sweeps_done = m.sweep_kernel_stats()
    variant, sweeps_per_pass, sweep_launches = m.kernel_info()
    probe_ms = m.probe_ms() if series else None
    tab = loc if isinstance(loc, np.ndarray) else loc.cpu().numpy()
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out if isinstance(out, np.ndarray) else out.cpu().numpy(), m.field, nloc)
    ms_per_step = ms_total / args.steps
    value = total / (ms_per_step * 1e-3)
    # every rank's solves must have converged (err 0) or stopped on their round-off floor (err 4); sweep range over all ranks
    ok = float(np.all((tab[:, 2] == 0) | (tab[:, 2] == 4)))
    n_floor = int((tab[:, 2] == 4).sum())
    sw_min, sw_max = float(tab[:, 0].min()), float(tab[:, 0].max())
    if world > 1:
        t = torch.tensor([ok, sw_min], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN); ok = float(t[0].item()); sw_min = float(t[1].item())
        t = torch.tensor([sw_max], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX); sw_max = float(t[0].item())
        t = torch.tensor([float(n_floor)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM); n_floor = int(t[0].item())
    assert ok == 1.0, "a solve hit max_iter or exploded on some rank: not converged"
    # roofline of the dominant kernel: useful point-sweeps actually performed (per-solve sweep counts) x bytes
    interior = (NR - 2) * (NZ - 2)
    cheb = args.method.endswith("chebyshev"); line = args.method.startswith("line")
    fields = 4 if cheb else 3                                      # psi read, psi write, f read (+ psi_{k-1} for Chebyshev)
    # (two-level method: the coarse correction adds no field pass - its prolongation is fused into the sweep kernel; its own
    #  traffic, 32 doubles per tile and solve out and two 3 x 8 coarse patches in, is ~0.7 B per point and left out)
    opw = (13 if line else 9)                                      # operator words per point: 9 coefficients (+ m, u and 4 float planes)
    b_alg = 8.0 * (fields + (opw if series else opw / nloc))       # one operator per solve: it streams with every sweep
    alg_bytes = float(tab[:, 0].sum()) * interior * b_alg * args.steps
    achieved = alg_bytes / (sweep_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak()
    k = workload_constants()
    # dram bytes of ONE full-batch launch of this variant from its ncu --set full capture (profiles/), None if not captured
    tkey = f"sweep_kernel_dram_bytes_per_launch_v{variant}" + ("_two_level" if args.method.startswith("line2") else "")
    traffic = None if series else k.get(tkey, k.get("sweep_kernel_dram_bytes_per_launch") if variant == 2 else None)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": KERNEL_NAMES.get(variant, "sweep") + " (K3/K4)",
                "sweeps_per_launch_T": sweeps_per_pass,
                "avg_launch_us": sweep_ms / max(sweep_launches, 1) * 1e3, "launches": sweep_launches,
                "avg_sweep_us": sweep_ms / max(sweeps_done, 1) * 1e3, "sweeps": sweeps_done,
                "algorithmic_bytes_per_point_sweep": b_alg, "kernel_share_of_step": sweep_ms / ms_total,
                "sweeps_per_solve": [sw_min, sw_max],
                "mean_active_fraction_of_batch": float(tab[:, 0].sum()) * args.steps / max(sweeps_done * nloc, 1)}
    if probe_ms is not None:
        roofline["spectral_probe_share_of_step"] = probe_ms / ms_total
    eff_range = [float(tab[:, 5].min()), float(tab[:, 5].max())]
    m.close()
    # ------------------------------------------------------------------ like for like: the reference's own iteration on the GPU
    lfl = None
    if rank == 0 and world == 1 and not args.no_cpu and not series:
        mj = EfficiencyMap(A, B, C, LR, LZ, nloc, "f64", arith="strict", method="jacobi", r1_rel=R1_REL, device=local)
        pj = X.SolveParams(max_iter=args.lfl_sweeps, check_step=100, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2)
        mj.run_dev(heat_t, table_t, pj); mj.sweep_kernel_stats(reset=True)
        mj.run_dev(heat_t, table_t, pj)
        jms, jsw = mj.sweep_kernel_stats()
        lfl = {"gpu_point_sweeps_per_s": nloc * jsw * interior / (jms * 1e-3), "gpu_sweeps_timed": int(jsw), "gpu_kernel_variant": mj.kernel_info()[0],
               "gpu_arithmetic": "strict (every operation separately rounded, reference order: iterates bit-identical to the oracle)"}
        mj.close()
    # ------------------------------------------------------------------ the streaming kernel on its own
    # The default (two-level) sweep kernel is instruction-bound by design (it also restricts the residual and adds the coarse
    # correction on the fly); the ONE-level kernel is the pure HBM-streaming variant of the same code.  One untimed + one timed
    # pass of the same workload with it, so that the driver's record carries its roofline next to the headline's.
    streaming = None
    if rank == 0 and world == 1 and not series and args.method.startswith("line2") and not args.no_streaming:
        ms1 = EfficiencyMap(A, B, C, LR, LZ, nloc, "f64", arith=args.arith, method="line_chebyshev", r1_rel=R1_REL, device=local)
        p1 = X.SolveParams(max_iter=args.max_iter, check_step=25, converge_time=2, r1=1.0, r2=0.0, alpha=1.0, sync_every=2, stall_checks=10)
        ms1.run_dev(heat_t, table_t, p1); ms1.sweep_kernel_stats(reset=True)
        t0 = time.perf_counter(); ms1.run_dev(heat_t, table_t, p1); torch.cuda.synchronize(); dt1 = time.perf_counter() - t0
        sms, ssw = ms1.sweep_kernel_stats(); t1 = table_t.cpu().numpy()
        b1 = 8.0 * (4 + 13.0 / nloc)
        a1 = float(t1[:, 0].sum()) * interior * b1 / (sms * 1e-3) / 1e9
        streaming = {"kernel": "sweep_line_kernel (v5, one-level: method line_chebyshev)", "bound": "hbm", "achieved": a1, "peak": peak, "unit": "GB/s",
                     "frac": a1 / peak, "traffic": k.get("sweep_kernel_dram_bytes_per_launch_v5"), "avg_launch_us": sms / max(ssw, 1) * 1e3,
                     "launches": int(ssw), "sweeps_per_solve": [float(t1[:, 0].min()), float(t1[:, 0].max())],
                     "mean_active_fraction_of_batch": float(t1[:, 0].sum()) / max(ssw * nloc, 1), "solves_per_s": nloc / dt1,
                     "algorithmic_bytes_per_point_sweep": b1}
        ms1.close()
    if not series:
        del heat_t, table_t
    # ------------------------------------------------------------------ e2e leg (host buffers, whole call)
    if series:
        hpar = torch.from_numpy(my).pin_memory()

        def e2e_step():
            mm = TimeSeries(NR, NZ, LR, LZ, nloc, "f64", arith=args.arith, method=args.method, r1_rel=R1_REL, device=local)
            t = mm.run(hpar.numpy(), prm)
            mm.close()
            return gather_rows(torch.from_numpy(t).cuda(), total) if world > 1 else t
        h2d, d2h = int(nloc * 21 * 8), int(nloc * (8 * 8 + 4 + 4 + 8 + 8))
        call = "TimeSeries(...).run(params host [n,21]) -> table host (xee_series_create + xee_series_run_host + xee_series_destroy)"
    else:
        hA, hB, hC = (torch.from_numpy(x).pin_memory() for x in (A, B, C))
        hheat = torch.from_numpy(my).pin_memory()

        def e2e_step():
            ts = [time.perf_counter()]
            mm = EfficiencyMap(hA.numpy(), hB.numpy(), hC.numpy(), LR, LZ, nloc, "f64", arith=args.arith, method=args.method,
                               r1_rel=R1_REL, device=local)
            ts.append(time.perf_counter())
            t = mm.run(hheat.numpy(), prm)
            ts.append(time.perf_counter())
            mm.close()
            ts.append(time.perf_counter())
            out = gather_rows(torch.from_numpy(t).cuda(), total) if world > 1 else t
            ts.append(time.perf_counter())
            if os.environ.get("XEE_TRACE"):
                print(f"[rank {rank}] e2e step: create {1e3*(ts[1]-ts[0]):.1f} run {1e3*(ts[2]-ts[1]):.1f} close {1e3*(ts[3]-ts[2]):.1f} gather {1e3*(ts[4]-ts[3]):.1f} ms", file=sys.stderr, flush=True)
            return out
        h2d, d2h = int(3 * NR * NZ * 4 + nloc * 40), int(nloc * (8 * 8 + 4 + 4 + 8 + 8))
        call = "EfficiencyMap(A,B,C host float32).run(heat host) -> table host (xee_map_create + xee_map_run_host + xee_map_destroy)"

    e2e = None
    if args.e2e_steps > 0:
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            out2 = e2e_step()
        barrier()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.e2e_steps
        e2e = {"value": total / (e2e_ms * 1e-3), "unit": "solves/s", "ms_per_step": e2e_ms, "steps": args.e2e_steps,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "call": call}
    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import oracle as O
        js, js_key = jacobi_sweeps_constant(args.workload)
        cores = O.max_threads()
        var = {}
        for name, sw in (("ref_O3", args.ref_sweeps), ("ref_O0", max(args.ref_sweeps // 8, 100)), ("fair", args.ref_sweeps)):
            r = cpu_sample(sw, cores, js or 1.0, name, args.workload)
            var[name] = {"point_sweeps_per_s": r["point_sweeps_per_s"], "solves_per_s": r["solves_per_s"] if js else None,
                         "sweeps_timed": sw, "seconds": r["seconds"]}
        var["ref_O3"]["what"] = "oracle literal restatement, reference loop order (stride-nx inner loop), 4 passes per sweep, g++ -O3"
        var["ref_O0"]["what"] = "the same code at -O0: what make-diagnosis.sh:10-11 builds (no optimisation flag)"
        var["fair"]["what"] = "fused passes, contiguous inner loop, planar operator: what a tuned CPU code would do per core"
        r = var["ref_O3"]
        cpu = {"value": r["solves_per_s"], "unit": "solves/s", "cores": cores, "kind": "port",
               "sample": f"{cores} solves x {r['sweeps_timed']} reference Jacobi sweeps (512x256 fp64, one solve per thread, {r['seconds']:.1f} s); "
                         f"extrapolated to {js:.0f} sweeps/solve (Jacobi to the bench tolerance, {js_key})" if js else "n/a",
               "point_sweeps_per_s": r["point_sweeps_per_s"], "extrapolated": True, "variants": var}
        if lfl:
            lfl.update({"cpu_point_sweeps_per_s": r["point_sweeps_per_s"], "cpu_variant": "ref_O3", "cpu_cores": cores,
                        "ratio": lfl["gpu_point_sweeps_per_s"] / r["point_sweeps_per_s"],
                        "ratio_vs_fair": lfl["gpu_point_sweeps_per_s"] / var["fair"]["point_sweeps_per_s"],
                        "what": "reference Jacobi point-sweeps/s on both sides, both measured, nothing extrapolated: the hardware factor"})
            if js:
                lfl["algorithmic_factor"] = js / float(tab[:, 0].mean())
    if rank == 0:
        line = {"metric": "elliptic_solves_per_sec", "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.total > 0 else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args, f"{args.method} ({args.arith} arithmetic)"),
                "roofline": roofline, "roofline_streaming_kernel": streaming, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                # the reference arm (--impl reference) runs the reference's plain Jacobi, extrapolated: not the same iteration
                "same_config": False,
                "same_config_note": "GPU arm: Chebyshev-accelerated (two-level) block-line relaxation to the same residual tolerance; reference arm: "
                                    "plain Jacobi (the reference's algorithm), a timed sample extrapolated to its sweep count; see like_for_like "
                                    "for the same-algorithm ratio",
                "like_for_like": lfl,
                "efficiency_range": eff_range,
                "solves_stopped_on_roundoff_floor": n_floor}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="map", choices=["map", "series"])
    ap.add_argument("--nheat", type=int, default=512, help="map: heating locations (independent solves) per GPU")
    ap.add_argument("--nsnap", type=int, default=128, help="series: snapshots (independent solves, one operator each) per GPU")
    ap.add_argument("--total", type=int, default=0, help="fix the TOTAL number of locations / snapshots (strong scaling); 0 = per-GPU count x GPUs")
    ap.add_argument("--method", default=None, choices=["chebyshev", "jacobi", "line_chebyshev", "line_jacobi", "line2_chebyshev"],
                    help="default: line2_chebyshev (two-level block-line Chebyshev), for both workloads")
    ap.add_argument("--check-step", type=int, default=0,
                    help="sweeps between residual checks (solve_elliptic's check_step); 0 = 100 for the point methods, 25 for the "
                         "line methods, which need ~4x fewer sweeps, 5 for the two-level method (a solve stops at the 2nd consecutive "
                         "check below r1)")
    ap.add_argument("--arith", default="fast", choices=["fast", "strict"])
    ap.add_argument("--max-iter", type=int, default=2000000)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--ref-sweeps", type=int, default=4000, help="Jacobi sweeps per solve in one CPU sample")
    ap.add_argument("--lfl-sweeps", type=int, default=300, help="GPU STRICT Jacobi sweeps timed for like_for_like")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-streaming", action="store_true", help="skip the extra one-level pass that reports the streaming kernel's roofline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's result table and a sample of its solution fields as DIR/<name>.npy")
    args = ap.parse_args()
    if args.method is None:
        args.method = "line2_chebyshev"
    if args.check_step <= 0:
        args.check_step = 5 if args.method.startswith("line2") else 25 if args.method.startswith("line") else 100
    args.per_gpu = args.nsnap if args.workload == "series" else args.nheat
    if args.total > 0:
        args.per_gpu = (args.total + max(args.gpus, 1) - 1) // max(args.gpus, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
