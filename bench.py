#!/usr/bin/env python
"""bench.py -- GDoF/s of the matrix-free multigrid hot path on B200.

A step = one V-cycle (VCycleMultigrid::vmult, reference include/multigrid/portable_v_cycle_multigrid.h:79-94)
on BASELINE.json configs[1]: 3-D Poisson, Q4, 64^3 cells (16 974 593 DoFs), polynomial multigrid
p = 4 -> 2 -> 1 followed by geometric levels down to one cell, V(2,2), Chebyshev(5)-Jacobi smoothing with
the reference drivers' parameters.  `value` = fine-level DoFs / device time per V-cycle, inputs resident in
HBM.  `e2e` = the same through the C-ABI's host-buffer entry (pmg_vcycle_vmult_host: H2D of the residual
from pinned memory, V-cycle, D2H of the correction).  `roofline` = the dominant kernel (the fused
Chebyshev step on the finest level) timed alone with CUDA events on the library's stream.
`--impl reference` times the reference's CPU algorithm (the oracle port: the reference itself cannot be
compiled here) on the host cores for the same metric and the same workload (the configuration's one-GPU mesh; by default
1 warm-up + 2 timed cycles, since one takes seconds).
`--dump-outputs DIR` writes the GPU V-cycle's output of the last timed step to DIR/vcycle_z.npy (float64; above DUMP_MAX
DoFs a fixed, seeded sample of them), so that two builds can be compared output for output on identical inputs.
The bench writes nothing into the source tree (it may be read-only): no bytecode, and the oracle for the CPU legs is
compiled into a temporary directory.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "portable-multigrid_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "GDoF/s of one multigrid V-cycle (fine-level DoFs / time); operator-apply GDoF/s in apply_gdofs"
UNIT = "GDoF/s"
DEGREE = 4
CELLS = 64
GPU_STEPS, GPU_WARMUP = 50, 5
REFERENCE_STEPS, REFERENCE_WARMUP = 2, 1  # the CPU arm: ~10-20 s per V-cycle at the flagship size
DUMP_MAX = 1 << 22  # values per dumped array: 32 MB of float64
DUMP_SEED = 0


def scaled_cells(n, world):
    """Weak scaling: per-GPU work fixed; cells doubled per direction z, y, x in turn."""
    c = [n, n, n]
    d, w = 2, world
    while w > 1:
        c[d] *= 2
        d = (d - 1) % 3
        w //= 2
    return tuple(c)


def hp_levels(p, cells):
    """(degree, (nx,ny,nz)) coarse -> fine: p -> p/2 -> .. -> 1 on the fine mesh, then geometric levels."""
    degs = [p]
    while degs[-1] > 1:
        degs.append(max(1, degs[-1] // 2))
    levels = [(d, tuple(cells)) for d in degs]
    c = list(cells)
    while all(x % 2 == 0 for x in c) and min(c) > 1:
        c = [x // 2 for x in c]
        levels.append((1, tuple(c)))
    return levels[::-1]


def h_levels(p, cells):
    """(degree, (nx,ny,nz)) coarse -> fine: the same degree on every level of the refinement hierarchy
    (reference geometric_multigrid driver)."""
    levels = [(p, tuple(cells))]
    c = list(cells)
    while all(x % 2 == 0 for x in c) and min(c) > 1:
        c = [x // 2 for x in c]
        levels.append((p, tuple(c)))
    return levels[::-1]


# BASELINE.json configs: "c2" = configs[1] (the one the metric is quoted on, default), "c1" = configs[0]; "c4" = configs[3]
# at its per-GPU size (Q3, 160^3 cells = 111 M DoFs per GPU, geometric hierarchy 5 .. 160 cells), "c5" = configs[4] at a
# single-GPU size (variable coefficient, Q5, 64^3 cells = 33 M DoFs per GPU; the named 160^3 cells need the 8-GPU box),
# p = 5 -> 2 -> 1 + geometric levels, CG to 1e-10
CONFIGS = {"c2": {"degree": 4, "cells": 64, "hierarchy": "hp", "cheb_degree": 5},
           "c1": {"degree": 2, "cells": 64, "hierarchy": "h", "cheb_degree": 3},
           "c4": {"degree": 3, "cells": 160, "hierarchy": "h", "cheb_degree": 5},
           "c5": {"degree": 5, "cells": 64, "hierarchy": "hp", "cheb_degree": 5, "coefficient": 1, "cg_tol": 1e-10}}


def workload_name(p, cells, world, hierarchy="hp", cheb_degree=5, coefficient=0):
    nd = 1
    for c in cells:
        nd *= c * p + 1
    degs = [p]
    while degs[-1] > 1:
        degs.append(max(1, degs[-1] // 2))
    hier = ("hp-multigrid p=%s + geometric levels" % "->".join(str(d) for d in degs)) if hierarchy == "hp" else "geometric multigrid, Q%d on every level" % p
    if coefficient:
        hier = "variable coefficient a = 1/(0.05 + 2|x|^2), " + hier
    return ("3D Poisson Q%d, %dx%dx%d cells (%d DoFs), %s, V(2,2) Chebyshev(%d)-Jacobi, one V-cycle per step"
            % (p, cells[0], cells[1], cells[2], nd, hier, cheb_degree)), nd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the GPU is under load."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu summary, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_cheb_step_q4_c2.json")) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


def load_oracle():
    """The oracle compiled into a temporary directory (the source tree may be read-only): -march=native, or, where that
    does not compile, the portable build.  Returns (module, kind)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as O

    with tempfile.TemporaryDirectory() as tmp:  # the library is loaded before the directory goes
        try:
            O.use_library(O.build(native=True, out_dir=tmp))
            return O, "port (-march=native)"
        except Exception:
            O.use_library(O.build(out_dir=tmp))
            return O, "port"


def dump_outputs(out_dir, name, v):
    """DIR/<name>.npy: v as float64, or, above DUMP_MAX entries, its entries at DUMP_MAX fixed, seeded, sorted indices."""
    if v.size > DUMP_MAX:
        v = v[np.sort(np.random.default_rng(DUMP_SEED).choice(v.size, DUMP_MAX, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v, dtype=np.float64))


def run_reference(args, cfg):
    """CPU arm: the oracle's V-cycle (port of the reference algorithm in the reference's data layout) on all host threads,
    on the SAME workload as the product arm at one GPU -- the configuration's own mesh and hierarchy (64^3 cells Q4 for c2:
    3.7 GB of stored indices / Jacobians, ~10-20 s per V-cycle), so by default 1 warm-up and 2 timed cycles (REFERENCE_STEPS,
    REFERENCE_WARMUP; --steps / --warmup as given otherwise).  Under torchrun the product arm weak-scales the mesh; this arm keeps the one-GPU mesh (the CPU's throughput
    does not depend on the size beyond its caches) and `config.workload` names what it ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers; this arm is meant to use all the host threads it can
    if "LOCAL_RANK" in os.environ or os.environ.get("OMP_NUM_THREADS") == "1":
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    O, kind = load_oracle()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    res = cpu_vcycle(O, cfg, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": res["steps"], "warmup": res["warmup"], "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": res["workload"], "timing": "host wall clock around the oracle's V-cycle",
                   "note": None if world == 1 else "the product arm runs this mesh per GPU, weak-scaled over %d GPUs" % world},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": "port", "sample": res["sample"], "build": kind},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "apply_gdofs": res["apply_gdofs"],
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_vcycle(O, cfg, steps, warmup):
    """The oracle's V-cycle on the configuration's one-GPU mesh: `warmup` untimed + `steps` timed cycles."""
    from helpers import splitmix_src

    p, cells = cfg["degree"], (cfg["cells"],) * 3
    coef = cfg.get("coefficient", 0)
    levels = hp_levels(p, cells) if cfg["hierarchy"] == "hp" else h_levels(p, cells)
    mfs = [O.MatrixFree(3, d, c, coef=("c5" if coef else None)) for (d, c) in levels]
    trs = [O.Transfer(mfs[l - 1], mfs[l], "h" if levels[l][0] == levels[l - 1][0] else "p") for l in range(1, len(levels))]
    vc = O.VCycle(mfs, trs, degree=cfg["cheb_degree"])
    vc.estimate()
    n = mfs[-1].n_dofs
    r = splitmix_src(n, mfs[-1].constrained())
    for _ in range(warmup):
        vc.vmult(r)
    t0 = time.perf_counter()
    for _ in range(steps):
        vc.vmult(r)
    dt = (time.perf_counter() - t0) / steps
    t0 = time.perf_counter()
    for _ in range(2):
        mfs[-1].vmult(r)
    dta = (time.perf_counter() - t0) / 2
    name, _ = workload_name(p, cells, 1, cfg["hierarchy"], cfg["cheb_degree"], coef)
    return {"value": n / dt / 1e9, "ms_per_step": dt * 1e3, "cores": O.num_threads(), "apply_gdofs": n / dta / 1e9,
            "steps": steps, "warmup": warmup, "workload": name,
            "sample": "the full workload (%d DoFs), %d warm-up + %d timed V-cycles; reference data layout "
                      "(stored indices, masks, per-q-point Jacobians)" % (n, warmup, steps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed V-cycles (default %d; %d with --impl reference)" % (GPU_STEPS, REFERENCE_STEPS))
    ap.add_argument("--warmup", type=int, default=None,
                    help="untimed V-cycles before them (default %d, at least 3 on the GPU: eager, capture, replay; "
                         "%d with --impl reference)" % (GPU_WARMUP, REFERENCE_WARMUP))
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json workload (default: the one the metric is quoted on)")
    ap.add_argument("--degree", type=int, default=None)
    ap.add_argument("--cells", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the GPU V-cycle's output of the last timed step to DIR/vcycle_z.npy")
    args = ap.parse_args()
    reference = args.impl == "reference"
    if args.steps is None:
        args.steps = REFERENCE_STEPS if reference else GPU_STEPS
    if args.warmup is None:
        args.warmup = REFERENCE_WARMUP if reference else GPU_WARMUP
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if reference and args.dump_outputs:
        # the CPU arm runs its own residual (zero on Dirichlet DoFs): nothing it computes is comparable with a GPU dump
        ap.error("--dump-outputs writes the GPU path's output; it does not apply to --impl reference")
    cfg = dict(CONFIGS[args.config])
    if args.degree is not None:
        cfg["degree"] = args.degree
    if args.cells is not None:
        cfg["cells"] = args.cells
    if reference:
        return run_reference(args, cfg)

    import torch
    import pmg_b200 as G
    from helpers import splitmix_src

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    nccl_id = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        obj = [G.Context.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        nccl_id = obj[0]
    ctx = G.Context(local, rank, world, nccl_id)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    p = cfg["degree"]
    cells = scaled_cells(cfg["cells"], world)
    levels = hp_levels(p, cells) if cfg["hierarchy"] == "hp" else h_levels(p, cells)
    coefficient = cfg.get("coefficient", 0)
    name, n_dofs = workload_name(p, cells, world, cfg["hierarchy"], cfg["cheb_degree"], coefficient)
    ops, transfers, smoothers, mg = G.build_hierarchy(ctx, levels, degree=cfg["cheb_degree"], coefficient=coefficient)
    top = ops[-1]
    r_host = splitmix_src(n_dofs)
    r, z = top.vector_from(r_host), top.initialize_dof_vector()
    for s in smoothers:
        s.info()  # eigenvalue estimates outside the timed region (setup, as in the reference's first vmult)

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        ctx.sync()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / k)

    # kernels per V-cycle, counted on an eager (non-graph) cycle
    mg.set_graph(False)
    c0 = ctx.launch_count()
    mg.vmult(z, r)
    ctx.sync()
    launches_per_cycle = ctx.launch_count() - c0
    mg.set_graph(True)
    for _ in range(max(args.warmup, 3)):
        mg.vmult(z, r)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(lambda: mg.vmult(z, r), args.steps)
    value = n_dofs / (ms * 1e-3) / 1e9
    if args.dump_outputs:
        z_host = z.export_host()  # now: the measurements below reuse z; with several ranks a collective gather
        if rank == 0:
            dump_outputs(args.dump_outputs, "vcycle_z", z_host)
        del z_host

    # operator apply alone (LaplaceOperator::vmult), and the dominant kernel of the cycle
    u, b, xo = top.vector_from(splitmix_src(n_dofs, salt=1)), top.vector_from(splitmix_src(n_dofs, salt=2)), top.initialize_dof_vector()
    for _ in range(3):
        top.vmult(z, u)
    ms_apply = timed(lambda: top.vmult(z, u), 20)
    for _ in range(3):
        top.chebyshev_step(xo, u, xo, b, 0.3, 0.1)
    ms_step = timed(lambda: top.chebyshev_step(xo, u, xo, b, 0.3, 0.1), 20)

    # the drivers' solve (program.cc:345-355): CG preconditioned by one V-cycle, to 1e-12 ||b||, on the load vector of f = 1
    rhs, sol = top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(rhs)
    cg_tol = cfg.get("cg_tol", 1e-12)
    G.cg_solve(top, sol, rhs, mg, rel_tol=cg_tol)  # warm-up (also leaves the graph captured)
    sol.set(0.0)
    barrier()
    t0 = time.perf_counter()
    cg_it, cg_hist, cg_rc = G.cg_solve(top, sol, rhs, mg, rel_tol=cg_tol)
    ctx.sync()
    cg_s = max_over_ranks(time.perf_counter() - t0)
    cg = {"iterations": int(cg_it), "converged": cg_rc == 0, "ms": cg_s * 1e3, "gdofs_x_iterations_per_s": n_dofs * max(cg_it, 1) / cg_s / 1e9,
          "final_relative_residual": float(cg_hist[-1] / cg_hist[0]) if len(cg_hist) and cg_hist[0] > 0 else None}

    # end to end through the host-buffer entry point: pinned host memory, H2D + V-cycle + D2H every step
    n_local_bytes = n_dofs * 8
    e2e = None
    if world == 1:
        src_pin = torch.from_numpy(r_host).pin_memory()
        dst_pin = torch.empty(n_dofs, dtype=torch.float64).pin_memory()
        for _ in range(2):
            mg.vmult_host(dst_pin.data_ptr(), src_pin.data_ptr())
        k = max(3, min(args.steps, 10))
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            mg.vmult_host(dst_pin.data_ptr(), src_pin.data_ptr())  # returns after the D2H copy completed
        dt = (time.perf_counter() - t0) / k
        e2e = {"value": n_dofs / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": n_local_bytes, "d2h_bytes_per_step": n_local_bytes,
               "ms_per_step": dt * 1e3, "checksum": float(dst_pin.double().abs().sum())}
    else:
        # distributed: every rank uploads the owned part of the residual from pinned memory and downloads the owned part of the
        # correction (pmg_vcycle_vmult_host_owned: no collective outside the V-cycle, no global vector on any rank)
        tmpv = top.initialize_dof_vector()
        plane, z0l, nzl_, zlo, zhi = tmpv.local_range()
        del tmpv
        n_own = plane * (zhi - zlo)
        src_pin = torch.from_numpy(np.ascontiguousarray(r_host[zlo * plane:zhi * plane])).pin_memory()
        dst_pin = torch.empty(n_own, dtype=torch.float64).pin_memory()
        for _ in range(2):
            mg.vmult_host_owned(dst_pin.data_ptr(), src_pin.data_ptr())
        k = max(3, min(args.steps, 10))
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            mg.vmult_host_owned(dst_pin.data_ptr(), src_pin.data_ptr())
        dt = max_over_ranks((time.perf_counter() - t0) / k)
        e2e = {"value": n_dofs / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(n_own * 8), "d2h_bytes_per_step": int(n_own * 8),
               "ms_per_step": dt * 1e3, "note": "per rank: its owned slab, pinned host buffers"}
    clocks = sampler.stop() if rank == 0 else None
    # one eager V-cycle with event marks between its phases: device ms per level on this rank (smoother / transfer / ghost
    # exchange / residual + copies) -- the breakdown BASELINE configs[4] asks for; outside every timed region
    per_level = None
    try:
        barrier()
        mg.profile(z, r)  # first eager cycle after the graph replays: absorbs one-off host-side delays and rank skew
        barrier()
        f0 = ctx.fused_halo_count()
        prof = mg.profile(z, r)
        per_level = {"columns": ["smoother", "transfer", "ghost_exchange", "residual_and_copies"],
                     "ms": [[round(float(x), 4) for x in row] for row in prof],
                     "applies_without_exchange": int(ctx.fused_halo_count() - f0),
                     "note": "rank 0, eager launches (the timed cycles replay a CUDA graph); row l = level l of config.levels"}
    except Exception as e:  # never fatal for the bench line
        per_level = {"error": str(e)}

    peak, peak_src = measured_peaks()
    n_local = n_dofs / world
    # fused Chebyshev step: read u, x_old, b; write x_new (Dinv is a table); variable coefficient: + Dinv vector + one
    # coefficient per quadrature point (SURVEY 8d)
    bytes_per_dof = 32.0 + ((8.0 + 8.0 * (p + 1) ** 3 / p ** 3) if coefficient else 0.0)
    algo_bytes = bytes_per_dof * n_local
    achieved = algo_bytes / (ms_step * 1e-3) / 1e9
    n1 = p + 1
    # FP64 work per DoF (DESIGN.md, kernel K1): the kernel executes 7 one-dimensional sweeps of (p+1)^2 / p FMAs per DoF
    # plus the epilogue; the reference's cell loop needs [24 (p+1)^4 + 39 (p+1)^3] / p^3 flops per DoF (SURVEY 8d)
    flops_per_dof = (2.0 * 7.0 * n1 * n1 / p + 8.0) if not coefficient else (2.0 * 12.0 * n1 ** 4 / p ** 3 + 8.0)
    ref_flops_per_dof = (24.0 * n1 ** 4 + 39.0 * n1 ** 3) / p ** 3
    fp64 = None
    try:
        mb = ctx.microbench() if rank == 0 else None
    except Exception:
        mb = None
    if mb:
        fl = flops_per_dof * n_local
        fp64 = {"flops_per_launch": fl, "achieved_tflops": fl / (ms_step * 1e-3) / 1e12, "peak_fma_tflops": mb["fp64_fma_tflops"],
                "peak_dmma_tflops": mb["fp64_dmma_tflops"], "frac": fl / (ms_step * 1e-3) / 1e12 / mb["fp64_fma_tflops"],
                "reference_algorithm_flops_per_launch": ref_flops_per_dof * n_local,
                "frac_if_counted_as_reference_flops": ref_flops_per_dof * n_local / (ms_step * 1e-3) / 1e12 / mb["fp64_fma_tflops"],
                "hbm_copy_gbs_here": mb["hbm_copy_gbs"],
                "note": "executed flops of owned DoFs (7 sweeps + epilogue); halo recompute not counted"}

    # BASELINE configs[2] point of this degree (standalone apply on a ~100 M-DoF cube, SURVEY 8 "C3"): the same operator call on
    # n = round(464 / p) cells per direction.  Last GPU work of the run and never a dependency of the line above.
    apply_c3, apply_c3_sweep = None, None
    if world == 1 and args.config == "c2" and not coefficient:
        # BASELINE configs[2]: the degree 1..9 sweep of the standalone apply at ~100 M DoFs, with both rooflines per degree --
        # HBM (16 B/DoF at the measured copy bandwidth) and FP64 (the 7 one-dimensional band-matrix sweeps of p + 2 FMAs per
        # DoF at the measured DFMA rate) -- and the degree where the FP64 roof drops below the HBM roof (the "crossover").
        fma_peak = mb["fp64_fma_tflops"] if mb else None
        sweep = []
        for q in range(1, 10):
            try:
                n3 = int(round(464.0 / q))
                big = G.LaplaceOperator(ctx, q, n3)
                ub, zb = big.initialize_dof_vector(), big.initialize_dof_vector()
                ub.set(1.0)
                for _ in range(3):
                    big.vmult(zb, ub)
                ms_big = timed(lambda: big.vmult(zb, ub), 5)
                nb = int(big.m())
                gd = nb / (ms_big * 1e-3) / 1e9
                ent = {"degree": q, "cells_per_dir": n3, "n_dofs": nb, "ms": ms_big, "gdofs": gd, "hbm_frac": 16.0 * gd / peak,
                       "kernel": "pmg_plane_kernel" if q <= 6 else "pmg_sweep_kernel", "hbm_roof_gdofs": peak / 16.0}
                if fma_peak:
                    fma_per_dof = 7.0 * (q + 2)
                    ent["fp64_roof_gdofs"] = fma_peak * 1e3 / (2.0 * fma_per_dof)
                    ent["fp64_frac"] = gd / ent["fp64_roof_gdofs"]
                    ent["binding_roof"] = "hbm" if ent["hbm_roof_gdofs"] <= ent["fp64_roof_gdofs"] else "fp64"
                sweep.append(ent)
                del ub, zb, big
            except Exception as e:
                sweep.append({"degree": q, "error": repr(e)})
        cross = [e["degree"] for e in sweep if e.get("binding_roof") == "fp64"]
        apply_c3_sweep = {"points": sweep, "fp64_fma_per_dof": "7 (p + 2)", "crossover_degree": min(cross) if cross else None,
                          "note": "from crossover_degree on the FP64 roof of the formulation is below the HBM roof; DMMA has the same peak as DFMA on B200 (fp64 block)"}
        apply_c3 = next((e for e in sweep if e.get("degree") == p and "gdofs" in e), None)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": name, "levels": [[d, list(c)] for d, c in levels], "cache": "inputs larger than L2 (3-4 fine vectors of %.0f MB each)" % (n_local_bytes / world / 1e6),
                   "parallelism": "z-slabs x%d" % world, "cuda_graph": True},
        "apply_gdofs": n_dofs / (ms_apply * 1e-3) / 1e9, "apply_ms": ms_apply,
        "apply_hbm_frac": 16.0 * n_local / (ms_apply * 1e-3) / 1e9 / peak,
        "apply_c3": apply_c3, "apply_c3_sweep": apply_c3_sweep,
        "cg_solve": cg,
        "e2e": e2e, "gpu_launches": int(launches_per_cycle * args.steps), "launches_per_cycle": int(launches_per_cycle),
        "clocks": clocks, "per_level_ms": per_level,
        "roofline": {"kernel": ("pmg_var_kernel<%d>" if coefficient else "pmg_plane_kernel<%d>" if p <= 6 else "pmg_sweep_kernel<%d>") % p + " (fused Chebyshev step, finest level)",
                     "bound": "hbm", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic() if args.config == "c2" and world == 1 else None,
                     "peak_source": peak_src, "algorithmic_bytes_per_dof": bytes_per_dof, "ms_per_launch": ms_step, "fp64": fp64},
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            O, _ = load_oracle()
            res = cpu_vcycle(O, cfg, steps=1, warmup=1)
            line["cpu_baseline"] = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": "port", "sample": res["sample"],
                                    "apply_gdofs": res["apply_gdofs"]}
        except Exception as e:  # the baseline is a reported number, never a dependency of the product path
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
