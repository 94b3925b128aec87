#!/usr/bin/env python
"""Throughput of the Laplace operator on a deformed mesh (pmg_laplace_operator_create_mapped) on one GPU.

  python tools/bench_mapped.py [--out DIR] [--reps R]      (--out: also write DIR/bench_mapped.json)

1. Degrees 2..6 on >= 30 M DoFs of a randomly distorted mesh (every interior vertex moved by up to 0.2 h per coordinate):
   the apply (vmult) and the fused Chebyshev step, in GDoF/s, with
   - the HBM fraction at the algorithmic bytes  16 + 48 (p+1)^3 / p^3  B/DoF (apply; + 16 for the step's b and x_old): the
     two vectors plus the six doubles of G_q per quadrature point;
   - the FP64 fraction at the algorithmic flops per DoF  (12 sweeps of 2 (p+1)^4 + 18 (p+1)^3 for G g) / p^3,  no recomputed
     halo cells;
   and beside both the variable-coefficient kernel (K1v: one double w a per point, 16 + 8 (p+1)^3 / p^3 B/DoF) at the same
   size and degree.  The fractions are over the copy bandwidth and the FMA rate measured by pmg_microbench in the same
   run (and the HBM fraction also over the data sheet's 7.7 TB/s).
2. One V-cycle and the CG solve (to 1e-12 ||b||) of the BASELINE config-2-shaped hierarchy Q4 -> Q2 -> Q1 -> h-levels on
   64^3 cells, on the mesh of the smooth map x -> x + 0.1 sin(pi x) sin(pi y) sin(pi z) (1, 1, 1) and undistorted.

Times: host clock around R repetitions closed by a device synchronise, after warm-up; every vector is larger than the L2.
The card's name and power limit are read in the same run.  Prints a table.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "portable-multigrid_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import pmg_b200 as G
from helpers import hierarchy_levels, splitmix_src
from mapped_mesh import random_vertices, smooth_map_vertices

HBM_DATASHEET_GBS = 7700.0
CELLS = {2: 156, 3: 104, 4: 78, 5: 63, 6: 52}  # n p + 1 >= 313: >= 30.6 M DoFs


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # the numbers are still measured; the card stays unnamed
        return "unknown (%s)" % e


def timed(ctx, f, reps):
    f()
    ctx.sync()
    t = time.perf_counter()
    for _ in range(reps):
        f()
    ctx.sync()
    return (time.perf_counter() - t) / reps


def kernel_rates(ctx, p, n, vertices, reps):
    coef = 0 if vertices is not None else 1
    op = G.LaplaceOperator(ctx, p, (n, n, n), coefficient=coef, vertices=vertices)
    m = op.m()
    op.compute_diagonal()
    u = op.vector_from(splitmix_src(m, salt=1))
    b, xo, d = op.vector_from(splitmix_src(m, salt=2)), op.vector_from(splitmix_src(m, salt=3)), op.initialize_dof_vector()
    t_apply = timed(ctx, lambda: op.vmult(d, u), reps)
    t_step = timed(ctx, lambda: op.chebyshev_step(d, u, xo, b, 0.3, 0.7), reps)
    del op, u, b, xo, d
    return m, t_apply, t_step


def solve(ctx, levels, vertices):
    ops, _, smoothers, mg = G.build_hierarchy(ctx, levels, vertices=vertices)
    for s in smoothers:
        s.info()  # eigenvalue estimates outside the timed parts
    top = ops[-1]
    b, x, z = top.initialize_dof_vector(), top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    for _ in range(3):  # eager, graph capture, replay
        mg.vmult(z, b)
    t_cycle = timed(ctx, lambda: mg.vmult(z, b), 10)
    x.set(0.0)
    ctx.sync()
    t = time.perf_counter()
    it, _, rc = G.cg_solve(top, x, b, mg)
    ctx.sync()
    t_cg = time.perf_counter() - t
    return dict(dofs=top.m(), vcycle_ms=t_cycle * 1e3, cg_ms=t_cg * 1e3, cg_iterations=it, rc=rc, norm=top.solution_norm(x))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    ctx = G.Context(0)
    res = dict(card=card(), microbench=ctx.microbench(), kernels=[], solves={})
    hbm, fma = res["microbench"]["hbm_copy_gbs"], res["microbench"]["fp64_fma_tflops"]
    print("card: %s; measured copy %.0f GB/s, FP64 FMA %.1f TFLOP/s" % (res["card"], hbm, fma))
    print("%2s %10s | %-44s | %-44s" % ("p", "DoFs", "mapped: apply / step GDoF/s (HBM%, FP64%)", "K1v: apply / step GDoF/s (HBM%)"))
    for p in range(2, 7):
        n = CELLS[p]
        r = (p + 1) ** 3 / p ** 3
        by_geo, by_var = 16 + 48 * r, 16 + 8 * r
        fl_geo = (24 * (p + 1) ** 4 + 18 * (p + 1) ** 3) / p ** 3
        m, ta, ts = kernel_rates(ctx, p, n, random_vertices((n,) * 3, 0.2, seed=p), a.reps)
        _, va, vs = kernel_rates(ctx, p, n, None, a.reps)
        row = dict(p=p, cells=n, dofs=m, bytes_per_dof_apply=by_geo, bytes_per_dof_step=by_geo + 16, flops_per_dof=fl_geo,
                   apply_gdofs=m / ta / 1e9, step_gdofs=m / ts / 1e9, k1v_apply_gdofs=m / va / 1e9, k1v_step_gdofs=m / vs / 1e9)
        for k, t, by in (("apply", ta, by_geo), ("step", ts, by_geo + 16)):
            row[k + "_hbm_frac_measured_copy"] = m * by / t / 1e9 / hbm
            row[k + "_hbm_frac_datasheet"] = m * by / t / 1e9 / HBM_DATASHEET_GBS
            row[k + "_fp64_frac_measured_fma"] = m * fl_geo / t / 1e12 / fma
        for k, t, by in (("k1v_apply", va, by_var), ("k1v_step", vs, by_var + 16)):
            row[k + "_hbm_frac_measured_copy"] = m * by / t / 1e9 / hbm
        res["kernels"].append(row)
        print("%2d %10d | %6.2f (%4.0f%%, %4.0f%%) / %6.2f (%4.0f%%, %4.0f%%)       | %6.2f (%4.0f%%) / %6.2f (%4.0f%%)" % (
            p, m, row["apply_gdofs"], 100 * row["apply_hbm_frac_measured_copy"], 100 * row["apply_fp64_frac_measured_fma"],
            row["step_gdofs"], 100 * row["step_hbm_frac_measured_copy"], 100 * row["step_fp64_frac_measured_fma"],
            row["k1v_apply_gdofs"], 100 * row["k1v_apply_hbm_frac_measured_copy"], row["k1v_step_gdofs"],
            100 * row["k1v_step_hbm_frac_measured_copy"]), flush=True)
    levels = hierarchy_levels("hp", 4, 64)
    for name, v in (("distorted", smooth_map_vertices((64,) * 3, 0.1)), ("undistorted", None)):
        res["solves"][name] = s = solve(ctx, levels, v)
        print("config-2 hierarchy %-11s: %d DoFs, V-cycle %.3f ms, CG %d iterations %.1f ms, ||u|| = %.10f" % (
            name, s["dofs"], s["vcycle_ms"], s["cg_iterations"], s["cg_ms"], s["norm"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_mapped.json"), "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
