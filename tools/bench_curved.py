#!/usr/bin/env python
"""Cost of curved cells (pmg_laplace_operator_create_curved, MappingQ(k)) against trilinear ones
(pmg_laplace_operator_create_mapped) on one GPU.

  python tools/bench_curved.py [--out DIR] [--reps R]      (--out: also write DIR/bench_curved.json)

1. Set-up: the time of create_curved(k = p) and of create_mapped (G_q of every quadrature point, validity check, inverse
   diagonal) at Q4 64^3 and Q2 128^3 cells, on the quarter cylindrical shell; the median of three creations each, the
   node / vertex arrays prepared beforehand.  Beside it the bytes of G (48 B per quadrature point) over the data sheet's
   7.7 TB/s, the least time writing G could take.
2. Apply: vmult of both operators, alternated in one loop (the same kernel K1g streams the same bytes, so expected equal).
3. A config-2-shaped shell solve: Q4 64^3, p 4 -> 2 -> 1 then h-levels, MappingQ(level degree) on every level: the
   hierarchy's set-up, its eigenvalue estimates, CG iterations (to 1e-12 ||b||), V-cycle and solve time, the norm's error.

Times: host clock around work closed by a device synchronise, after warm-up; every vector is larger than the L2.  The
card's name and power limit are read in the same run.
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
from curved_mesh import SHELL_FACES, SHELL_NORM, shell_map
from helpers import hierarchy_levels, splitmix_src

HBM_DATASHEET_GBS = 7700.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still measured; the card stays unnamed
        return "unknown (%s)" % e


def create_time(ctx, make):
    ts = []
    for _ in range(3):
        ctx.sync()
        t = time.perf_counter()
        op = make()
        ctx.sync()
        ts.append(time.perf_counter() - t)
        del op
    return float(np.median(ts))


def setup_and_apply(ctx, p, n, reps):
    nodes = G.mesh_nodes(shell_map, n, p)
    verts = G.mesh_nodes(shell_map, n, 1)
    t_cur = create_time(ctx, lambda: G.LaplaceOperator(ctx, p, n, SHELL_FACES, nodes=nodes))
    t_tri = create_time(ctx, lambda: G.LaplaceOperator(ctx, p, n, SHELL_FACES, vertices=verts))
    cur = G.LaplaceOperator(ctx, p, n, SHELL_FACES, nodes=nodes)
    tri = G.LaplaceOperator(ctx, p, n, SHELL_FACES, vertices=verts)
    m = cur.m()
    u = cur.vector_from(splitmix_src(m, salt=1))
    d = cur.initialize_dof_vector()
    for op in (cur, tri):  # warm-up
        op.vmult(d, u)
    ctx.sync()
    acc = {"curved": 0.0, "trilinear": 0.0}
    for _ in range(reps):
        for name, op in (("curved", cur), ("trilinear", tri)):
            ctx.sync()
            t = time.perf_counter()
            op.vmult(d, u)
            ctx.sync()
            acc[name] += time.perf_counter() - t
    nq = (n * (p + 1)) ** 3
    return dict(p=p, cells=n, dofs=m, create_curved_ms=t_cur * 1e3, create_mapped_ms=t_tri * 1e3,
                g_write_bound_ms=48.0 * nq / (HBM_DATASHEET_GBS * 1e9) * 1e3,
                apply_curved_ms=acc["curved"] / reps * 1e3, apply_mapped_ms=acc["trilinear"] / reps * 1e3)


def shell_solve(ctx):
    levels = hierarchy_levels("hp", 4, 64)
    ctx.sync()
    t = time.perf_counter()
    ops, _, smoothers, mg = G.build_hierarchy(ctx, levels, faces=SHELL_FACES, mapping=shell_map)
    ctx.sync()
    t_build = time.perf_counter() - t
    t = time.perf_counter()
    for s in smoothers:
        s.info()  # eigenvalue estimates
    ctx.sync()
    t_eig = time.perf_counter() - t
    top = ops[-1]
    b, x, z = top.initialize_dof_vector(), top.initialize_dof_vector(), top.initialize_dof_vector()
    top.assemble_rhs(b)
    for _ in range(3):  # eager, graph capture, replay
        mg.vmult(z, b)
    ctx.sync()
    t = time.perf_counter()
    for _ in range(10):
        mg.vmult(z, b)
    ctx.sync()
    t_cycle = (time.perf_counter() - t) / 10
    x.set(0.0)
    ctx.sync()
    t = time.perf_counter()
    it, _, rc = G.cg_solve(top, x, b, mg)
    ctx.sync()
    t_cg = time.perf_counter() - t
    norm = top.solution_norm(x)
    return dict(dofs=top.m(), hierarchy_setup_ms=t_build * 1e3, eigenvalue_estimates_ms=t_eig * 1e3, vcycle_ms=t_cycle * 1e3,
                cg_ms=t_cg * 1e3, cg_iterations=it, rc=rc, norm=norm, norm_rel_error=abs(norm - SHELL_NORM) / SHELL_NORM)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    ctx = G.Context(0)
    res = dict(card=card(), setup=[], shell=None)
    print("card: %s" % res["card"])
    print("%2s %5s %10s | %-38s | %-30s" % ("p", "cells", "DoFs", "create ms: curved(k=p) / mapped / G-write bound",
                                            "vmult ms: curved / mapped"))
    for p, n in ((4, 64), (2, 128)):
        r = setup_and_apply(ctx, p, n, a.reps)
        res["setup"].append(r)
        print("%2d %5d %10d | %9.2f / %9.2f / %9.3f         | %8.3f / %8.3f" % (
            p, n, r["dofs"], r["create_curved_ms"], r["create_mapped_ms"], r["g_write_bound_ms"], r["apply_curved_ms"],
            r["apply_mapped_ms"]), flush=True)
    res["shell"] = s = shell_solve(ctx)
    print("shell, config-2 hierarchy Q4 64^3 MappingQ(level degree): %d DoFs, set-up %.1f ms, eigenvalue estimates %.1f ms, "
          "V-cycle %.3f ms, CG %d iterations %.1f ms, ||u|| = %.12f, relative error %.2e" % (
              s["dofs"], s["hierarchy_setup_ms"], s["eigenvalue_estimates_ms"], s["vcycle_ms"], s["cg_iterations"], s["cg_ms"],
              s["norm"], s["norm_rel_error"]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_curved.json"), "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
