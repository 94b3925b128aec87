#!/usr/bin/env python
"""Set-up cost of the problem-data entries on one GPU.

  python tools/bench_problem_data.py [--out DIR] [--reps R]      (--out: also write DIR/bench_problem_data.json)

At Q4 on 64^3 cells, on the unit cube (box operator) and on the quarter cylindrical shell with MappingQ(4) cells: the device
time of support_points, assemble_rhs_data(f, g) and assemble_rhs (f = 1), each the median of R calls bracketed by CUDA
events on the context's stream after one warm-up call.  Every vector (17.0 M DoFs, 136 MB) and the shell's w |det J| grid
(32.8 M points, 262 MB) exceed the 126 MB L2.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "portable-multigrid_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import pmg_b200 as G
from curved_mesh import SHELL_FACES, shell_map
from helpers import splitmix_src


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still measured; the card stays unnamed
        return "unknown (%s)" % e


def device_ms(ctx, fn, reps):
    """median device time of fn() in ms: CUDA events recorded on the context's stream around each call, after a warm-up"""
    stream = torch.cuda.ExternalStream(ctx.stream())
    fn()
    ctx.sync()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--degree", type=int, default=4)
    ap.add_argument("--cells", type=int, default=64)
    a = ap.parse_args()
    p, n = a.degree, a.cells
    torch.cuda.init()
    ctx = G.Context(0)
    res = dict(card=card(), degree=p, cells=n)
    for name, kw in (("box", dict()), ("shell", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, p)))):
        op = G.LaplaceOperator(ctx, p, n, **kw)
        m = op.m()
        x, y, z = (op.initialize_dof_vector() for _ in range(3))
        f, g = op.vector_from(splitmix_src(m, salt=1)), op.vector_from(splitmix_src(m, salt=2))
        rhs = op.initialize_dof_vector()
        lib = G.lib()
        r = dict(dofs=m)
        r["support_points_ms"] = device_ms(ctx, lambda: lib.pmg_laplace_operator_support_points(op.h, x.h, y.h, z.h), a.reps)
        r["assemble_rhs_data_f_g_ms"] = device_ms(ctx, lambda: op.assemble_rhs_data(rhs, f=f, g=g), a.reps)
        r["assemble_rhs_data_f_ms"] = device_ms(ctx, lambda: op.assemble_rhs_data(rhs, f=f), a.reps)
        r["assemble_rhs_ms"] = device_ms(ctx, lambda: op.assemble_rhs(rhs), a.reps)
        res[name] = r
        print("%-6s Q%d %d^3 cells, %d DoFs: support_points %.3f ms, assemble_rhs_data(f, g) %.3f ms, (f) %.3f ms, "
              "assemble_rhs %.3f ms" % (name, p, n, m, r["support_points_ms"], r["assemble_rhs_data_f_g_ms"],
                                        r["assemble_rhs_data_f_ms"], r["assemble_rhs_ms"]), flush=True)
        del op, x, y, z, f, g, rhs
    print("card: %s" % res["card"])
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_problem_data.json"), "w") as fh:
            json.dump(res, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
