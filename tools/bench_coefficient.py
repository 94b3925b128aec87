#!/usr/bin/env python
"""Cost of the coefficient from the caller on one GPU.

  python tools/bench_coefficient.py [--out DIR] [--reps R]      (--out: also write DIR/bench_coefficient.json)

- set_coefficient (upload of a, check, refill of the per-point data, inverse diagonal) at Q4 on 64^3 cells, on the unit cube
  (box operator: the w a grid, 32.8 M points, 262 MB) and on the quarter cylindrical shell with MappingQ(4) cells (six G
  grids, 1.6 GB): host wall time around the call, which ends in a device synchronise, median of R calls after a warm-up.
- The 2-D apply and V-cycle at the polynomial driver's size (Q7, 64^2 cells, 201 601 DoFs, seven p-levels) with a caller
  coefficient (the two-pass kernel of csrc/pmg_dim2_var.h) against the constant-coefficient 2-D kernel: device time by CUDA
  events on the context's stream, median of R x 100 calls.  These sizes live in L2: the times are launch- and
  latency-bound, which is what that driver runs.
- A 3-D V-cycle (Q4, h-hierarchy to 64^3 cells) with a caller coefficient against coefficient 1: the same kernels, so the
  same time is expected.
The card's name and power limit are read in the same run.
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
import torch
import pmg_b200 as G
from curved_mesh import SHELL_FACES, shell_map
from helpers import hierarchy_levels, splitmix_src


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers are still measured; the card stays unnamed
        return "unknown (%s)" % e


def device_ms(ctx, fn, reps, inner=1):
    """median device time of one fn() in ms: CUDA events on the context's stream around `inner` calls, after a warm-up"""
    stream = torch.cuda.ExternalStream(ctx.stream())
    fn()
    ctx.sync()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(inner):
            fn()
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b) / inner)
    return float(np.median(ts))


def wall_ms(ctx, fn, reps):
    fn()
    ctx.sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ctx.sync()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts))


def jump(*X):
    P = np.stack(X, axis=1)
    return np.where(np.all((P >= 0.25) & (P <= 0.75), axis=1), 100.0, 1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    torch.cuda.init()
    ctx = G.Context(0)
    res = dict(card=card())
    # set_coefficient, Q4 64^3
    p, n = 4, 64
    for name, kw in (("box", dict()), ("shell", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, p)))):
        op = G.LaplaceOperator(ctx, p, n, coefficient=G.PMG_COEFFICIENT_CALLER, **kw)
        vals = op.evaluate_at_quadrature_points(lambda x, y, z: 1.0 + 99.0 * (np.hypot(x, y) < 1.5))
        res["set_coefficient_%s_q4_64_ms" % name] = wall_ms(ctx, lambda: op.set_coefficient(vals), a.reps)
        res["quadrature_points_%s_q4_64_ms" % name] = wall_ms(ctx, op.quadrature_points, a.reps)
        print("set_coefficient %-5s Q4 64^3 (%d points): %.2f ms; quadrature_points %.2f ms" % (
            name, len(vals), res["set_coefficient_%s_q4_64_ms" % name], res["quadrature_points_%s_q4_64_ms" % name]), flush=True)
        del op, vals
    # 2-D, the polynomial driver's hierarchy
    levels2 = [(q, 64) for q in range(1, 8)]
    for name, coef in (("constant", 0), ("caller", jump)):
        ops, _, _, mg = G.build_hierarchy(ctx, levels2, dim=2, faces=0xF, coefficient=coef)
        top = ops[-1]
        u, d = top.vector_from(splitmix_src(top.m(), salt=1)), top.initialize_dof_vector()
        b = top.vector_from(splitmix_src(top.m(), salt=2))
        res["dim2_q7_64_apply_%s_us" % name] = 1e3 * device_ms(ctx, lambda: top.vmult(d, u), a.reps, 100)
        res["dim2_q7_64_cheb_step_%s_us" % name] = 1e3 * device_ms(ctx, lambda: top.chebyshev_step(d, u, None, b, 0.3, 0.7), a.reps, 100)
        res["dim2_q7_64_vcycle_%s_us" % name] = 1e3 * device_ms(ctx, lambda: mg.vmult(d, b), a.reps, 20)
        print("2-D Q7 64^2 %-8s: apply %.2f us, Chebyshev step %.2f us, V-cycle %.1f us" % (
            name, res["dim2_q7_64_apply_%s_us" % name], res["dim2_q7_64_cheb_step_%s_us" % name],
            res["dim2_q7_64_vcycle_%s_us" % name]), flush=True)
        del ops, mg, top, u, d, b
    # 3-D V-cycle: caller coefficient vs coefficient 1
    levels3 = hierarchy_levels("h", 4, 64)
    c5 = lambda x, y, z: 1.0 / (0.05 + 2.0 * (x * x + y * y + z * z))  # noqa: E731
    for name, coef in (("coefficient1", 1), ("caller", c5)):
        ops, _, _, mg = G.build_hierarchy(ctx, levels3, coefficient=coef)
        top = ops[-1]
        d, b = top.initialize_dof_vector(), top.vector_from(splitmix_src(top.m(), salt=3))
        res["dim3_q4_64_vcycle_%s_ms" % name] = device_ms(ctx, lambda: mg.vmult(d, b), a.reps, 5)
        print("3-D Q4 64^3 V-cycle %-12s: %.3f ms" % (name, res["dim3_q4_64_vcycle_%s_ms" % name]), flush=True)
        del ops, mg, top, d, b
    print("card: %s" % res["card"])
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_coefficient.json"), "w") as fh:
            json.dump(res, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
