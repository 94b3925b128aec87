#!/usr/bin/env python
"""Multi-GPU parity of the problem-data entries (run under torchrun, one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/dist_check_problem_data.py
On z-slabs of the box and of the quarter cylindrical shell (MappingQ(p) and trilinear cells), every rank's stored planes --
ghost planes included -- of support_points, assemble_rhs_data(f, g) and distribute must equal the single-GPU result of rank 0
(an operator on a one-rank context on the same device) to 1e-14; then a manufactured shell solve (radial u*, CG + V-cycle,
distribute) must match the single-GPU solve: the same iteration count and the solution to 1e-10."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "portable-multigrid_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist
import pmg_b200 as G
from helpers import hierarchy_levels, splitmix_src
from curved_mesh import SHELL_FACES, shell_map


def radial(x, y, z):
    r = np.hypot(x, y)
    return r * r + np.sin(np.pi * r), -4.0 + np.pi ** 2 * np.sin(np.pi * r) - np.pi * np.cos(np.pi * r) / r


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    obj = [G.Context.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    ctx = G.Context(local, rank, world, obj[0])
    ctx.set_coarse_threshold(2000)
    one = G.Context(local)  # the single-GPU reference, on every rank (each compares its own stored planes)
    ok = True

    def report(name, err, tol):
        nonlocal ok
        errs = [None] * world
        dist.all_gather_object(errs, float(err))
        if rank == 0:
            print("%-52s %.3e %s" % (name, max(errs), "ok" if max(errs) <= tol else "FAIL"), flush=True)
        ok = ok and max(errs) <= tol

    def local_of(vec_one, like):
        pl, z0, nz, _, _ = like.local_range()
        return vec_one.export_host()[pl * z0: pl * (z0 + nz)]

    p, n = 3, 4 * world
    cases = [("box", dict(dirichlet_faces=0x15)),
             ("shell MappingQ(3)", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, p))),
             ("shell trilinear", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, 1), geometry_degree=1))]
    for name, kw in cases:
        op, ref = G.LaplaceOperator(ctx, p, n, **kw), G.LaplaceOperator(one, p, n, **kw)
        P, Pr = op.support_points(), ref.support_points()  # export_host: the full vectors
        report(name + ": support points (full)", np.abs(P - Pr).max(), 1e-14)
        xs = [op.initialize_dof_vector() for _ in range(3)]
        G.lib().pmg_laplace_operator_support_points(op.h, xs[0].h, xs[1].h, xs[2].h)
        xr = [ref.initialize_dof_vector() for _ in range(3)]
        G.lib().pmg_laplace_operator_support_points(ref.h, xr[0].h, xr[1].h, xr[2].h)
        report(name + ": support points (stored planes)",
               max(np.abs(a.export_local() - local_of(b, a)).max() for a, b in zip(xs, xr)), 1e-14)
        m = op.m()
        f, g = splitmix_src(m, salt=31), splitmix_src(m, salt=32)
        b, br = op.initialize_dof_vector(), ref.initialize_dof_vector()
        op.assemble_rhs_data(b, f=op.vector_from(f), g=op.vector_from(g))
        ref.assemble_rhs_data(br, f=ref.vector_from(f), g=ref.vector_from(g))
        scale = np.abs(br.export_host()).max()
        report(name + ": assemble_rhs_data (stored planes)", np.abs(b.export_local() - local_of(br, b)).max() / scale, 1e-14)
        u, ur = op.vector_from(f), ref.vector_from(f)
        op.distribute(u, op.vector_from(g))
        ref.distribute(ur, ref.vector_from(g))
        report(name + ": distribute (stored planes)", np.abs(u.export_local() - local_of(ur, u)).max(), 0.0)

    levels = hierarchy_levels("h", p, n)
    results = []
    for c in (ctx, one):
        ops, _, _, mg = G.build_hierarchy(c, levels, faces=SHELL_FACES, mapping=shell_map)
        top = ops[-1]
        vu, vf = top.interpolate(lambda x, y, z: radial(x, y, z)[0]), top.interpolate(lambda x, y, z: radial(x, y, z)[1])
        b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
        top.assemble_rhs_data(b, f=vf, g=vu)
        it, _, rc = G.cg_solve(top, x, b, mg)
        top.distribute(x, vu)
        vu.sadd(-1.0, 1.0, x)
        results.append((it, rc, x.export_host(), top.solution_norm(vu)))
        del ops, mg, top, vu, vf, b, x
    (it, rc, x, err), (it1, rc1, x1, err1) = results
    report("shell solve: CG iterations %d vs %d" % (it, it1), float(abs(it - it1) + abs(rc) + abs(rc1)), 0.0)
    report("shell solve: solution", np.abs(x - x1).max(), 1e-10)
    report("shell solve: ||u_h - I_h u*|| %.6e vs %.6e" % (err, err1), abs(err - err1) / err1, 1e-8)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DIST CHECK PASSED" if flag.item() == 1 else "DIST CHECK FAILED", flush=True)
    ctx.close()
    one.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
