#!/usr/bin/env python
"""Multi-GPU parity of the coefficient from the caller (run under torchrun, one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/dist_check_coefficient.py
On z-slabs of the box, of the trilinear and of the MappingQ(3) quarter cylindrical shell, every rank evaluates a jump
coefficient at its own quadrature_points() -- the halo cell layer below its owned layers included -- and sets it.  Each
rank's points must equal the single-GPU points of the same q-planes bit for bit; the apply and the inverse diagonal must
equal the single-GPU operator's (an operator on a one-rank context on the same device) to 1e-14; then a CG + V-cycle solve
must match the single-GPU solve: the same iteration count and the solution to 1e-10."""
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


def jump(x, y, z):
    return np.where(np.hypot(x, y) < 1.5, 100.0, 1.0) * np.where((z > 0.3) & (z < 0.6), 3.0, 1.0)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    obj = [G.Context.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    ctx = G.Context(local, rank, world, obj[0])
    ctx.set_coarse_threshold(2000)
    one = G.Context(local)
    ok = True

    def report(name, err, tol):
        nonlocal ok
        errs = [None] * world
        dist.all_gather_object(errs, float(err))
        if rank == 0:
            print("%-56s %.3e %s" % (name, max(errs), "ok" if max(errs) <= tol else "FAIL"), flush=True)
        ok = ok and max(errs) <= tol

    def local_of(vec_one, like):
        pl, z0, nz, _, _ = like.local_range()
        return vec_one.export_host()[pl * z0: pl * (z0 + nz)]

    p, n = 3, 4 * world
    cases = [("box", dict(dirichlet_faces=0x15)),
             ("trilinear shell", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, 1), geometry_degree=1)),
             ("shell MappingQ(3)", dict(dirichlet_faces=SHELL_FACES, nodes=G.mesh_nodes(shell_map, n, p)))]
    for name, kw in cases:
        op = G.LaplaceOperator(ctx, p, n, coefficient=jump, **kw)
        ref = G.LaplaceOperator(one, p, n, coefficient=jump, **kw)
        qx, qy, qz0, nqz = op.quadrature_grid()
        P, Pr = op.quadrature_points(), ref.quadrature_points()
        report(name + ": points of the stored q-planes (bits)", np.abs(P - Pr[qx * qy * qz0: qx * qy * (qz0 + nqz)]).max(), 0.0)
        u = splitmix_src(op.m(), salt=21)
        s, d, sr, dr = op.vector_from(u), op.initialize_dof_vector(), ref.vector_from(u), ref.initialize_dof_vector()
        op.vmult(d, s)
        ref.vmult(dr, sr)
        scale = np.abs(dr.export_host()).max()
        report(name + ": vmult (owned planes)", np.abs(d.export_host() - dr.export_host()).max() / scale, 1e-14)
        op.compute_diagonal()
        ref.compute_diagonal()
        di, dir_ = op.get_matrix_diagonal_inverse(), ref.get_matrix_diagonal_inverse()
        report(name + ": inverse diagonal (stored planes)",
               np.abs(di.export_local() - local_of(dir_, di)).max() / np.abs(dir_.export_host()).max(), 1e-14)
        del op, ref, s, d, sr, dr

    levels = hierarchy_levels("h", p, n)
    results = []
    for c in (ctx, one):
        ops, _, _, mg = G.build_hierarchy(c, levels, faces=SHELL_FACES, mapping=shell_map, coefficient=jump)
        top = ops[-1]
        b, x = top.initialize_dof_vector(), top.initialize_dof_vector()
        top.assemble_rhs(b)
        it, _, rc = G.cg_solve(top, x, b, mg)
        results.append((it, rc, x.export_host()))
        del ops, mg, top, b, x
    (it, rc, x), (it1, rc1, x1) = results
    report("shell solve: CG iterations %d vs %d" % (it, it1), float(abs(it - it1) + abs(rc) + abs(rc1)), 0.0)
    report("shell solve: solution", np.abs(x - x1).max() / np.abs(x1).max(), 1e-10)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DIST CHECK PASSED" if flag.item() == 1 else "DIST CHECK FAILED", flush=True)
    ctx.close()
    one.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
