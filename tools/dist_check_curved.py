#!/usr/bin/env python
"""Multi-GPU parity of the operator on curved cells (run under torchrun, one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/dist_check_curved.py
Every rank builds the slab-distributed hierarchy on the quarter cylindrical shell with MappingQ(p) cells on every level
(each rank uploads the node planes of its own cell layers only), rank 0 additionally runs the CPU oracle; apply, V-cycle,
right-hand side, CG and the solution norm must agree with the oracle to the single-GPU tolerances and the iteration count
must be identical."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "portable-multigrid_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist
import pmg_b200 as G
from helpers import hierarchy_levels, rel_l2, splitmix_src
from curved_mesh import SHELL_FACES, nodes_of, shell_map
from curved_oracle import curved_matrix_free, l2_norm_curved


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    obj = [G.Context.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    ctx = G.Context(local, rank, world, obj[0])
    ctx.set_coarse_threshold(2000)
    import pyoracle as O

    ok = True

    def report(name, err, tol):
        nonlocal ok
        if rank == 0:
            print("%-44s %.3e %s" % (name, err, "ok" if err <= tol else "FAIL"), flush=True)
        ok = ok and (err <= tol)

    p, n = 3, 4 * world
    levels = hierarchy_levels("h", p, n)
    ops, _, _, mg = G.build_hierarchy(ctx, levels, faces=SHELL_FACES, mapping=shell_map)
    top = ops[-1]
    mfs = [curved_matrix_free(O, q, m, nodes_of(shell_map, m, q), q, faces=SHELL_FACES) for (q, m) in levels]
    trs = [O.Transfer(mfs[l - 1], mfs[l], "h") for l in range(1, len(levels))]
    vc = O.VCycle(mfs, trs)
    vc.estimate()
    u = splitmix_src(mfs[-1].n_dofs, salt=3)
    s, d = top.vector_from(u), top.initialize_dof_vector()
    top.vmult(d, s)
    report("vmult", rel_l2(d.export_host(), mfs[-1].vmult(u)), 1e-12)
    r = splitmix_src(mfs[-1].n_dofs, mfs[-1].constrained(), salt=4)
    dr, dz = top.vector_from(r), top.initialize_dof_vector()
    mg.vmult(dz, dr)
    report("V-cycle", rel_l2(dz.export_host(), vc.vmult(r)), 1e-10)
    b = top.initialize_dof_vector()
    top.assemble_rhs(b)
    b_ref = mfs[-1].assemble_rhs()
    report("rhs", rel_l2(b.export_host(), b_ref), 1e-13)
    x_ref, it_ref, hist_ref, _ = O.cg_solve(mfs[-1], b_ref, vc)
    x = top.initialize_dof_vector()
    it, hist, rc = G.cg_solve(top, x, b, mg)
    report("CG iterations %d vs %d" % (it, it_ref), float(abs(it - it_ref)), 0.0)
    report("CG residual history", float(np.max(np.abs(hist - hist_ref)) / hist_ref[0]) if it == it_ref else 1.0, 1e-10)
    report("solution", rel_l2(x.export_host(), x_ref), 1e-9)
    report("solution norm", abs(top.solution_norm(x) - l2_norm_curved(mfs[-1], x_ref)), 1e-10)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DIST CHECK PASSED" if flag.item() == 1 else "DIST CHECK FAILED", flush=True)
    del ops, mg, top, s, d, dr, dz, b, x
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
