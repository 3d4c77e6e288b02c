"""One rank of the multi-GPU check of the default step-size option on PDHG slabs (launched by
tests/test_gpu_multi_gpu_defaults.py through ``python -m torch.distributed.run``).  Every rank runs its column slab
with ``scale_steps_operator = 1``, i.e. the power iteration of the operator norm on the global operator; rank 0 also
solves the whole problem on one GPU and compares the step sizes after Initialize, the iterates and the residuals."""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def cases(world):
    from prost_b200 import synthetic as syn
    identity = ("identity",)
    return {
        "rof_alpha": (lambda: syn.rof(64, 48), dict(stepsize="alg1", residual_iter=3), 40, False),
        # |K| ~ sqrt(8): the steps really are rescaled
        "rof_identity": (lambda: dict(syn.rof(64, 48), scaling=identity), dict(stepsize="boyd", residual_iter=4), 40,
                         False),
        "tvl1": (lambda: syn.tvl1(40, 32, nc=3), dict(stepsize="boyd", residual_iter=5), 40, False),
        "tv3d": (lambda: syn.tv3d(14, 16, 6), dict(stepsize="alg1", residual_iter=5), 30, False),
        "lifting": (lambda: syn.lifting(18, 12, 6), dict(stepsize="boyd", residual_iter=5), 30, False),
        # a given global start vector, each rank passes its slice
        "rof_identity_x0": (lambda: dict(syn.rof(50, 40), scaling=identity), dict(stepsize="alg1", residual_iter=3),
                            30, True),
        # world + 1 columns: every rank but the first owns ONE column
        "rof_one_column": (lambda: dict(syn.rof(world + 1, 40), scaling=identity),
                           dict(stepsize="goldstein", residual_iter=2), 30, False),
    }


def main():
    import torch
    import torch.distributed as dist
    import prost_b200 as pb
    from prost_b200 import distributed as pbd

    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    ctx = pb.Context(local)
    comm = pbd.init_comm(ctx)
    report = {"world": world, "p2p": comm.peer_to_peer, "cases": {}}
    tol = dict(tol_rel_primal=1e-4, tol_rel_dual=1e-4, tol_abs_primal=1e-4, tol_abs_dual=1e-4)

    for name, (make, opts, iters, with_x0) in cases(world).items():
        desc = make()
        nx, ny, L = pbd._grid_of(desc)
        part = pbd.SlabPartition(nx, world)
        local_desc = pbd.shard_description(desc, part, rank)
        x0_global = np.random.default_rng(7).random(desc["ncols"]).astype(np.float32) if with_x0 else None

        def run(d, c, x0):
            prob = pb.create_problem(ctx, d)
            popts = pb.pdhg_options(scale_steps_operator=1, **opts)
            if x0 is not None:
                popts.normest_x0 = x0.ctypes.data_as(C.POINTER(C.c_float))
            sopts = pb.solver_options(verbose=0, max_iters=iters, num_cback_calls=0, **tol)
            be = pb.BackendPDHG(ctx, prob, popts, sopts, comm=c)
            prob.Initialize()
            be.Initialize()
            steps0 = be.stepsizes()
            be.PerformIteration(iters)
            x, z, y, w = be.current_solution()
            return dict(x=x, z=z, y=y, w=w, res=be.residuals(), steps0=steps0)

        x0_local = None
        if with_x0:
            x0_local = pbd.slice_planar(x0_global, nx, ny, *part.range(rank))
        mine = run(local_desc, comm, x0_local)
        gathered = [None] * world
        dist.gather_object({k: mine[k] for k in ("x", "z", "y", "w")}, gathered if rank == 0 else None, dst=0)
        if rank == 0:
            ref = run(desc, None, x0_global)
            f32 = np.float32
            steps_ulps = [int(abs(np.int64(f32(a).view(np.int32)) - np.int64(f32(b).view(np.int32))))
                          for a, b in zip(mine["steps0"][:2], ref["steps0"][:2])]
            out = {"steps0": mine["steps0"], "steps0_single": ref["steps0"], "steps_ulps": steps_ulps,
                   "res": mine["res"], "res_single": ref["res"], "err": {}, "bit_equal": {}}
            for k in ("x", "z", "y", "w"):
                glob = pbd.gather_planar([g[k] for g in gathered], part, ny)
                denom = max(float(np.abs(ref[k]).max()), 1e-30)
                out["err"][k] = float(np.abs(glob.astype(np.float64) - ref[k]).max() / denom)
                out["bit_equal"][k] = bool(np.array_equal(glob, ref[k]))
            report["cases"][name] = out
        comm.barrier()

    if rank == 0:
        c = report["cases"]
        report["steps_bit_equal"] = sum(1 for v in c.values() if max(v["steps_ulps"]) == 0)
        report["iterates_bit_equal"] = sum(1 for v in c.values() if all(v["bit_equal"].values()))
        print("DEFAULTS_SLAB_REPORT " + json.dumps(report), flush=True)
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
