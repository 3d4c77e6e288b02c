"""One rank of the multi-GPU check of the default (alpha) preconditioners on BackendADMM row shards (launched by
tests/test_gpu_multi_gpu_defaults.py through ``python -m torch.distributed.run``).  Every rank solves its block of
rows with Pock-Chambolle alpha scaling; rank 0 also solves the whole problem on one GPU and compares Sigma, T, the
iterates, the residuals and the iteration counts."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def empty_carry(world, m=1200, n=300):
    """LASSO whose K has empty rows straddling the boundary between ranks 0 and 1 and up to the last row of the
    first shard, plus an empty first column: the row carry crosses ranks and column 0 takes the carry of the
    globally last row."""
    import scipy.sparse as sp
    from prost_b200 import distributed as pbd
    from prost_b200 import synthetic as syn
    d = syn.lasso(m, n, nnz_per_row=5)
    K = sp.csr_matrix(d["blocks"][0][3][0])
    keep = np.ones(m, dtype=np.float32)
    b = pbd.RowPartition(m, max(world, 2)).range(0)[1]
    keep[b - 7:b + 5] = 0                       # the last rows of rank 0 and the first rows of rank 1
    keep[-3:] = 0                               # the globally last rows are empty too
    cols = np.ones(n, dtype=np.float32)
    cols[0] = 0
    K = (sp.diags(keep) @ K @ sp.diags(cols)).tocsr()
    K.eliminate_zeros()
    d["blocks"] = [("sparse", 0, 0, [K.tocsc()])]
    return d


def cases(world):
    from prost_b200 import synthetic as syn

    def alpha(make, a):
        def f():
            d = make()
            d["scaling"] = ("alpha", a)
            return d
        return f

    sparse = lambda: syn.lasso(3000, 700, nnz_per_row=5)                      # noqa: E731
    dense = lambda: syn.lasso(2500, 640, nnz_per_row=6, dense=96)            # noqa: E731
    return {
        "lasso_a1": (alpha(sparse, 1.0), 25, dict(residual_iter=1)),
        "lasso_a05": (alpha(sparse, 0.5), 25, dict(residual_iter=1)),
        "lasso_dense_a1": (alpha(dense, 1.0), 25, dict(residual_iter=2)),
        "lasso_dense_a05": (alpha(dense, 0.5), 25, dict(residual_iter=2)),
        "empty_carry": (alpha(lambda: empty_carry(world), 1.0), 25, dict(residual_iter=1)),
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
    tol = dict(tol_rel_primal=0, tol_rel_dual=0, tol_abs_primal=0, tol_abs_dual=0)

    for name, (make, iters, opts) in cases(world).items():
        desc = make()
        part = pbd.RowPartition(desc["nrows"], world)
        local_desc = pbd.shard_rows(desc, part, rank)

        def run(d, c):
            prob = pb.create_problem(ctx, d)
            sopts = pb.solver_options(verbose=0, max_iters=iters, num_cback_calls=0, **tol)
            be = pb.BackendADMM(ctx, prob, pb.admm_options(**opts), sopts, comm=c)
            solver = pb.Solver(prob, be)
            solver.SetOptions(sopts)
            solver.Initialize()
            left, right = prob.scaling()
            solver.Solve()
            return dict(x=np.array(solver.cur_primal_sol), z=np.array(solver.cur_primal_constr_sol),
                        y=np.array(solver.cur_dual_sol), w=np.array(solver.cur_dual_constr_sol), res=be.residuals(),
                        iterations=int(solver.iterations), sigma=left, T=right)

        mine = run(local_desc, comm)
        gathered = [None] * world
        dist.gather_object({k: mine[k] for k in ("x", "z", "y", "w", "sigma", "T")}, gathered if rank == 0 else None,
                           dst=0)
        if rank == 0:
            ref = run(desc, None)
            sigma = np.concatenate([g["sigma"] for g in gathered])
            T = gathered[0]["T"]
            out = {"res": mine["res"], "res_single": ref["res"], "iterations": mine["iterations"],
                   "iterations_single": ref["iterations"], "err": {},
                   "sigma_bit_equal": bool(np.array_equal(sigma, ref["sigma"])),
                   "T_identical_on_ranks": bool(all(np.array_equal(g["T"], T) for g in gathered)),
                   "T_rel_err": float((np.abs(T.astype(np.float64) - ref["T"]) / np.abs(ref["T"])).max()),
                   "T_bit_equal": bool(np.array_equal(T, ref["T"]))}
            glob = {"x": gathered[0]["x"], "w": gathered[0]["w"],
                    "z": np.concatenate([g["z"] for g in gathered]), "y": np.concatenate([g["y"] for g in gathered])}
            for k in ("x", "z", "y", "w"):
                denom = max(float(np.abs(ref[k]).max()), 1e-30)
                out["err"][k] = float(np.abs(glob[k].astype(np.float64) - ref[k]).max() / denom)
            report["cases"][name] = out
        comm.barrier()
    if rank == 0:
        print("DEFAULTS_SHARD_REPORT " + json.dumps(report), flush=True)
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
