"""Wall time of BackendPDHG.Initialize on column slabs, with and without the operator-norm step rescaling
(``scale_steps_operator``).  Run one process per GPU:

    python -m torch.distributed.run --nproc-per-node=N scripts/initialize_cost.py [--nx 4096 --ny 4096] [--out f]

Every rank builds its slab of ``synthetic.rof(nx, ny)`` and times Initialize (host clock around a call that ends
in a stream synchronise; the slowest rank counts) ``--reps`` times per setting after one untimed call.  World 1
also times the same problem without a communicator.  Prints one JSON line with the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--ny", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import numpy as np
    import torch
    import torch.distributed as dist
    import prost_b200 as pb
    from prost_b200 import distributed as pbd
    from prost_b200 import synthetic as syn

    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    world = int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    ctx = pb.Context(local)
    comm = pbd.init_comm(ctx)
    desc = pbd.shard_description(syn.rof(a.nx, a.ny), pbd.SlabPartition(a.nx, world), rank)
    prob = pb.create_problem(ctx, desc)
    prob.Initialize()

    def timed(scale, c):
        be = pb.BackendPDHG(ctx, prob, pb.pdhg_options(scale_steps_operator=scale), pb.solver_options(verbose=0),
                            comm=c)
        be.Initialize()
        out = []
        for _ in range(a.reps):
            if c is not None:
                c.barrier()
            t0 = time.perf_counter()
            be.Initialize()
            dt = np.array([time.perf_counter() - t0])
            if c is not None:
                dt = np.array([c.allreduce_sum(np.eye(world)[rank] * dt[0]).max()])
            out.append(float(dt[0]))
        return dict(seconds=out, tau=be.stepsizes()[0])

    res = {"world": world, "nx": a.nx, "ny": a.ny, "p2p": comm.peer_to_peer, "gpu": gpu_info(local)}
    for scale in (0, 1):
        res[f"slab_scale{scale}"] = timed(scale, comm)
        if world == 1:
            res[f"single_scale{scale}"] = timed(scale, None)
    if rank == 0:
        line = json.dumps(res)
        print("INITIALIZE_COST " + line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
