"""Wall time of the flow initialisation on the 256^3 hex channel: initialize_flow_new and initialize_flow (iteration_count 50).

One rank: the whole mesh on one GPU. N ranks (torchrun --nproc-per-node N): each rank builds only its z-slab window
(synthetic.slab_partition), so no rank ever holds the global mesh. Every timed call sits between a device synchronisation and a
barrier, and the slowest rank's time is reported. Prints one JSON line (and writes it to --out), with the card name and power
limit read in the same run.

    python scripts/init_scale.py --out profiles/init_scale_256_1gpu.json
    torchrun --nnodes=1 --nproc-per-node 8 scripts/init_scale.py --out profiles/init_scale_256_8gpu.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(local_rank):
    q = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--iterations", type=int, default=50, help="iteration_count of initialize_flow")
    ap.add_argument("--repeats", type=int, default=2, help="timed calls per function, after one untimed call")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import orc_b200
    from orc_b200 import synthetic as syn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    ctx = orc_b200.Context(local_rank)
    n = args.size
    t0 = time.perf_counter()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
        rank = dist.get_rank()
        ctx.comm_init()
        arrays, cuts, off, n_global = syn.slab_partition(n, n, n, rank, world)
        mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
        syn.channel_bcs(mesh)
        mesh = mesh.partition_window(rank, world, cuts, off, n_global)
    else:
        dist, rank = None, 0
        mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(n, n, n)))
        syn.channel_bcs(mesh)
    setup_s = time.perf_counter() - t0

    def timed(fn, *a):
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        t = time.perf_counter()
        fn(*a, ctx=ctx)
        ctx.synchronize()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t) * 1e3
        if dist:
            v = torch.tensor([ms], dtype=torch.float64, device=device)
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            ms = float(v.item())
        return ms

    mu, rho = 1e-3, 1000.0
    res = {"config": f"hex channel {n}^3", "cells": n ** 3, "ranks": world,
           "partition": "windowed z-slabs (synthetic.slab_partition)" if world > 1 else "whole mesh",
           "initialize_flow_iteration_count": args.iterations, "mesh_setup_s": round(setup_s, 2)}
    res.update(card(local_rank))
    for name, fn, fargs in (("initialize_flow_new", orc_b200.initialize_flow_new, (mesh, mu, rho, 0)),
                            ("initialize_flow", orc_b200.initialize_flow, (mesh, mu, rho, args.iterations))):
        timed(fn, *fargs)   # untimed: first launches, allocator warm-up
        res[f"{name}_ms"] = [round(timed(fn, *fargs), 2) for _ in range(args.repeats)]
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
