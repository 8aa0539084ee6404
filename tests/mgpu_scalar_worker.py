"""Multi-GPU worker for the passive scalar transport (run under torchrun, one rank per GPU; used by
tests/test_gpu_multi_scalar.py): the partitioned assembly and scalar solves against one GPU and against the sequential model
with the oracle's partition emulation. Prints one JSON line on rank 0."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import orc_b200  # noqa: E402
from orc_b200 import discretization as disc  # noqa: E402
from orc_b200 import synthetic as syn  # noqa: E402
from orc_b200.settings import MomentumDiscretization, SolutionMethod, TvdLimiter  # noqa: E402
from cases import smooth_fields  # noqa: E402
from mgpu_worker import gather_owned  # noqa: E402

RHO, MU, GAMMA = 1000.0, 1e-3, 2e-3
FIXED = orc_b200.ScalarCondition.Fixed


def settings(**kw):
    ms = orc_b200.MatrixSolverSettings(**{k: kw.pop(k) for k in ("solver_type", "iterations", "relative_convergence_threshold") if k in kw})
    return orc_b200.NumericalSettings(matrix_solver=ms, **kw)


def main():
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = orc_b200.Context(local_rank)
    ctx.comm_init()
    single = orc_b200.Context(local_rank)   # no communicator: the single-GPU path
    arrays = syn.hex_box(12, 8, 8)
    gmesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(gmesh)
    gmesh.set_zone_scalar("INLET", FIXED, 1.0)
    gmesh.set_zone_scalar("WALL", FIXED, 0.25)
    n = gmesh.n_cells
    u, v, w, p = smooth_fields(gmesh.export())
    phi = np.random.default_rng(5).uniform(0.0, 1.0, n)
    part = gmesh.partition(rank, world)   # inherits the zones' scalar conditions
    info = part.partition_info()
    l2g = part.partition_maps()["local_to_global"]
    own = slice(info["n_lo"], info["n_lo"] + info["n_own"])
    out = {"world": world, "cells": n}

    # 1. the assembly: owned rows of the partition == the same rows of the whole mesh, bit for bit (unit diagonals)
    rows_equal = True
    for kw in (dict(), dict(momentum=MomentumDiscretization.TVD, limiter=TvdLimiter.QUICK)):
        s = settings(**kw)
        ga = [disc.initialize_momentum_matrix(gmesh, single) for _ in range(3)]
        a_g, b_g = disc.build_scalar_transport(gmesh, *ga, u, v, w, p, phi, GAMMA, RHO, s)
        la_ = [disc.initialize_momentum_matrix(part, ctx) for _ in range(3)]
        a_l, b_l = disc.build_scalar_transport(part, *la_, u[l2g], v[l2g], w[l2g], p[l2g], phi[l2g], GAMMA, RHO, s)
        grp, gco, gva = a_g.arrays()
        lrp, lco, lva = a_l.arrays()
        for i in range(own.start, own.stop):
            gi = l2g[i]
            ok = (np.array_equal(l2g[lco[lrp[i]:lrp[i + 1]]], gco[grp[gi]:grp[gi + 1]]) and np.array_equal(lva[lrp[i]:lrp[i + 1]], gva[grp[gi]:grp[gi + 1]])
                  and b_l[i] == b_g[gi])
            rows_equal = rows_equal and bool(ok)
    flags = torch.tensor([1.0 if rows_equal else 0.0], dtype=torch.float64, device=device)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    out["assembly_rows_equal"] = bool(flags.item() == 1.0)

    # 2. Jacobi with a fixed iteration count (threshold 0): phi bit-identical to one GPU
    def solve(mesh, c, s, sweeps, fields):
        st = orc_b200.SteadySolver(mesh, s, RHO, MU, c)
        st.set_fields(*fields)
        x = st.solve_scalar(GAMMA, None, sweeps)
        st.close()
        return x

    sj = settings(solver_type=SolutionMethod.Jacobi, iterations=40, relative_convergence_threshold=0.0)
    local = solve(part, ctx, sj, 2, [f[l2g][own] for f in (u, v, w, p)])
    got = gather_owned(local, info, n, device)
    want = solve(gmesh, single, sj, 2, [u, v, w, p])
    out["jacobi_equal"] = bool(np.array_equal(got, want))
    out["jacobi_max_diff"] = float(np.abs(got - want).max())

    # 3. Multigrid against the model with the oracle's partition emulation (per-partition coarse correction)
    sm = settings()
    local = solve(part, ctx, sm, 1, [f[l2g][own] for f in (u, v, w, p)])
    got = gather_owned(local, info, n, device)
    cuts = [None] * world
    dist.all_gather_object(cuts, info["g0"])
    if rank == 0:
        from oracle import pyoracle as po
        import scalar_oracle as so
        om = po.Mesh.from_arrays(*syn.mesh_args(arrays))
        syn.channel_bcs(om)
        bcs = so.ScalarBcs(om)
        bcs.set("INLET", so.FIXED, 1.0)
        bcs.set("WALL", so.FIXED, 0.25)
        po.set_partition(cuts + [n])
        try:
            want = so.solve(om, bcs, u, v, w, p, np.zeros(n), *so.unit_diagonals(om), GAMMA, RHO, po.Settings(), 1)
        finally:
            po.set_partition(None)
        single_gpu = solve(gmesh, single, sm, 1, [u, v, w, p])
        out["multigrid_vs_model"] = float(np.linalg.norm(got - want) / np.linalg.norm(want))
        out["multigrid_vs_single"] = float(np.linalg.norm(got - single_gpu) / np.linalg.norm(single_gpu))
        out["finite"] = bool(np.isfinite(got).all())
        print("MGPU_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
