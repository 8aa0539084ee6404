"""Multi-GPU worker for the steps around the SIMPLE loop (run under torchrun, one rank per GPU): flow initialisation, Jacobi as the
loop's solver, gradients of the resident fields and run files on partition meshes, against one GPU with the whole mesh (rank 0,
a context without a communicator, ReductionMode.Fast) and the oracle. Prints one JSON line. Used by tests/test_gpu_multi_init.py:

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 tests/mgpu_init_worker.py
"""
import json
import os
import shutil
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import orc_b200  # noqa: E402
from orc_b200 import io as oio  # noqa: E402
from orc_b200 import synthetic as syn  # noqa: E402
from orc_b200 import discretization as disc  # noqa: E402
from orc_b200.settings import (GradientReconstructionMethods as G, MatrixSolverSettings, ReductionMode, SolutionMethod,  # noqa: E402
                               VelocityInterpolation)
from mgpu_check import gather_owned, partition_parity  # noqa: E402

RHO, MU = 1000.0, 1e-3
FAST = ReductionMode.Fast


def arrays_of(kind):
    return syn.hex_box(12, 8, 8) if kind == "hex" else syn.tet_box(4, 3, 4)


def velocity_bcs(m):
    """velocity inlet + pressure outlet: a VelocityOnly system (initialize_velocity_field)"""
    m.set_zone("INLET", 10, 0.0, (1e-3, 0.0, 0.0))
    m.set_zone("OUTLET", 5, 0.0, (0.0, 0.0, 0.0))
    m.set_zone("WALL", 3, 0.0, (0.0, 0.0, 0.0))
    m.set_zone("SYM", 7, 0.0, (0.0, 0.0, 0.0))


def global_mesh(kind, bcs):
    g = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays_of(kind)))
    bcs(g)
    return g


def rank_part(kind, bcs, window):
    """this rank's partition: cut from the global mesh, or built from a z-slab window (no global mesh on the rank)"""
    rank, world = dist.get_rank(), dist.get_world_size()
    if not window:
        return global_mesh(kind, bcs).partition(rank, world)
    slab = syn.slab_partition(12, 8, 8, rank, world) if kind == "hex" else syn.tet_slab_partition(4, 3, 4, rank, world)
    arrays, cuts, off, n_global = slab
    w = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    bcs(w)
    return w.partition_window(rank, world, cuts, off, n_global)


def gather(cols, part, device):
    """owned columns of every rank -> global arrays (2-D arrays column by column)"""
    info = part.partition_info()
    out = []
    for a in cols:
        a = np.asarray(a)
        if a.ndim == 1:
            out.append(gather_owned(a, info, info["n_global"], device)[0])
        else:
            flat = a.reshape(a.shape[0], -1)
            g = np.stack([gather_owned(np.ascontiguousarray(flat[:, k]), info, info["n_global"], device)[0] for k in range(flat.shape[1])], 1)
            out.append(g.reshape((info["n_global"],) + a.shape[1:]))
    return out


def vel_dev(got, ref):
    vel = np.sqrt(sum(np.linalg.norm(b) ** 2 for b in ref[:3]))
    return max(float(np.linalg.norm(a - b)) for a, b in zip(got[:3], ref[:3])) / vel


def equal(a, b):
    return bool(all(np.array_equal(x, y) for x, y in zip(a, b)))


def init_cases(ctx, single, device, out):
    from oracle import pyoracle as po
    rank = dist.get_rank()
    for kind in ("hex", "tet"):
        res = {}
        got = {}
        for window in (False, True):
            tag = "window" if window else "cut"
            part = rank_part(kind, syn.channel_bcs, window)
            c0 = ctx.launch_count()
            got[tag, "flow"] = gather(orc_b200.initialize_flow(part, MU, RHO, 6, ctx=ctx), part, device)
            lockstep_launches = ctx.launch_count() - c0
            if not window:   # the lockstep u/v/w solve: fewer launches than three solves, the same bits
                os.environ["ORC_B200_BATCH"] = "0"
                c0 = ctx.launch_count()
                seq = gather(orc_b200.initialize_flow(part, MU, RHO, 6, ctx=ctx), part, device)
                seq_launches = ctx.launch_count() - c0
                del os.environ["ORC_B200_BATCH"]
                res["lockstep"] = bool(lockstep_launches < seq_launches and equal(seq, got[tag, "flow"]))
            got[tag, "new_p"] = gather(orc_b200.initialize_flow_new(part, MU, RHO, 0, ctx=ctx), part, device)
            vpart = rank_part(kind, velocity_bcs, window)
            got[tag, "new_v"] = gather(orc_b200.initialize_flow_new(vpart, MU, RHO, 0, ctx=ctx), vpart, device)
        res["window_equals_cut"] = all(equal(got["window", k], got["cut", k]) for k in ("flow", "new_p", "new_v"))
        if rank == 0:
            g = global_mesh(kind, syn.channel_bcs)
            s = orc_b200.initialize_flow(g, MU, RHO, 6, ctx=single, reduction_mode=FAST)
            om = po.Mesh.from_arrays(*syn.mesh_args(arrays_of(kind)))
            syn.channel_bcs(om)
            o = om.initialize_flow(MU, RHO, 6)
            f = got["cut", "flow"]
            res["flow_p_equal_single"] = bool(np.array_equal(f[3], s[3]))
            res["flow_p_equal_oracle"] = bool(np.array_equal(f[3], o[3]))
            res["flow_uvw_vs_single"] = vel_dev(f, s)
            res["flow_uvw_vs_oracle"] = vel_dev(f, o)
            sn = orc_b200.initialize_flow_new(g, MU, RHO, 0, ctx=single, reduction_mode=FAST)
            res["new_pressure_p_equal"] = bool(np.array_equal(got["cut", "new_p"][3], sn[3]))
            sv = orc_b200.initialize_flow_new(global_mesh(kind, velocity_bcs), MU, RHO, 0, ctx=single, reduction_mode=FAST)
            res["new_velocity_vs_single"] = vel_dev(got["cut", "new_v"], sv)
            res["new_velocity_nonzero"] = bool(np.abs(sv[0]).max() > 0)
        out[f"init_{kind}"] = res


def wrap_case(ctx, single, device, out):
    """u16 wrap of the moving-wall face count: 22 x 42 x 69 hexes have 3 * 65536 faces (PressureOnly), 22 x 42 x 68 do not"""
    rank, world = dist.get_rank(), dist.get_world_size()
    for nz in (69, 68):
        arrays = syn.hex_box(22, 42, nz)
        g = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
        g.set_zone("WALL", 3, 0.0, (1e-3, 0.0, 0.0))
        g.set_zone("INLET", 3, 0.0, (0.0, 0.0, 0.0))
        g.set_zone("OUTLET", 5, 1e-2, (0.0, 0.0, 0.0))
        part = g.partition(rank, world)
        f = gather(orc_b200.initialize_flow_new(part, MU, RHO, 0, ctx=ctx), part, device)
        if rank == 0:
            s = orc_b200.initialize_flow_new(g, MU, RHO, 0, ctx=single, reduction_mode=FAST)
            out[f"wrap_{nz}"] = {"faces": g.counts()["faces"], "constraint": int(orc_b200.check_boundary_conditions(g)),
                                 "equal_single": equal(f, s), "p_nonzero": bool(np.abs(f[3]).max() > 0)}


def jacobi_cases(ctx, single, device, out):
    from oracle import pyoracle as po
    rank, world = dist.get_rank(), dist.get_world_size()
    jac = MatrixSolverSettings(solver_type=SolutionMethod.Jacobi)
    settings = orc_b200.NumericalSettings(velocity_interpolation=VelocityInterpolation.LinearWeighted, matrix_solver=jac, reduction_mode=FAST)
    g = global_mesh("hex", syn.channel_bcs)
    part = g.partition(rank, world)
    st = orc_b200.SteadySolver(part, settings, RHO, MU, ctx)
    st.iterate(3)
    f = gather(st.get_fields(), part, device)
    st.close()
    if rank == 0:
        ss = orc_b200.SteadySolver(g, settings, RHO, MU, single)
        ss.iterate(3)
        out["jacobi_linear_weighted_equal_single"] = equal(f, ss.get_fields())
        ss.close()
    par = partition_parity(ctx, device, shape=(12, 8, 8), iters=3,
                           settings=orc_b200.NumericalSettings(matrix_solver=MatrixSolverSettings(solver_type=SolutionMethod.Jacobi)),
                           oracle_settings=po.Settings(solver_type=po.JACOBI))
    if rank == 0:
        out["jacobi_oracle_partition_parity"] = par
    # a relaxation far past stability: the solver's magnitude check fires, on every rank alike, and the contexts stay usable
    bad = orc_b200.NumericalSettings(matrix_solver=MatrixSolverSettings(solver_type=SolutionMethod.Jacobi, relaxation=40.0), reduction_mode=FAST)
    st = orc_b200.SteadySolver(part, bad, RHO, MU, ctx)
    code = 0
    try:
        st.iterate(2)
    except orc_b200.OrcError as e:
        code = e.code
    st.close()
    codes = [None] * world
    dist.all_gather_object(codes, code)
    st = orc_b200.SteadySolver(part, settings, RHO, MU, ctx)
    st.iterate(1)
    ok = bool(all(np.isfinite(a).all() for a in st.get_fields()))
    st.close()
    oks = [None] * world
    dist.all_gather_object(oks, ok)
    out["divergence"] = {"codes": codes, "next_call_ok": oks}


def gradient_and_file_cases(ctx, single, device, out, tmp):
    rank, world = dist.get_rank(), dist.get_world_size()
    res = {}
    grads = {}
    for window in (False, True):
        part = rank_part("hex", syn.channel_bcs, window)
        st = orc_b200.SteadySolver(part, orc_b200.NumericalSettings(reduction_mode=FAST), RHO, MU, ctx)
        st.iterate(3)
        local = st.get_fields()
        fields = gather(local, part, device)
        for scheme in (G.GreenGaussCellBased, G.LeastSquares):
            grads[window, scheme] = gather(st.gradients(scheme), part, device)
        if not window:
            oio.write_data(part, *local, os.path.join(tmp, f"data_{rank}.csv"))
            st.write_gradients(os.path.join(tmp, f"grad_{rank}.csv"), 7, G.LeastSquares)
        st.close()
        if not window:
            cut_fields = fields
    res["window_equals_cut"] = all(equal(grads[True, s], grads[False, s]) for s in (G.GreenGaussCellBased, G.LeastSquares))
    dist.barrier()
    if rank == 0:
        g = global_mesh("hex", syn.channel_bcs)
        for scheme in (G.GreenGaussCellBased, G.LeastSquares):
            res[f"equal_single_{int(scheme)}"] = equal(grads[False, scheme], disc.calculate_gradients(g, *cut_fields, scheme, single))
        oio.write_data(g, *cut_fields, os.path.join(tmp, "data.csv"))
        oio.write_gradients(g, *cut_fields, os.path.join(tmp, "grad.csv"), 7, G.LeastSquares, single)
        for name in ("data", "grad"):
            cat = b"".join(open(os.path.join(tmp, f"{name}_{r}.csv"), "rb").read() for r in range(world))
            res[f"{name}_file_equal"] = cat == open(os.path.join(tmp, f"{name}.csv"), "rb").read()
    out["gradients_and_files"] = res


def main():
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = orc_b200.Context(local_rank)
    ctx.comm_init()
    single = orc_b200.Context(local_rank) if rank == 0 else None   # a context without a communicator: the single-GPU path
    out = {"world": world, "peer": bool(ctx.peer)}
    tmp = [tempfile.mkdtemp(prefix="orc_mgpu_init_") if rank == 0 else None]
    dist.broadcast_object_list(tmp, 0)
    init_cases(ctx, single, device, out)
    wrap_case(ctx, single, device, out)
    jacobi_cases(ctx, single, device, out)
    gradient_and_file_cases(ctx, single, device, out, tmp[0])
    dist.barrier()
    if rank == 0:
        shutil.rmtree(tmp[0], ignore_errors=True)
        print("MGPU_RESULT " + json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
