#!/usr/bin/env python
"""bench.py — SIMPLE iterations/s of the B200 path on BASELINE.json's workload (synthetic hex channel, defaults:
CD1 momentum, SecondOrder pressure, Rhie-Chow, Multigrid with BiCGSTAB smoothing, 50 inner iterations, fp64).

One "step" = one SIMPLE iteration (the body of the loop at src/solver.rs:60-222 of the reference).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--size n]            # our arm (weak scaling: N slabs of n^3 cells)
  python bench.py --scaling strong [--size 256] --gpus N                    # ONE size^3 mesh cut into N slabs
  python bench.py --mesh couette|channel|tet                                # BASELINE.json configs 1, 2 and 5 (in kind)
  python bench.py --impl reference [--steps K] [--warmup W]                 # the reference's CPU path (oracle restatement)
  python bench.py ... --dump-outputs DIR                                    # also write u, v, w, p of the last timed step as DIR/*.npy

Prints ONE JSON line (rank 0). See DESIGN.md §7 for what every key means and how the roofline figures are derived.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RHO, MU = 1000.0, 1e-3
P_RELAX = 1e-4        # pressure relaxation (README of the reference: "<< 0.1"); every other setting is the reference default
SPMV_SAMPLE = 17      # CUDA events around every 17th SpMV launch inside the timed region (odd: alternates between the two SpMVs of a BiCGSTAB iteration)
RESET_EVERY = 6       # SIMPLE iterations between resets of the fields (see run_ours.step)
METRIC = "SIMPLE iters/s"
GOLDEN = os.path.join(ROOT, "tests", "golden")
DUMP_BYTES = 64_000_000   # --dump-outputs: the most all arrays may take together
DUMP_SAMPLE = 1 << 20     # cells kept when the full fields would take more


def workload_name(shape):
    cells = int(np.prod(shape))
    dims = f"{shape[0]}^3" if shape[0] == shape[1] == shape[2] else "x".join(str(s) for s in shape)
    return f"synthetic {dims} hex channel ({cells / 1e6:.1f}M cells), SIMPLE + AMG-BiCGSTAB fp64"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        try:
            if self.proc:
                self.proc.terminate()
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx.append(float(s[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


ORACLE_PHASES = ("momentum_assembly", "momentum_solves", "pressure_assembly", "pressure_solve", "correction")


def oracle_run(m, steps=1, warmup=0):
    """`steps` SIMPLE iterations of the CPU restatement of the reference path on an m^3 hex channel with the bench settings
    (1 thread, like ORC). Returns (cells, seconds, per-phase seconds of the timed iterations)."""
    from oracle import pyoracle as po
    from orc_b200 import synthetic as syn
    a = syn.hex_box(m, m, m)
    om = po.Mesh.from_arrays(*syn.mesh_args(a))
    del a
    syn.channel_bcs(om)
    n = om.n_cells
    z = [np.zeros(n) for _ in range(4)]
    if warmup:
        z = list(om.solve_steady(*z, po.Settings(pressure_relaxation=P_RELAX), RHO, MU, warmup, 0)[:4])
    t0 = time.perf_counter()
    out = om.solve_steady(*z, po.Settings(pressure_relaxation=P_RELAX), RHO, MU, steps, 0)
    dt = time.perf_counter() - t0
    return n, dt, dict(zip(ORACLE_PHASES, (float(x) for x in out[5])))


def run_reference(args, rank, world):
    """The reference's path on the host cores, as oracle/ restates it in C++ (single-threaded like ORC; DESIGN.md §2 says why the
    Rust crate itself is not timed), on THE SAME MESH as our arm's N = 1 workload (size^3 cells, default 128^3): --warmup untimed
    SIMPLE iterations from rest, then --steps timed ones. One iteration takes about two minutes of one core at 128^3.
    At N > 1 our arm's global mesh has N x size^3 cells (weak scaling): the reference is still timed on size^3 and its rate is
    expressed in global-mesh iterations (cell count ratio), `same_config` false."""
    if rank != 0:
        return
    n = args.size if args.size else 128
    steps = args.steps
    t_wall = time.perf_counter()
    cells, dt, phases = oracle_run(n, steps=steps, warmup=args.warmup)
    cell_rate = cells * steps / dt
    strong = args.scaling == "strong"
    gcells = cells if strong else world * cells
    iters_global = cell_rate / gcells
    value = iters_global if strong else world * iters_global      # same units as our arm's `value`
    shape = (n, n, n)
    sample = (f"{steps} full SIMPLE iteration(s) after {args.warmup} untimed one(s) from rest on the {n}^3 hex channel itself ({cells} cells, "
              f"{dt:.1f} s), same settings as our arm")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "iter/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "steps_timed": steps, "warmup_done": args.warmup,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(shape), "solver": "Multigrid(BiCGSTAB x50, 3 levels, Jacobi precond)", "momentum": "CD1",
                       "velocity_interpolation": "RhieChow", "pressure_interpolation": "SecondOrder", "pressure_relaxation": P_RELAX,
                       "same_config": world == 1 or strong,
                       "note": None if world == 1 else f"our arm at {world} GPUs runs a {gcells}-cell mesh; the CPU path is timed on {cells} cells and "
                                                       f"its cell-update rate expressed in the same units"},
            "cpu_baseline": {"value": value, "unit": "iter/s", "cores": 1, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "phases_ms_per_step": {k: 1e3 * v / steps for k, v in phases.items()},
            "phases_note": "per-phase wall time of the timed iteration(s) (BASELINE.md §4 split), C++ restatement of the reference path",
            "cell_updates_per_s": cell_rate, "global_iters_per_s": iters_global, "gpu_launches": 0,
            "wall_s": time.perf_counter() - t_wall}
    print(json.dumps(line), flush=True)


# ---- the reference's own example meshes (BASELINE.json configs 1 and 2), from the committed connectivity fixtures ----------------
def small_mesh(kind):
    """(mesh, settings, description). kind 'couette': configs[0] — couette_flow_128x64x1.msh, BCs of src/tests.rs:60-76, CD1 momentum,
    Gauss-Seidel (the intended lexicographic formula: the reference's own GS panics, SURVEY Q10). kind 'channel': configs[1] —
    channel_flow.msh, TVD-QUICK, Rhie-Chow, SecondOrder, Multigrid with BiCGSTAB smoothing."""
    import orc_b200
    from orc_b200 import settings as S
    name = {"couette": "couette_flow_128x64x1", "channel": "channel_flow"}[kind]
    z = np.load(os.path.join(GOLDEN, f"mesh_{name}.npz"), allow_pickle=False)
    mesh = orc_b200.Mesh.from_arrays(int(z["dims"]), z["xyz"], z["face_node_offsets"], z["face_nodes"], z["c0"], z["c1"], z["face_zone"],
                                     z["zone_ids"], z["zone_types"], [str(s) for s in z["zone_names"]])
    if kind == "couette":
        for zn in ("TOP_WALL", "BOTTOM_WALL"):
            mesh.set_zone(zn, 3, 0.0, (5e-4 if zn == "TOP_WALL" else 0.0, 0.0, 0.0))
        dp_dx = 10.0
        ms = orc_b200.MatrixSolverSettings(solver_type=S.SolutionMethod.GaussSeidel, iterations=50)
        settings = orc_b200.NumericalSettings(matrix_solver=ms, gs_mode=S.GaussSeidelMode.Lexicographic)
        desc = "examples/couette_flow_128x64x1.msh (8001 cells): SIMPLE + Gauss-Seidel x50 (lexicographic dataflow sweep), CD1, Rhie-Chow"
    else:
        mesh.set_zone("WALL", 3, 0.0, (0.0, 0.0, 0.0))
        dp_dx = 5.0
        settings = orc_b200.NumericalSettings(momentum=S.MomentumDiscretization.TVD, limiter=S.TVD_QUICK)
        desc = "examples/channel_flow.msh (1008 cells): SIMPLE + AMG(BiCGSTAB x50), TVD-QUICK, Rhie-Chow, SecondOrder"
    mesh.set_zone("INLET", 4, -dp_dx * 0.002, (0.0, 0.0, 0.0))
    mesh.set_zone("OUTLET", 5, 0.0, (0.0, 0.0, 0.0))
    mesh.set_zone("PERIODIC_-Z", 7, 0.0, (0.0, 0.0, 0.0))
    mesh.set_zone("PERIODIC_+Z", 7, 0.0, (0.0, 0.0, 0.0))
    return mesh, settings, desc


def time_small(kind, ctx, torch, steps=10, warmup=3):
    import orc_b200
    mesh, settings, desc = small_mesh(kind)
    solver = orc_b200.SteadySolver(mesh, settings, RHO, MU, ctx)
    solver.set_fields(*(np.zeros(mesh.n_cells) for _ in range(4)))
    solver.iterate(warmup)
    stream = torch.cuda.current_stream()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    rep = solver.iterate(steps)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = {"config": desc, "cells": mesh.n_cells, "ms_per_iteration": ms, "iters_per_s": 1e3 / ms,
           "launches_per_iteration": (ctx.launch_count() - l0) / steps, "steps": steps, "warmup": warmup, "u_avg": rep["u_avg"]}
    solver.close()
    return out


def run_e2e(args, world, dist, torch, orc_b200, mesh, settings, solver, ctx, barrier):
    """e2e: the reference-facing call (solve_steady through the C ABI) with HOST buffers, copies inside the timed region."""
    solver.reset()
    solver.iterate(2)
    start_fields = solver.get_fields()   # every e2e step starts from the same host fields (2 iterations from rest)
    e2e_steps = args.e2e_steps
    sets = [[torch.from_numpy(f.copy()).pin_memory().numpy() for f in start_fields] for _ in range(e2e_steps)]
    # one untimed call first: the one-shot entry creates its own device state (5 matrices, 15 vectors), and the caching
    # allocator has to see those sizes once — like the W warm-up steps of the resident leg
    warm = [f.copy() for f in start_fields]
    with contextlib.redirect_stdout(sys.stderr):   # the mirror prints the reference's "Solving..." lines; stdout carries the JSON line only
        orc_b200.solve_steady(mesh, *warm, settings, RHO, MU, 1, 0, ctx=ctx, on_report=lambda d: None)
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        tk = time.perf_counter()
        with contextlib.redirect_stdout(sys.stderr):
            orc_b200.solve_steady(mesh, *sets[k], settings, RHO, MU, 1, 0, ctx=ctx, on_report=lambda d: None)
        print(f"[e2e] step {k}: {(time.perf_counter() - tk) * 1e3:.1f} ms", file=sys.stderr, flush=True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    return e2e_steps / e2e_s     # global-mesh iterations per second


def multi_gpu_parity(ctx, torch, dist, orc_b200, syn, local_rank, rank, world):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from mgpu_check import partition_parity, gather_owned
    device = torch.device("cuda", local_rank)
    out = partition_parity(ctx, device, iters=3)          # {vs_oracle_partitioned, vs_oracle_single}: 12 x 8 x 4N cells, reference defaults
    if rank == 0:
        out["note"] = ("relative L2 (u, v, w against the norm of the velocity field, p against ||p||). vs_oracle_partitioned: the CPU oracle "
                       "emulating the same partition (diagonals across a cut lag by one exchange, Multigrid coarse correction per partition "
                       "block): only the summation order of the dot products differs; oracle_sensitivity_to_1ulp_of_rho is the yardstick — how far "
                       "the oracle itself moves when the density changes by one ulp (the unguarded solvers amplify rounding, more so on larger "
                       "systems). vs_oracle_single: what that partitioning changes. "
                       "(On meshes beyond ~1 k cells the reference's unguarded BiCGSTAB amplifies ANY rounding difference into the leading "
                       "digits, DESIGN.md §5, so larger comparisons say nothing about the partitioning.)")
    dist.barrier()
    return out


def dump_outputs(path, fields):
    """Writes u, v, w, p as <path>/{u,v,w,p}.npy (float64). When the four fields together exceed DUMP_BYTES, every field keeps the
    same DUMP_SAMPLE cells, drawn with a fixed seed, so two builds of the project on the same mesh write the same cells;
    <path>/cell_index.npy (float64) then lists them."""
    os.makedirs(path, exist_ok=True)
    out = dict(zip("uvwp", fields))
    n = out["u"].size
    if 4 * 8 * n > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
        out = {k: f[idx] for k, f in out.items()}
        out["cell_index"] = idx
    for k, f in out.items():
        np.save(os.path.join(path, f"{k}.npy"), np.asarray(f, dtype=np.float64))


def pooled(detail, peak, codes):
    """detail records pooled by (rows, systems): the matrices of one AMG level differ from step to step and between the momentum
    and the pressure system. R has <= 4 entries per row, R^T <= 2: the short-row transfer products are left out."""
    pool = {}
    for r, z, k, t, b, cnt in detail:
        if k in codes and cnt and t > 0 and z > 4.5 * r:
            e = pool.setdefault((r, codes[k]), [0.0, 0.0, 0, 0.0])
            e[0] += t; e[1] += b; e[2] += cnt; e[3] += z * cnt
    return pool


def run_ours(args, rank, world):
    import torch
    import orc_b200
    from orc_b200 import synthetic as syn

    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.current_stream()
    ctx = orc_b200.Context(local_rank, stream.cuda_stream)
    strong = args.scaling == "strong"
    n = args.size if args.size else (256 if strong else 128)
    small = args.mesh in ("couette", "channel")
    tet = args.mesh == "tet"

    # Multi-GPU (DESIGN.md §6). Weak scaling (default): the global mesh has `world` x size^3 cells (1: n^3, 2: n x n x 2n,
    # 4: n x 2n x 2n, 8: (2n)^3 — the 256^3 / 16.8M-cell config at n = 128), cut into z-slabs of size^3 cells per rank. Strong
    # scaling: ONE size^3 mesh (default 256^3) cut into `world` z-slabs. Every rank builds only its slab (+2 layers per side) of
    # the box and takes its partition from that window; halo exchange over NCCL send/recv, BiCGSTAB scalars over NCCL allreduce.
    if strong:
        gshape = (n, n, n)
    else:
        gshape = {1: (n, n, n), 2: (n, n, 2 * n), 4: (n, 2 * n, 2 * n), 8: (2 * n, 2 * n, 2 * n)}.get(world, (n, n, n * world))
    # The domain grows with the mesh (the cells keep the size they have in the n^3 box of 0.004 x 0.001 x 0.001 m), so that every
    # rank of a weak-scaling run assembles the coefficients of the N = 1 workload. (Round 1 kept the domain fixed: at N = 2 the cells
    # were half as thick in z, the strongest couplings all pointed along z, the AMG levels had 20-30 % fewer entries and the greedy
    # restriction ran 3.5 x faster — a different problem, which is what the "efficiency 1.12 at N = 2" of SCALE_r01 measured.)
    if tet and not strong:
        # tets: a duct of `world` cubes along z, one n^3-lattice cube (6 n^3 tets) per rank. (Chosen when z-slabs of a wide lattice, e.g.
        # 150 x 150 x 19 per rank, still cost the restriction kernel ~240 ns per row; that was its ticket shape and is fixed —
        # profiles/r2_restriction_rows.txt — the duct stays as the weak-scaling shape: every rank has the N = 1 workload.)
        gshape = (n, n, n * world)
    box = dict(lx=0.004 * gshape[0] / n, ly=0.001 * gshape[1] / n, lz=0.001 * gshape[2] / n)
    if small:
        assert world == 1, "the reference's example meshes run on one GPU"
        mesh, settings, small_desc = small_mesh(args.mesh)
        gshape = None
    elif tet:
        # BASELINE.json configs[4] in kind: every hex of the lattice split into 6 tetrahedra (hex-major numbering), TVD-UMIST momentum.
        # The AMG smoother stays BiCGSTAB: with the reference's algorithm a Gauss-Seidel or Jacobi smoother panics on the coarse
        # levels (DESIGN.md §5). TVD makes a_u, a_v, a_w differ, so the three momentum solves run one after the other.
        if world == 1:
            arrays = syn.tet_box(*gshape, **box)
            mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
            syn.channel_bcs(mesh, fully_3d=True)
        else:
            ctx.comm_init(rank, world)
            arrays, cuts, off, n_global = syn.tet_slab_partition(*gshape, rank, world, **box)
            window = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
            syn.channel_bcs(window, fully_3d=True)
            mesh = window.partition_window(rank, world, cuts, off, n_global)
            del window
        del arrays
    elif world == 1:
        arrays = syn.hex_box(*gshape, **box)
        mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
        syn.channel_bcs(mesh)
        del arrays
    else:
        ctx.comm_init(rank, world)
        arrays, cuts, off, n_global = syn.slab_partition(*gshape, rank, world, **box)
        window = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
        syn.channel_bcs(window)
        mesh = window.partition_window(rank, world, cuts, off, n_global)
        del window, arrays
    cells = mesh.partition_info()["n_own"] if world > 1 else mesh.n_cells
    counts = mesh.counts()
    gcells = cells
    if world > 1:
        t = torch.tensor([cells], device="cuda", dtype=torch.int64)
        dist.all_reduce(t)
        gcells = int(t.item())
    if not small:
        settings = orc_b200.NumericalSettings(pressure_relaxation=P_RELAX)
        if tet:
            settings = orc_b200.NumericalSettings(pressure_relaxation=P_RELAX, momentum=orc_b200.MomentumDiscretization.TVD, limiter=orc_b200.TVD_UMIST)
    reset_every = 0 if small else args.reset_every      # the reference's own cases converge: no reset
    solver = orc_b200.SteadySolver(mesh, settings, RHO, MU, ctx)
    solver.set_fields(*(np.zeros(cells) for _ in range(4)))
    done = [0]

    def step():
        # The reference's algorithm does not converge on the synthetic boxes (oracle-confirmed at 64^3, DESIGN.md §5): its unguarded
        # BiCGSTAB / multigrid eventually produce NaN ("Multigrid diverged"). The work per iteration does not depend on that, so
        # the fields are put back to the start state every RESET_EVERY iterations; the reset (a few memsets) is inside the
        # timed region.
        if reset_every and done[0] and done[0] % reset_every == 0:   # reset_every: the enclosing function's current value
            solver.reset()
        done[0] += 1
        return solver.iterate(1)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # checker leg (N > 1, outside the timed region): the partitioned path on a small box against the oracle with its partition
    # emulation, and the partitioned vs the single-GPU result at 64^3 (what per-partition aggregates + lagged diagonals change)
    parity = None
    if world > 1 and not args.no_parity and not tet:
        parity = multi_gpu_parity(ctx, torch, dist, orc_b200, syn, local_rank, rank, world)

    def measure():
        for _ in range(args.warmup):
            step()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()
            time.sleep(0.3)
        barrier()
        # roofline legs, live in the timed region: (i) CUDA events around every SPMV_SAMPLE-th SpMV launch (the dominant kernel);
        # (ii) ONE event pair around each whole BiCGSTAB call (all 50 iterations of one solve on one level: 250 launches that run back
        # to back, unperturbed). The per-class breakdown comes from one extra, untimed step below.
        ctx.prof_config(classes=["spmv", "bicgstab"], sample_every=SPMV_SAMPLE)
        ctx.prof_enable(True)
        phases0 = solver.phase_ms()
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        rep = None
        for _ in range(args.steps):
            rep = step()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ctx.launch_count() - l0
        prof = ctx.prof_get()
        sp_ref_bytes = ctx.prof_ref_bytes("spmv")
        sp_detail = ctx.prof_spmv_detail()
        ctx.prof_enable(False)
        phases = {k: (v - phases0[k]) / args.steps for k, v in solver.phase_ms().items()}   # timed steps only
        batched = solver.batched
        fields = solver.get_fields() if args.dump_outputs else None    # before the untimed step below moves them on
        ctx.prof_config(classes=None, sample_every=1)
        ctx.prof_enable(True)
        step()                                  # untimed: device time per kernel class, events around every launch
        classes = ctx.prof_get()
        classes.pop("bicgstab", None)           # brackets the other classes
        ctx.prof_enable(False)
        clocks = sampler.finish() if sampler else None
        return ms, launches, prof, sp_ref_bytes, sp_detail, phases, batched, classes, clocks, rep, fields

    # The reference's algorithm is marginally unstable on the synthetic boxes (DESIGN.md §5): how many iterations a start from
    # rest survives depends on rounding (summation orders, the partitioning). If a run meets "Multigrid diverged" the whole
    # measurement starts over with an earlier reset of the fields; the restarts are reported in `config`.
    restarts = 0
    while True:
        try:
            ms, launches, prof, sp_ref_bytes, sp_detail, phases, batched, classes, clocks, rep, fields = measure()
            break
        except orc_b200.OrcError as e:
            if "diverged" not in str(e) or not reset_every or reset_every <= 2 or restarts >= 3:
                raise
            restarts += 1
            reset_every = max(2, reset_every - 2)
            ctx.prof_enable(False)
            ctx.prof_config(classes=None, sample_every=1)
            solver.reset()
            done[0] = 0
            if rank == 0:
                print(f"bench: '{e}' inside the measurement; restarting with the fields reset every {reset_every} iterations", file=sys.stderr, flush=True)
    if dist is not None:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fields)
    global_iters = args.steps / (ms * 1e-3)             # SIMPLE iterations of the GLOBAL mesh per second
    # weak scaling: one global problem of world x size^3 cells; `value` counts size^3-cell-equivalent iterations (= cell-updates/s
    # / size^3) so that it is a whole-job aggregate; strong scaling and N = 1: iterations of the one mesh.
    value = global_iters if (strong or small) else world * global_iters

    # ---- e2e: the reference-facing call (solve_steady through the C ABI) with HOST buffers, copies inside the timed region
    if args.no_e2e:
        e2e_global = None
    else:
        e2e_global = run_e2e(args, world, dist, torch, orc_b200, mesh, settings, solver, ctx, barrier)
    e2e_value = None if e2e_global is None else (e2e_global if (strong or small) else world * e2e_global)

    small_runs = None
    if rank == 0 and world == 1 and not small and not tet and not args.no_small:
        small_runs = {k: time_small(k, ctx, torch) for k in ("couette", "channel")}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    sp_ms, sp_bytes, sp_count = prof["spmv"]
    achieved = sp_bytes / (sp_ms * 1e-3) / 1e9 if sp_ms > 0 else 0.0
    achieved_ref = sp_ref_bytes / (sp_ms * 1e-3) / 1e9 if sp_ms > 0 else 0.0
    by_matrix = [{"rows": r, "systems_per_launch": k, "entries_per_row": round(e[3] / e[2] / r, 1), "launches_timed": e[2],
                  "us_per_launch": round(1e3 * e[0] / e[2], 1), "GB/s": round(e[1] / (e[0] * 1e-3) / 1e9, 1),
                  "frac": round(e[1] / (e[0] * 1e-3) / 1e9 / peak, 3) if peak else None}
                 for (r, k), e in sorted(pooled(sp_detail, peak, {1: 1, 3: 3}).items(), key=lambda kv: (-kv[0][0], kv[0][1]))]
    bicg_by_level = [{"rows": r, "systems": k, "entries_per_row": round(e[3] / e[2] / r, 1), "solves_timed": e[2],
                      "ms_per_solve": round(e[0] / e[2], 3), "GB/s": round(e[1] / (e[0] * 1e-3) / 1e9, 1),
                      "frac": round(e[1] / (e[0] * 1e-3) / 1e9 / peak, 3) if peak else None}
                     for (r, k), e in sorted(pooled(sp_detail, peak, {5: 1, 7: 3}).items(), key=lambda kv: (-kv[0][0], kv[0][1]))]
    bi_ms, bi_bytes, bi_count = prof["bicgstab"]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    if os.path.exists(tpath) and gshape:
        with open(tpath) as f:
            traffic = json.load(f).get(str(n))
    levels = solver.level_sizes()
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not tet and not small:   # the CPU sample is the hex channel
        m = args.cpu_sample
        ccells, cdt, cph = oracle_run(m)
        cpu = {"value": ccells / cdt / cells, "unit": "iter/s", "cores": 1, "kind": "port",
               "sample": f"1 SIMPLE iteration on a {m}^3 hex channel ({ccells} cells, {cdt:.1f} s), same settings, C++ restatement of the "
                         f"reference path (oracle/), single thread like ORC; cell-update rate expressed in iterations of the {cells}-cell "
                         f"workload (`bench.py --impl reference` times the full {n}^3 mesh instead)",
               "phases_s": cph}
    # SURVEY.md §8d byte model of the WHOLE SIMPLE iteration as the reference performs it: 4 solves x 50 BiCGSTAB iterations on
    # every level (multiplicity 1, 2, 2, 1: pre- and post-smoothing), one iteration = 24 nnz_l + 152 n_l bytes. This is the
    # figure the "60 % of HBM roofline" target of BASELINE.json is stated in (SURVEY: 0.37 MB per cell per iteration for hexes).
    mult = [1, 2, 2, 1]
    per_set = sum(m * (24.0 * z + 152.0 * r) for m, (r, z) in zip(mult, levels)) if len(levels) == 4 else None
    step_model = None
    if per_set:
        model_bytes = 4 * 50 * per_set
        eff = model_bytes / (ms / args.steps * 1e-3) / 1e9
        step_model = {"bytes_per_iteration_model": model_bytes, "bytes_per_cell": model_bytes / cells, "effective_GB/s": eff,
                      "frac_of_measured_peak": eff / peak if peak else None, "frac_of_nominal_8TB/s": eff / 8000.0,
                      "note": "whole-iteration throughput in the reference's own byte model (SURVEY.md §8d): 4 solves x 50 BiCGSTAB iterations x "
                              "levels (1,2,2,1) x (24 nnz + 152 n) bytes, divided by the measured time per iteration — set-up, assembly and "
                              "launch gaps included in the time, the lockstep saving counted as throughput"}
    # assembly phases against the HBM roofline (SURVEY.md §8d bytes): the phase times are CUDA-event pairs around each phase of
    # every timed iteration (orc_steady_phase_ms)
    N_, F_, Z_ = counts["cells"], counts["faces"], counts["nnz"]
    asm_bytes = {"momentum_assembly": 32.0 * Z_ + 160.0 * N_ + 68.0 * F_, "pressure_assembly": 8.0 * Z_ + 120.0 * N_ + 68.0 * F_,
                 "correction": 96.0 * N_ + 44.0 * F_}
    asm = {k: {"ms": phases[k], "GB/s": b / (phases[k] * 1e-3) / 1e9 if phases[k] > 0 else None,
               "frac": b / (phases[k] * 1e-3) / 1e9 / peak if phases[k] > 0 else None, "algorithmic_bytes": b}
           for k, b in asm_bytes.items()}
    asm["note"] = ("SURVEY.md §8d bytes (momentum 32 nnz + 160 N + 68 F incl. grad p, pressure 8 nnz + 120 N + 68 F, correction 96 N + 44 F) / "
                   "in-situ phase time; momentum assembly runs in EXACT mode (the reference's in-place diagonal recurrence, Q2)")
    if small:
        workload = small_desc
    elif tet:
        workload = f"synthetic tet box: {'x'.join(str(s) for s in gshape)} lattice x 6 tets ({gcells / 1e6:.2f}M cells), SIMPLE + AMG-BiCGSTAB fp64, TVD-UMIST"
    else:
        workload = workload_name(gshape)
    line = {
        "metric": METRIC, "value": value, "unit": "iter/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "global_iters_per_s": global_iters,
        "config": {"workload": workload,
                   "solver": "Gauss-Seidel x50" if args.mesh == "couette" else "Multigrid(BiCGSTAB x50, 3 levels, Jacobi precond)",
                   "momentum": "TVD-UMIST" if tet else ("TVD-QUICK" if args.mesh == "channel" else "CD1"),
                   "velocity_interpolation": "RhieChow", "pressure_interpolation": "SecondOrder", "assembly_mode": "exact",
                   "pressure_relaxation": settings.pressure_relaxation, "fields_reset_every": reset_every, "divergence_restarts": restarts,
                   "momentum_solves": ("u, v, w in lockstep: a_u == a_v == a_w bit for bit (checked on the device every iteration), one matrix "
                                       "pass and one AMG hierarchy for the three systems; every system's arithmetic is that of its own solve"
                                       if batched else "three sequential solves"),
                   "parallelism": "1 GPU" if world == 1 else f"{world} z-slabs of {cells} cells, NCCL halo send/recv + allreduce, per-partition AMG",
                   "global_mesh": list(gshape) if gshape else None, "domain_m": [box["lx"], box["ly"], box["lz"]] if gshape else None, "global_cells": gcells, "cells_per_gpu": cells,
                   "value_counts": ("SIMPLE iterations of the global mesh per second" if (strong or small or world == 1) else
                                    f"weak scaling: {world} x (SIMPLE iterations of the {gcells}-cell global mesh per second) = iterations of one GPU's "
                                    f"{cells}-cell share; global_iters_per_s is the unscaled figure"),
                   "l2": "inputs larger than L2 (fine matrix 175 MB at 128^3, 5 matrices + coarse levels); no flush needed" if not small else
                         "small mesh: everything is L2 resident (launch-bound case)",
                   "amg_levels_rows_nnz": levels},
        "cell_updates_per_s": global_iters * gcells,
        "roofline": {"bound": "hbm", "kernel": "k_spmv (all fused epilogues, all AMG levels)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_src, "launches": sp_count,
                     "bytes_per_launch_model": "12*nnz_l + 4*n_l + 16*K*n_l of the level it runs on (K = systems per launch: 3 for the lockstep momentum solves, 1 for p')",
                     "timed": f"CUDA events around every {SPMV_SAMPLE}th SpMV launch inside the timed region ({sp_count} launches)",
                     "by_matrix": by_matrix,
                     "by_matrix_note": "the same timed launches per AMG level (rows) and systems per launch; the short-row R / R^T products are omitted",
                     "achieved_in_reference_units": achieved_ref,
                     "reference_units_note": "same launches counted as the reference's SpMVs (12*nnz + 20*n each): a lockstep launch does three of them in one matrix pass",
                     "time_share_of_step": classes["spmv"][0] / max(1e-9, sum(v[0] for v in classes.values())),
                     "bicgstab": {"achieved": bi_bytes / (bi_ms * 1e-3) / 1e9 if bi_ms > 0 else None,
                                  "frac": bi_bytes / (bi_ms * 1e-3) / 1e9 / peak if bi_ms > 0 else None, "solves_timed": bi_count,
                                  "ms_per_step": bi_ms / args.steps, "by_level": bicg_by_level,
                                  "note": "ONE event pair around each whole BiCGSTAB call in the timed region (50 iterations x 5 launches, back to back): "
                                          "algorithmic bytes = 50 x (2 SpMV + 104 K n of vector passes) + the initial residual"},
                     "assembly": asm,
                     "whole_iteration": step_model},
        "kernel_classes_ms_per_step": {k: v[0] for k, v in classes.items()},
        "kernel_classes_note": "device time per kernel class of ONE extra untimed step with events around every launch",
        "phases_ms_per_step": phases,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "iter/s", "global_iters_per_s": e2e_global, "h2d_bytes_per_step": 32 * cells, "d2h_bytes_per_step": 32 * cells,
                "call": "orc_solve_steady(iteration_count=1) per step, pinned host u/v/w/p", "steps": args.e2e_steps},
        "small_meshes": small_runs,
        "partition_parity": parity,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "last_report": rep,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=int(os.environ.get("ORC_BENCH_N", "0")), help="edge of the box (default 128; 256 with --scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: size^3 cells PER GPU; strong: one size^3 mesh cut into N slabs")
    ap.add_argument("--cpu-sample", type=int, default=64, help="edge of the hex box the CPU baseline is timed on")
    ap.add_argument("--mesh", default="hex", choices=["hex", "tet", "couette", "channel"],
                    help="hex: the headline channel; tet: size^3 lattice split into 6 tets per hex, TVD-UMIST (BASELINE.json configs[4] in kind); "
                         "couette / channel: the reference's own example meshes (configs[0], configs[1])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-small", action="store_true", help="skip the two example-mesh legs of the default run")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the partition parity check that runs before the timed region")
    ap.add_argument("--reset-every", type=int, default=RESET_EVERY, help="SIMPLE iterations between resets of the fields (the reference's "
                    "algorithm diverges on the synthetic boxes after a few iterations; sooner on larger ones)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs under ncu)")
    ap.add_argument("--e2e-steps", type=int, default=3, help="calls timed in the end-to-end leg (each copies the fields in and out)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="one GPU: write u, v, w, p after the last timed step to DIR/<name>.npy "
                    "(float64; a fixed, seeded sample of cells when the four fields exceed 64 MB, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.e2e_steps < 1:
        ap.error("--steps and --e2e-steps must be at least 1, --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        ap.error("--dump-outputs writes the fields of the GPU path (--impl ours) on one GPU only")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
