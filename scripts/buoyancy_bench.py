"""Buoyancy coupling on the 128^3 bench channel (one B200): ms per SIMPLE iteration of an uncoupled handle and of a handle coupled with
one scalar sweep per iteration (gravity across the walls, the WALL zone at phi = 0 and the INLET at phi = 1),
alternated block by block in the same process; then, in a separate torch.profiler pass, the device time of
k_momentum_source_buoyancy against its algorithmic traffic of 88 B per cell (reads b x3, b_di x3, phi, V; writes b x3). Both
handles are reset every RESET_EVERY iterations as bench.py does: the synthetic channel diverges from rest (DESIGN.md §5). The
card's name and power limit are read in the same run. Prints one JSON object and writes it to --out if given.

    python scripts/buoyancy_bench.py --out profiles/buoyancy_bench_128cubed_1gpu.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import orc_b200  # noqa: E402
from orc_b200 import synthetic as syn  # noqa: E402

RHO, MU, GAMMA, BETA, PHI_REF, G = 1000.0, 1e-3, 2e-3, 1e-3, 0.5, (0.0, -9.81, 0.0)
P_RELAX, RESET_EVERY = 1e-4, 6   # bench.py's settings


def card():
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    vals = [x.strip() for x in out.stdout.strip().split(",")]
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"query_failed": out.stderr.strip()}


def run_block(st, iterations, done):
    """`iterations` iterate(1) calls with a reset every RESET_EVERY iterations; -> ms per iteration (host clock, synchronised)"""
    t0 = time.perf_counter()
    for _ in range(iterations):
        if done[0] and done[0] % RESET_EVERY == 0:
            st.reset()
        st.iterate(1)
        done[0] += 1
    st.ctx.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iterations


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--blocks", type=int, default=5, help="alternated timing blocks per handle")
    ap.add_argument("--block-iterations", type=int, default=12)
    ap.add_argument("--profile-iterations", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("buoyancy_bench.py measures on the GPU: none found")
    ctx = orc_b200.default_context(0)
    mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(a.n, a.n, a.n)))
    syn.channel_bcs(mesh)
    mesh.set_zone_scalar("INLET", orc_b200.ScalarCondition.Fixed, 1.0)
    mesh.set_zone_scalar("WALL", orc_b200.ScalarCondition.Fixed, 0.0)
    n = mesh.n_cells
    s = orc_b200.NumericalSettings(pressure_relaxation=P_RELAX)
    handles = {}
    for name in ("uncoupled", "coupled"):
        st = orc_b200.SteadySolver(mesh, s, RHO, MU, ctx)
        st.set_fields(*(np.zeros(n) for _ in range(4)))
        if name == "coupled":
            st.couple_scalar(GAMMA, BETA, PHI_REF, G, 1)
        handles[name] = (st, [0])
        run_block(st, 2, handles[name][1])   # warm-up: every shape and the AMG set-up
    ms = {"uncoupled": [], "coupled": []}
    for _ in range(a.blocks):
        for name in ("uncoupled", "coupled"):
            st, done = handles[name]
            ms[name].append(run_block(st, a.block_iterations, done))
    phi = handles["coupled"][0].get_scalar()
    # the kernel, in a profiler pass of its own
    from torch.profiler import ProfilerActivity, profile
    st, done = handles["coupled"]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_block(st, a.profile_iterations, done)
    k = [e for e in prof.key_averages() if e.key.split("(")[0].endswith("k_momentum_source_buoyancy")]
    assert k and k[0].count == a.profile_iterations, [(e.key, e.count) for e in prof.key_averages()][:40]
    total = getattr(k[0], "device_time_total", None)
    dev_us = (total if total is not None else k[0].cuda_time_total) / k[0].count
    bytes_per_launch = 88 * n
    res = {"workload": f"{a.n}^3 hex channel, bench.py settings (CD1, Rhie-Chow, Multigrid/BiCGSTAB x50, pressure relaxation {P_RELAX}), "
                       f"fields reset every {RESET_EVERY} iterations; coupled: gamma {GAMMA}, beta {BETA}, phi_ref {PHI_REF}, g {G}, "
                       f"1 sweep, INLET phi = 1, WALL phi = 0",
           "cells": n,
           "ms_per_iteration": {name: {"median": float(np.median(v)), "min": float(np.min(v)), "blocks": v} for name, v in ms.items()},
           "coupled_over_uncoupled": float(np.median(ms["coupled"]) / np.median(ms["uncoupled"])),
           "k_momentum_source_buoyancy": {"us": dev_us, "launches": k[0].count, "algorithmic_bytes": bytes_per_launch,
                                          "achieved_gbs": bytes_per_launch / (dev_us * 1e-6) / 1e9},
           "phi_range": [float(phi.min()), float(phi.max())], "card": card(),
           "timing": f"host clock around {a.block_iterations} synchronised iterations per block, {a.blocks} blocks per handle, "
                     "alternated; kernel: torch.profiler device time, averaged over its launches, in a separate pass"}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
