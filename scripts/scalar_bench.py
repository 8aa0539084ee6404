"""Passive scalar transport on the 128^3 bench mesh (one B200): device time of the face-flux kernel and of the assembly kernel
(CUDA events of the context's kernel profiler, assembly class), and host time of one whole solve_scalar call with the default
settings (CD1, Rhie-Chow, Multigrid; the call ends in a device synchronise). Algorithmic bytes per launch come from the model
below (every array the kernel must touch, read or written once); the share of peak is bytes / time over MEASURED_PEAKS.json
hbm_gbs (the data sheet's 7.7 TB/s when that file is absent). Prints one JSON object and writes it to --out if given. The card's name and power limit are read in the same run.

    python scripts/scalar_bench.py --out profiles/scalar_bench_128cubed_1gpu.json
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

RHO, MU, GAMMA = 1000.0, 1e-3, 2e-3


def card():
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    vals = [x.strip() for x in out.stdout.strip().split(",")]
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"query_failed": out.stderr.strip()}


def peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    return 7700.0, "HBM3e bandwidth of the B200 data sheet (MEASURED_PEAKS.json absent): a bound, not a reached rate"


def traffic(counts, tvd):
    """Algorithmic bytes of one launch of each kernel (index arrays int32, values fp64)."""
    N, F, S, nnz = counts["cells"], counts["faces"], counts["cell_faces"], counts["nnz"]
    # k_scalar_face_flux (Rhie-Chow): per face c0, c1, zone (12 B) + normal (24 B) + F out (8 B); per cell u, v, w, p, grad p,
    # volume, centroid, du, dv, dw (14 doubles)
    flux = F * (12 + 24 + 8) + N * 14 * 8
    # k_scalar_transport: cf_ptr, per slot cf_face + cf_slot; per face c0, c1, zone, area, F; per cell centroid, diag index, phi (+ grad
    # phi for TVD), b out; the matrix values out
    asm = 4 * (N + 1) + 8 * S + F * (12 + 16) + N * (24 + 4 + 8 + (24 if tvd else 0) + 8) + 8 * nnz
    return {"k_scalar_face_flux": flux, "k_scalar_transport": asm}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--simple", type=int, default=3, help="SIMPLE iterations before the scalar")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("scalar_bench.py measures on the GPU: none found")
    ctx = orc_b200.default_context(0)
    mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(a.n, a.n, a.n)))
    syn.channel_bcs(mesh)
    mesh.set_zone_scalar("INLET", orc_b200.ScalarCondition.Fixed, 1.0)
    mesh.set_zone_scalar("WALL", orc_b200.ScalarCondition.Fixed, 0.0)
    counts = mesh.counts()
    s = orc_b200.NumericalSettings()
    st = orc_b200.SteadySolver(mesh, s, RHO, MU, ctx)
    st.set_fields(*(np.zeros(counts["cells"]) for _ in range(4)))
    st.iterate(a.simple)
    phi = st.solve_scalar(GAMMA, None, 1)   # warm-up: every shape and the AMG set-up once
    # kernel times: the assembly class of the profiler holds exactly the face-flux launch for sweeps = 0, and the face-flux launch plus
    # one k_scalar_transport per sweep otherwise
    ctx.prof_config(classes=["assembly"])
    ctx.prof_enable(True)
    for _ in range(a.reps):
        st.solve_scalar(GAMMA, phi, 0)
    flux_ms, _, flux_n = ctx.prof_get()["assembly"]
    ctx.prof_enable(False)
    ctx.prof_enable(True)
    sweeps = 4
    for _ in range(a.reps):
        st.solve_scalar(GAMMA, phi, sweeps)
    both_ms, _, both_n = ctx.prof_get()["assembly"]
    ctx.prof_enable(False)
    assert flux_n == a.reps and both_n == a.reps * (1 + sweeps), (flux_n, both_n)
    t_flux = flux_ms / a.reps
    t_asm = (both_ms - t_flux * a.reps) / (a.reps * sweeps)
    # one whole solve (face flux + one CD1 sweep with the Multigrid solve, phi to and from the host)
    walls = []
    for _ in range(5):
        t0 = time.perf_counter()
        st.solve_scalar(GAMMA, None, 1)
        walls.append((time.perf_counter() - t0) * 1e3)
    peak, peak_src = peak_gbs()
    by = traffic(counts, tvd=False)
    kernels = {}
    for name, ms in (("k_scalar_face_flux", t_flux), ("k_scalar_transport", t_asm)):
        gbs = by[name] / (ms * 1e-3) / 1e9
        kernels[name] = {"ms": ms, "algorithmic_bytes": by[name], "achieved_gbs": gbs, "share_of_peak": (gbs / peak) if peak else None}
    res = {"workload": f"passive scalar on the {a.n}^3 hex channel after {a.simple} SIMPLE iterations, default settings (CD1, Rhie-Chow, "
                       f"Multigrid/BiCGSTAB x50)", "cells": counts["cells"], "faces": counts["faces"], "nnz": counts["nnz"],
           "kernels": kernels, "solve_ms_host_clock": {"median": float(np.median(walls)), "min": float(np.min(walls)), "runs": walls},
           "phi_range": [float(phi.min()), float(phi.max())], "peak_gbs": peak, "peak_source": peak_src, "card": card(),
           "timing": f"CUDA events around each launch, {a.reps} calls each; whole solve: host clock around a synchronising call"}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
