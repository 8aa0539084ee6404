"""Multi-GPU worker for the Boussinesq coupling (run under torchrun, one rank per GPU; used by tests/test_gpu_multi_buoyancy.py):
coupled iterations on a partitioned hex channel against the coupled model with the oracle's partition emulation, and the zone
fluxes of a partitioned handle against one GPU on the same fields. Prints one JSON line on rank 0."""
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
from orc_b200 import synthetic as syn  # noqa: E402
from cases import smooth_fields  # noqa: E402
from mgpu_worker import gather_owned  # noqa: E402

RHO, MU, GAMMA, BETA, PHI_REF, G = 1000.0, 1e-3, 2e-3, 0.0125, 0.5, (0.0, -10.0, 0.0)
FIXED = orc_b200.ScalarCondition.Fixed
ZONES = ("INLET", "OUTLET", "WALL", "SYM")


def main():
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=device)
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = orc_b200.Context(local_rank)
    ctx.comm_init()
    single = orc_b200.Context(local_rank)   # no communicator: the single-GPU path
    arrays = syn.hex_box(12, 8, 4 * world)
    gmesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(gmesh)
    gmesh.set_zone_scalar("INLET", FIXED, 1.0)
    gmesh.set_zone_scalar("WALL", FIXED, 0.0)
    n = gmesh.n_cells
    part = gmesh.partition(rank, world)   # inherits the zones' scalar conditions
    info = part.partition_info()
    l2g = part.partition_maps()["local_to_global"]
    own = slice(info["n_lo"], info["n_lo"] + info["n_own"])
    s = orc_b200.NumericalSettings()
    out = {"world": world, "cells": n}

    # 1. three coupled iterations from rest, partitioned
    st = orc_b200.SteadySolver(part, s, RHO, MU, ctx)
    st.set_fields(*(np.zeros(info["n_own"]) for _ in range(4)))
    st.couple_scalar(GAMMA, BETA, PHI_REF, G, 1)
    st.iterate(3)
    got = [gather_owned(f, info, n, device) for f in (*st.get_fields(), st.get_scalar())]
    st.close()
    cuts = [None] * world
    dist.all_gather_object(cuts, info["g0"])

    # 2. the zone fluxes of one state (smooth fields, random phi, fresh diagonals): partitioned and on one GPU
    u, v, w, p = smooth_fields(gmesh.export())
    phi = np.random.default_rng(5).uniform(0.0, 1.0, n)

    def fluxes(mesh, c, fields, ph):
        h = orc_b200.SteadySolver(mesh, s, RHO, MU, c)
        h.set_fields(*fields)
        h.set_scalar(ph)
        h.couple_scalar(GAMMA, BETA, PHI_REF, G, 1)
        r = {z: h.scalar_zone_flux(z) for z in ZONES}
        h.close()
        return r

    part_flux = fluxes(part, ctx, [f[l2g][own] for f in (u, v, w, p)], phi[l2g][own])
    one_flux = fluxes(gmesh, single, [u, v, w, p], phi)
    if rank == 0:
        from oracle import pyoracle as po
        import buoyancy_model as bm
        import fast_simple as fs
        import scalar_oracle as so
        om = po.Mesh.from_arrays(*syn.mesh_args(arrays))
        syn.channel_bcs(om)
        bcs = so.ScalarBcs(om)
        bcs.set("INLET", so.FIXED, 1.0)
        bcs.set("WALL", so.FIXED, 0.0)
        os_ = po.Settings()
        z = np.zeros(n)
        po.set_partition(cuts + [n])
        try:
            rec = bm.coupled_iterations(om, bcs, os_, RHO, MU, (z, z, z, z), z, 3, fs.oracle_solve(os_), GAMMA, BETA, PHI_REF, G)[-1]
        finally:
            po.set_partition(None)
        want = [rec[k] for k in ("u", "v", "w", "p", "phi")]
        vel = np.sqrt(sum(np.linalg.norm(b) ** 2 for b in want[:3]))
        out["vs_oracle_partitioned"] = {k: float(np.linalg.norm(a - b) / (vel if k in "uvw" else np.linalg.norm(b)))
                                        for k, a, b in zip(("u", "v", "w", "p", "phi"), got, want)}
        out["finite"] = bool(all(np.isfinite(a).all() for a in got))
        # gamma_m * sum |terms| per zone and component, the terms from the model on the same state (bit-identical per face)
        state = fs.State(om, MU)
        flux_ok, margins = True, {}
        for zname in ZONES:
            terms = bm.zone_terms(om, bcs, dict(u=u, v=v, w=w, p=p, phi=phi), state, os_, GAMMA, RHO, zname)
            m = max(len(terms), 1) + world
            gam = m * 2.0 ** -53 / (1 - m * 2.0 ** -53)
            for q in range(2):
                bound = gam * np.abs(terms[:, q]).sum()
                diff = abs(part_flux[zname][q] - one_flux[zname][q])
                flux_ok = flux_ok and diff <= bound
                margins[f"{zname}_{q}"] = [diff, bound]
        out["flux_ok"] = bool(flux_ok)
        out["flux"] = {"partitioned": part_flux, "one_gpu": one_flux, "diff_and_bound": margins}
        print("MGPU_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
