"""Run files written from a partition mesh (io.write_data): each rank writes the lines of its owned cells, and the rank files
concatenated in rank order are the whole mesh's file byte for byte. Host-only: partitions and their geometry are built on the CPU."""
import numpy as np
import pytest

import orc_b200
from orc_b200 import io as oio
from orc_b200 import synthetic as syn


def _fields(n, seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(n) * s for s in (1e-3, 2e-4, 3e-5, 1e2)]


def _rank_meshes(kind, shape, nranks, window):
    """[(partition mesh, g0, g1)] of every rank: cut from the global mesh, or built from a z-slab window (no global mesh)."""
    out = []
    for r in range(nranks):
        if window:
            slab = syn.slab_partition if kind == "hex" else syn.tet_slab_partition
            arrays, cuts, off, n_global = slab(*shape, r, nranks)
            part = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays)).partition_window(r, nranks, cuts, off, n_global)
        else:
            box = syn.hex_box if kind == "hex" else syn.tet_box
            part = orc_b200.Mesh.from_arrays(*syn.mesh_args(box(*shape))).partition(r, nranks)
        info = part.partition_info()
        out.append((part, info["g0"], info["g1"]))
    return out


@pytest.mark.parametrize("kind,shape", [("hex", (6, 4, 8)), ("tet", (3, 3, 4))])
@pytest.mark.parametrize("nranks", [1, 2, 3, 4])
@pytest.mark.parametrize("window", [False, True])
@pytest.mark.parametrize("precision", [None, 5])
def test_write_data_rank_files_concatenate_to_the_whole_file(tmp_path, kind, shape, nranks, window, precision):
    box = syn.hex_box if kind == "hex" else syn.tet_box
    whole = orc_b200.Mesh.from_arrays(*syn.mesh_args(box(*shape)))
    n = whole.n_cells
    u, v, w, p = _fields(n, nranks)
    oio.write_data(whole, u, v, w, p, str(tmp_path / "whole.csv"), precision)
    parts = _rank_meshes(kind, shape, nranks, window)
    assert parts[0][1] == 0 and parts[-1][2] == n and all(a[2] == b[1] for a, b in zip(parts, parts[1:]))
    text = b""
    for r, (part, g0, g1) in enumerate(parts):
        path = tmp_path / f"rank{r}.csv"
        oio.write_data(part, u[g0:g1], v[g0:g1], w[g0:g1], p[g0:g1], str(path), precision)
        text += path.read_bytes()
    assert text == (tmp_path / "whole.csv").read_bytes()


def test_write_data_refuses_fields_that_do_not_fit_the_owned_cells(tmp_path):
    part = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(6, 4, 8))).partition(0, 2)
    n_local = part.n_cells   # halo cells included: the length a caller could mistake for the right one
    assert n_local > part.partition_info()["n_own"]
    with pytest.raises(ValueError):
        oio.write_data(part, *(np.zeros(n_local) for _ in range(4)), str(tmp_path / "x.csv"))
