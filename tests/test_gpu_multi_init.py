"""Multi-GPU flow initialisation, Jacobi solves, gradients and run files on partition meshes (needs >= `world` GPUs on the box;
skipped otherwise): tests/mgpu_init_worker.py runs the cases under torchrun and reports one JSON line. "Single" is one GPU with
the whole mesh and ReductionMode.Fast."""
import json
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    import torch
    return torch.cuda.device_count()


def run_worker(world):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_init_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    lines = [l for l in out.stdout.splitlines() if l.startswith("MGPU_RESULT ")]
    assert lines, out.stdout[-2000:] + out.stderr[-4000:]
    return json.loads(lines[-1][len("MGPU_RESULT "):])


@pytest.fixture(scope="module", params=[2, 4])
def result(request):
    world = request.param
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    res = run_worker(world)
    assert res["world"] == world
    print(json.dumps(res))
    return res


@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_initialize_flow_on_partitions(result, kind):
    r = result[f"init_{kind}"]
    # the Laplace pressure field by distributed Jacobi: the iterates are the single GPU's bit for bit (and the oracle's)
    assert r["flow_p_equal_single"] and r["flow_p_equal_oracle"], r
    # the velocity rounds of BiCGSTAB: only the summation order of the dot products differs
    assert r["flow_uvw_vs_single"] <= 1e-8 and r["flow_uvw_vs_oracle"] <= 1e-8, r
    assert r["lockstep"], r


@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_initialize_flow_new_on_partitions(result, kind):
    r = result[f"init_{kind}"]
    assert r["new_pressure_p_equal"], r
    print(f"VelocityOnly, {kind}, world {result['world']}: distance to single = {r['new_velocity_vs_single']:.3e}")
    assert r["new_velocity_nonzero"] and r["new_velocity_vs_single"] <= 1e-9, r


@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_windowed_partitions_initialise_like_cut_partitions(result, kind):
    assert result[f"init_{kind}"]["window_equals_cut"]


def test_boundary_condition_count_wraps_like_the_whole_mesh(result):
    w, n = result["wrap_69"], result["wrap_68"]
    assert w["faces"] == 196608 == 3 * 65536 and w["constraint"] == 0 and n["constraint"] == 1, (w, n)
    assert w["equal_single"] and w["p_nonzero"], w
    assert n["equal_single"] and not n["p_nonzero"], n


def test_jacobi_as_the_loop_solver(result):
    assert result["jacobi_linear_weighted_equal_single"]
    par = result["jacobi_oracle_partition_parity"]
    print("Jacobi, partitioned GPU run vs oracle:", par)
    assert max(par["vs_oracle_partitioned"].values()) <= 1e-8, par


def test_jacobi_divergence_is_reported_alike_on_every_rank(result):
    from orc_b200 import _lib
    d = result["divergence"]
    assert d["codes"] == [_lib.E_JACOBI_DIVERGED] * result["world"], d
    assert all(d["next_call_ok"]), d


def test_gradients_of_partitions(result):
    r = result["gradients_and_files"]
    assert r["equal_single_0"] and r["equal_single_2"], r
    assert r["window_equals_cut"], r


def test_rank_run_files_concatenate_to_the_single_gpu_files(result):
    r = result["gradients_and_files"]
    assert r["data_file_equal"] and r["grad_file_equal"], r
