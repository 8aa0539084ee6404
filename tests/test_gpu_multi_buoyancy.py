"""Boussinesq coupling on 2 and 4 GPUs (skipped with fewer): the partitioned coupled iterations of tests/mgpu_buoyancy_worker.py
against the coupled model with the oracle's partition emulation, and the zone fluxes summed over the ranks against one GPU."""
import json
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_worker(world):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_buoyancy_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    lines = [l for l in out.stdout.splitlines() if l.startswith("MGPU_RESULT ")]
    assert lines, out.stdout[-2000:] + out.stderr[-4000:]
    return json.loads(lines[-1][len("MGPU_RESULT "):])


@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_coupled_iterations(world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    res = run_worker(world)
    print(res)
    assert res["world"] == world and res["finite"]
    assert max(res["vs_oracle_partitioned"].values()) <= 1e-8, res   # the bound tests/mgpu_check.py uses for the flow
    assert res["flux_ok"], res["flux"]
