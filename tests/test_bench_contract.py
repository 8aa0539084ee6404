"""bench.py's command-line contract: the reference arm (the oracle timed on the host cores) prints ONE JSON line with the keys
its readers expect, our own arm fails loudly on a machine without a CUDA device — the product path has no CPU fallback — and
--dump-outputs writes the fields of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--size", "10", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "SIMPLE iters/s" and d["unit"] == "iter/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["steps_timed"] == 2 and d["warmup_done"] == 1
    assert d["value"] > 0 and abs(d["value"] * d["ms_per_step"] / 1e3 - 1.0) < 1e-9 and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and cb["unit"] == "iter/s" and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    assert set(d["phases_ms_per_step"]) == {"momentum_assembly", "momentum_solves", "pressure_assembly", "pressure_solve", "correction"}


def test_reference_arm_runs_on_rank_zero_only():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--size", "10", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and r.stdout.strip() == "", (r.returncode, r.stdout[-500:], r.stderr[-500:])


def test_our_arm_fails_loudly_without_a_gpu():
    import orc_b200
    try:
        orc_b200.default_context(0)
    except orc_b200.OrcError:
        pass
    else:
        pytest.skip("a CUDA device is present")
    r = _run("--size", "8", "--steps", "1", "--warmup", "0", "--no-e2e", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "no CUDA device" in r.stderr or "NVIDIA" in r.stderr            # the library's own refusal, or torch's on the way to it
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())     # no result line of any kind


def test_dump_outputs_keeps_one_seeded_sample_within_64_mb(tmp_path):
    """Fields of the 128^3 workload's size (4 x 16.8 MB in float64) are cut to the same seeded sample of cells in every field and
    in every call, listed in cell_index.npy, all float64 and at most 64 MB together."""
    import bench
    n = 128 ** 3
    fields = [np.arange(n, dtype=np.float64) * (k + 1) for k in range(4)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), fields)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["cell_index.npy", "p.npy", "u.npy", "v.npy", "w.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    idx = np.load(tmp_path / "a" / "cell_index.npy")
    assert idx.dtype == np.float64 and idx.size == bench.DUMP_SAMPLE and np.all(np.diff(idx) > 0) and idx[-1] < n
    for k, name in enumerate("uvwp"):
        a = np.load(tmp_path / "a" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, idx * (k + 1)), name
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{name}.npy")), name


@pytest.mark.gpu
def test_dump_outputs_are_the_fields_after_the_last_timed_step(ctx, tmp_path):
    """--dump-outputs on a 16^3 box with 1 warm-up and 2 timed steps (before the first reset of the fields) writes the fields of
    3 SIMPLE iterations from rest: bit for bit, since on 4096 cells the default reduction mode takes the reference order. The
    end-to-end leg that runs afterwards times the --e2e-steps calls it is given and leaves the dump alone."""
    import bench
    import orc_b200
    from orc_b200 import synthetic as syn
    r = _run("--size", "16", "--steps", "2", "--warmup", "1", "--e2e-steps", "2", "--no-cpu-baseline", "--no-small", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and d["warmup"] == 1 and d["e2e"]["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["p.npy", "u.npy", "v.npy", "w.npy"]
    mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(16, 16, 16)))
    syn.channel_bcs(mesh)
    solver = orc_b200.SteadySolver(mesh, orc_b200.NumericalSettings(pressure_relaxation=bench.P_RELAX), bench.RHO, bench.MU, ctx)
    solver.set_fields(*(np.zeros(mesh.n_cells) for _ in range(4)))
    solver.iterate(3)
    for name, f in zip("uvwp", solver.get_fields()):
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, f), name
    solver.close()
