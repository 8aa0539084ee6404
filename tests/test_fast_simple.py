"""tests/fast_simple.py, the composed model of a fast-mode SIMPLE iteration, is the reference's iteration:

* with the oracle's own solver in place of fast_model's, it is oracle.solve_steady bit for bit (fields and all nine report columns)
  on a hex channel, a tet box with TVD-UMIST and the reference's channel_flow.msh, with Multigrid, BiCGSTAB and Jacobi;
* with fast_model's solves (5 inner iterations, where the solves still converge) it stays within 1e-6 of the oracle, the bar of
  test_gpu_scale.test_one_simple_iteration_at_size;
* a case that diverges fails with the same error in the same iteration as the oracle.

No GPU code runs here; tests/test_gpu_fast_simple.py pins the GPU to this model."""
import numpy as np
import pytest

import bench
import fast_model as fm
import fast_simple as fs
from cases import couette_bcs, load_mesh_arrays
from orc_b200 import _lib
from orc_b200 import synthetic as syn

RHO, MU = bench.RHO, bench.MU


def hex_channel(oracle, nx=12, ny=8, nz=6):
    om = oracle.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(nx, ny, nz)))
    syn.channel_bcs(om)
    return om, {}


def tet_box(oracle):
    om = oracle.Mesh.from_arrays(*syn.mesh_args(syn.tet_box(4, 4, 3)))
    syn.channel_bcs(om, fully_3d=True)
    return om, dict(momentum=oracle.TVD, limiter=oracle.PSI_UMIST)


def channel_flow(oracle):
    om = oracle.Mesh.from_arrays(*syn.mesh_args(load_mesh_arrays("channel_flow")))
    couette_bcs(om, u_wall=0.0, dp_dx=5.0, wall_zones=("WALL",), moving=None)
    return om, dict(momentum=oracle.TVD, limiter=oracle.PSI_QUICK)


MESHES = {"hex": hex_channel, "tet_umist": tet_box, "channel_flow_msh": channel_flow}
SOLVERS = {"multigrid": 2, "bicgstab": 3, "jacobi": 1}


def zeros(om):
    return [np.zeros(om.n_cells) for _ in range(4)]


def assert_equal_to_oracle(recs, oracle_out):
    uo, vo, wo, po_, reports, _ = oracle_out
    assert len(recs) == len(reports)
    for rec, rep in zip(recs, reports):
        assert np.array_equal(rec["report"], rep), (rec["iteration"], rec["report"], rep)
    last = recs[-1]
    for c, a, b in zip("uvwp", (last["u"], last["v"], last["w"], last["p"]), (uo, vo, wo, po_)):
        assert np.array_equal(a, b), c


@pytest.mark.parametrize("solver", list(SOLVERS))
@pytest.mark.parametrize("mesh", list(MESHES))
def test_driver_with_the_oracle_solver_is_solve_steady(oracle, mesh, solver):
    om, kw = MESHES[mesh](oracle)
    s = oracle.Settings(pressure_relaxation=bench.P_RELAX, solver_type=SOLVERS[solver], iterations=10, **kw)
    iters = 3
    try:
        want = om.solve_steady(*zeros(om), s, RHO, MU, iters, 1)
    except oracle.OraclePanic as e:   # channel_flow.msh + Jacobi: x turns NaN in iteration 1 ("diverged")
        assert (mesh, solver) == ("channel_flow_msh", "jacobi"), e
        with pytest.raises(oracle.OraclePanic, match=str(e)):
            fs.simple_iterations(om, s, RHO, MU, zeros(om), iters, fs.oracle_solve(s))
        return
    recs = fs.simple_iterations(om, s, RHO, MU, zeros(om), iters, fs.oracle_solve(s))
    assert_equal_to_oracle(recs, want)
    assert all(np.isfinite(r["report"]).all() for r in recs)
    # lockstep: a_u, a_v, a_w bit-identical unless TVD limits them differently (from rest every face takes the central
    # coefficient); Jacobi never runs in lockstep
    tvd = "momentum" in kw
    assert [r["batched"] for r in recs] == [solver != "jacobi" and (it == 0 or not tvd) for it in range(iters)]


def test_replayed_state_continues_the_run(oracle):
    """Starting at iteration 3 from the fields after iteration 2 and a state brought up by replaying the two momentum assemblies
    gives the run's iteration 3."""
    om, _ = hex_channel(oracle)
    s = oracle.Settings(pressure_relaxation=bench.P_RELAX, iterations=10)
    solve = fs.oracle_solve(s)
    recs = fs.simple_iterations(om, s, RHO, MU, zeros(om), 3, solve)
    state = fs.State(om, MU)
    state.replay(om, s, RHO, zeros(om))
    state.replay(om, s, RHO, [recs[0][k] for k in "uvwp"])
    again = fs.simple_iterations(om, s, RHO, MU, [recs[1][k] for k in "uvwp"], 1, solve, state=state, first=3)
    for k in ("u", "v", "w", "p", "report"):
        assert np.array_equal(again[0][k], recs[2][k]), k


@pytest.mark.parametrize("mesh", ["hex16", "channel_flow_msh"])
def test_driver_with_model_solves_is_near_the_oracle(oracle, mesh):
    """fast_model's summation orders, 5 inner iterations: <= 1e-6 of the velocity norm / of ||p|| after two iterations.
    channel_flow.msh starts from the oracle's fields after two iterations: from rest its v and w right-hand sides are ~1e-26, and
    in the fast mode's summation order the first lockstep solve meets 0 / 0 (see test_gpu_fast_simple)."""
    om, kw = hex_channel(oracle, 16, 16, 16) if mesh == "hex16" else channel_flow(oracle)
    s = oracle.Settings(pressure_relaxation=bench.P_RELAX, iterations=5, **kw)
    start = zeros(om) if mesh == "hex16" else list(om.solve_steady(*zeros(om), oracle.Settings(**kw), RHO, MU, 2, 0)[:4])
    ex = om.export()
    log = []
    recs = fs.simple_iterations(om, s, RHO, MU, start, 2, fs.model_solve(s, log), pos=fm.Positions(ex["cell_centroid"]))
    uo, vo, wo, po_, reports, _ = om.solve_steady(*start, s, RHO, MU, 2, 1)
    last = recs[-1]
    vel = np.sqrt(sum(np.linalg.norm(b) ** 2 for b in (uo, vo, wo)))
    errs = [np.linalg.norm(last[c] - b) / vel for c, b in zip("uvw", (uo, vo, wo))] + [np.linalg.norm(last["p"] - po_) / np.linalg.norm(po_)]
    print(f"{mesh}: model vs oracle after 2 iterations (u, v, w / |vel|, p):", [f"{e:.2e}" for e in errs], "levels:", log[:2])
    assert max(errs) <= 1e-6, errs
    assert len(log) == (2 if "momentum" not in kw else 4) * 2 and len(log[0]) == 4


def test_divergence_is_the_same_error_in_the_same_iteration(oracle):
    """The velocity-inlet start of the reference's default driver: from rest the v and w systems have a zero right-hand side, the
    unguarded BiCGSTAB divides 0 by 0 and Multigrid's residual check fails in iteration 1 on both sides."""
    om = oracle.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(10, 6, 4)))
    syn.channel_bcs(om)
    om.set_zone("INLET", 10, 0.0, (1e-3, 0.0, 0.0))
    s = oracle.Settings(iterations=5)
    with pytest.raises(oracle.OraclePanic, match=fm.MG_DIVERGED):
        om.solve_steady(*zeros(om), s, RHO, MU, 1, 0)
    seen = []
    with pytest.raises(oracle.OraclePanic, match=fm.MG_DIVERGED):
        fs.simple_iterations(om, s, RHO, MU, zeros(om), 2, fs.oracle_solve(s), on_iteration=seen.append)
    with pytest.raises(fm.ModelDiverged, match=fm.MG_DIVERGED) as e:
        fs.simple_iterations(om, s, RHO, MU, zeros(om), 2, fs.model_solve(s), on_iteration=seen.append)
    assert e.value.code == _lib.E_MG_DIVERGED and seen == []


def test_field_sum_check():
    fm.check_field_sums(np.ones(3), np.array([np.inf, 1.0]), np.array([-np.inf]))
    for bad in (np.array([1.0, np.nan]), np.array([np.inf, -np.inf])):
        with pytest.raises(fm.ModelDiverged, match=fm.DIVERGED) as e:
            fm.check_field_sums(np.ones(2), bad)
        assert e.value.code == _lib.E_DIVERGED
