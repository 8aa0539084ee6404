"""Whole fast-mode SIMPLE iterations on the GPU bit for bit against tests/fast_simple.py (the oracle's assemblies and correction,
the oracle's Multigrid hierarchies and fast_model's solves, composed in the order of steady_iterate). Every field comparison is
np.array_equal, every iteration. This pins what the per-solver pins of test_gpu_fast_model.py leave open: b += b_di, the lockstep
decision and the pack / unpack of the three systems, the Multigrid solve of the pressure-correction matrix with its own
hierarchy, p' *= 0, the correction, the diagonals carried from one iteration to the next, and SteadySolver.reset().

The report scalars are not pinned bit for bit: k_apply_correction and k_peclet sum over a grid sized from the SM count
(DESIGN.md §5). They are checked against exact sums with the bound of their summation tree, and the test asserts that the bound is
tight enough to catch a sum that leaves out one block's partial.

Run with -s: every case prints the lockstep flag, the level sizes and its runtime."""
import math
import os
import time

import numpy as np
import pytest

import bench
import fast_model as fm
import fast_simple as fs
import orc_b200
from orc_b200 import _lib
from orc_b200 import synthetic as syn
from orc_b200.settings import ReductionMode, SolutionMethod
from cases import couette_bcs, load_mesh_arrays, make_pair, settings_pair
from test_gpu_fast_model import mismatch

pytestmark = pytest.mark.gpu
RHO, MU = bench.RHO, bench.MU
U = 2.0 ** -53


def gamma(m):
    return m * U / (1.0 - m * U)


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def grid_for(n, block, cap):
    """common.cuh grid_for."""
    return int(max(1, min(-(-n // block), cap)))


def tree_depth(n, grid):
    """Additions a term passes through in a grid-stride kernel sum: the per-thread chain, block_sum (two 32-lane trees) and
    sum_partials (a chain over the block partials, then block_sum)."""
    return -(-n // (grid * 256)) + 10 + -(-grid // 256) + 10


def block_partials(x, grid):
    """Exact partial of every block of a grid-stride kernel: thread t of block b takes rows b * 256 + t + k * grid * 256."""
    x = np.asarray(x, dtype=np.float64)
    stride = grid * 256
    q = np.zeros(-(-x.size // stride) * stride)
    q[:x.size] = x
    q = q.reshape(-1, grid, 256)
    return np.array([math.fsum(q[:, b, :].ravel()) for b in range(grid)])


def peclet_cell_means(state):
    """Per-cell Peclet means of the last assembly, recovered from the matrix diagonals: a_ii = a_p + a_ii_di, Pe = a_p / a_ii_di
    (oracle build_momentum_advection_matrices). a_ii - a_ii_di gives a_p to a few ulps of a_ii, which is all the bite check of
    the Peclet mean needs (its margin is many orders of magnitude)."""
    def diag(a):
        m = fm.Mat.from_handle(a)
        return m.val[m.diag_index()]
    d_di = diag(state.a_di)
    pe = [(diag(a) - d_di) / d_di for a in state.a]
    return (((0. + pe[0]) + pe[1]) + pe[2]) / 3.


def check_report(rep, rec, p_prime, n, pe_cells=None):
    """The GPU's report of one iteration against the model's: Peclet extremes ==; the field averages and ||p'|| within
    gamma_{m+1} * sum |x_i| of math.fsum; the Peclet mean and ||velocity correction|| (the oracle gives their sequential sums only)
    within the sum of both sides' bounds. Returns the margins of the bite check: the smallest block partial over the bound
    (`pe_cells`, the per-cell Peclet means, adds the Peclet mean's)."""
    _, ua, va, wa, pe_avg, pe_min, pe_max, vc, ppn = rec["report"]
    assert rep["peclet_min"] == pe_min and rep["peclet_max"] == pe_max, (rep, rec["report"])
    g_cor = grid_for(n, 256, sm_count() * 8)
    g_pe = grid_for(n, 256, sm_count() * 4)
    m_cor, m_pe = tree_depth(n, g_cor) + 1, tree_depth(n, g_pe) + 1
    bites = {}
    for key, f in zip(("u_avg", "v_avg", "w_avg"), (rec["u"], rec["v"], rec["w"])):
        exact = math.fsum(f) / n
        bound = gamma(m_cor) * math.fsum(np.abs(f)) / n
        assert abs(rep[key] - exact) <= bound, (key, rep[key], exact, bound)
        bites[key] = np.abs(block_partials(f, g_cor)).min() / n / bound
    sq = p_prime * p_prime
    exact = math.sqrt(math.fsum(sq))
    bound = gamma(m_cor) * exact
    assert abs(rep["pressure_correction"] - exact) <= bound, (rep["pressure_correction"], exact, bound)
    bites["pressure_correction"] = block_partials(sq, g_cor).min() / (2.0 * exact) / bound   # d sqrt(S) = dS / (2 sqrt(S))
    bound = (gamma(m_cor) + gamma(n + 1)) * vc
    assert abs(rep["velocity_correction"] - vc) <= bound, (rep["velocity_correction"], vc, bound)
    mag = max(abs(pe_min), abs(pe_max))
    bound = (gamma(m_pe) + gamma(n + 2)) * mag
    assert abs(rep["peclet_avg"] - pe_avg) <= bound, (rep["peclet_avg"], pe_avg, bound)
    if pe_cells is not None:
        bites["peclet_avg"] = np.abs(block_partials(pe_cells, g_pe)).min() / n / bound
    return bites


def run_case(oracle, pm, om, ps, os_, iterations, start=None, pos=True, label=""):
    """`iterations` SteadySolver.iterate(1) calls from `start` (rest if None), each compared with the model's iteration as soon as
    the model has it. Returns (model records, GPU fields per iteration, bite margins per iteration, solver)."""
    n = pm.n_cells
    start = start if start is not None else [np.zeros(n) for _ in range(4)]
    solver = orc_b200.SteadySolver(pm, ps, RHO, MU)
    solver.set_fields(*start)
    got, bites, log = [], [], []
    t0 = time.perf_counter()

    def compare(rec):
        rep = solver.iterate(1)
        f = solver.get_fields()
        got.append(f)
        print(f"{label} iteration {rec['iteration']}: batched() = {solver.batched} (model {rec['batched']}), levels {solver.level_sizes()}, "
              f"{time.perf_counter() - t0:.1f} s")
        errs = [mismatch(g, rec[c], f"{label} iteration {rec['iteration']} {c}") for g, c in zip(f, "uvwp")]
        errs = [e for e in errs if e]
        assert not errs, "\n".join(errs)
        assert solver.batched == rec["batched"]
        bites.append(check_report(rep, rec, rec["p_prime"], n, peclet_cell_means(state)))

    P = fm.Positions(om.export()["cell_centroid"]) if pos else None
    state = fs.State(om, MU)
    model = fs.simple_iterations(om, os_, RHO, MU, start, iterations, fs.model_solve(os_, log), state=state, pos=P, on_iteration=compare)
    print(f"{label}: {iterations} iterations pinned in {time.perf_counter() - t0:.1f} s; model hierarchies (rows, nnz) of the first "
          f"two solves: {log[:2]}")
    return model, got, bites, solver


def hex_pair(oracle, nx, ny, nz):
    pm, om = make_pair(oracle, syn.hex_box(nx, ny, nz))
    for m in (pm, om):
        syn.channel_bcs(m)
    return pm, om


# ---- 48^3 hex channel, bench settings: RESET_EVERY iterations from rest, reset(), and the ordering's negative control ---------
_hex48 = {}


def hex48(oracle):
    if not _hex48:
        pm, om = hex_pair(oracle, 48, 48, 48)
        ps, os_ = settings_pair(oracle, pressure_relaxation=bench.P_RELAX)
        ps.reduction_mode = ReductionMode.Auto
        _hex48.update(pm=pm, om=om, ps=ps, os=os_)
    return _hex48


def test_hex48_bench_settings_from_rest_and_reset(oracle):
    s = hex48(oracle)
    pm = s["pm"]
    assert pm.n_cells > 16384   # ORC_AUTO_EXACT_MAX_ROWS: Auto runs the fast mode here
    t0 = time.perf_counter()
    model, got, bites, solver = run_case(oracle, pm, s["om"], s["ps"], s["os"], bench.RESET_EVERY, label="hex48")
    assert all(r["batched"] for r in model)
    for b in bites:
        print("  bite margins (smallest block partial / bound):", {k: f"{v:.2e}" for k, v in b.items()})
        assert b["u_avg"] > 2 and b["pressure_correction"] > 2 and b["peclet_avg"] > 2, b
    solver.reset()
    solver.iterate(1)
    f = solver.get_fields()
    errs = [mismatch(g, model[0][c], f"hex48 iteration 1 after reset() {c}") for g, c in zip(f, "uvwp")]
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)
    _hex48["model1"] = model[0]
    print(f"hex48: {time.perf_counter() - t0:.1f} s")


def test_hex48_without_the_ordering_is_pinned_by_the_model_without_positions(oracle, monkeypatch):
    """Negative control: with ORC_B200_REORDER=0 the GPU must differ from the model with positions and equal the model without:
    the pin resolves the summation order of the coarse-level smoothers."""
    s = hex48(oracle)
    t0 = time.perf_counter()
    with_pos = s.get("model1") or fs.simple_iterations(s["om"], s["os"], RHO, MU, [np.zeros(s["pm"].n_cells)] * 4, 1,
                                                       fs.model_solve(s["os"]), pos=fm.Positions(s["om"].export()["cell_centroid"]))[0]
    monkeypatch.setenv("ORC_B200_REORDER", "0")
    model, got, _, _ = run_case(oracle, s["pm"], s["om"], s["ps"], s["os"], 1, pos=False, label="hex48 ORC_B200_REORDER=0")
    assert not np.array_equal(got[0][0], with_pos["u"]) and not np.array_equal(got[0][3], with_pos["p"])
    print(f"hex48 ordering off: {time.perf_counter() - t0:.1f} s")


# ---- 30^3 x 6 tet box, TVD-UMIST: three hierarchies per iteration once the limiter tells the components apart --------------------
def test_tet30_umist_three_iterations(oracle):
    t0 = time.perf_counter()
    pm, om = make_pair(oracle, syn.tet_box(30, 30, 30))
    for m in (pm, om):
        syn.channel_bcs(m, fully_3d=True)
    ps, os_ = settings_pair(oracle, pressure_relaxation=bench.P_RELAX, momentum=3, limiter=4)
    ps.reduction_mode = ReductionMode.Auto
    model, _, _, _ = run_case(oracle, pm, om, ps, os_, 3, label="tet30")
    assert [r["batched"] for r in model] == [True, False, False]   # from rest every face takes the central coefficient
    print(f"tet30: {time.perf_counter() - t0:.1f} s")


# ---- 24^3 hex (13 824 cells: Auto would pick reference order), Fast forced: lockstep BiCGSTAB, then three Jacobi solves --------
@pytest.mark.parametrize("solver", ["bicgstab", "jacobi"])
def test_hex24_fast_bicgstab_and_jacobi(oracle, solver):
    t0 = time.perf_counter()
    pm, om = hex_pair(oracle, 24, 24, 24)
    ps, os_ = settings_pair(oracle, pressure_relaxation=bench.P_RELAX, solver_type={"bicgstab": 3, "jacobi": 1}[solver])
    assert ps.matrix_solver.solver_type == {"bicgstab": SolutionMethod.BiCGSTAB, "jacobi": SolutionMethod.Jacobi}[solver]
    model, _, _, _ = run_case(oracle, pm, om, ps, os_, 3, label=f"hex24 {solver}")
    assert [r["batched"] for r in model] == [solver == "bicgstab"] * 3
    print(f"hex24 {solver}: {time.perf_counter() - t0:.1f} s")


# ---- channel_flow.msh, TVD-QUICK + Multigrid, Fast forced: coarse levels of one virtual block ----------------------------------
def channel_flow_pair(oracle):
    pm, om = make_pair(oracle, load_mesh_arrays("channel_flow"))
    for m in (pm, om):
        couette_bcs(m, u_wall=0.0, dp_dx=5.0, wall_zones=("WALL",), moving=None)
    ps, os_ = settings_pair(oracle, momentum=3, limiter=3)
    return pm, om, ps, os_


def test_channel_flow_msh_tvd_quick_multigrid(oracle):
    """From the oracle's fields after two iterations (from rest the fast mode diverges: next test). The GPU's matrices start
    freshly initialised, like the model's State and like oracle.solve_steady."""
    pm, om, ps, os_ = channel_flow_pair(oracle)
    start = list(om.solve_steady(*[np.zeros(om.n_cells)] * 4, os_, RHO, MU, 2, 0)[:4])
    model, _, _, solver = run_case(oracle, pm, om, ps, os_, 3, start=start, label="channel_flow.msh")
    levels = solver.level_sizes()
    assert len(levels) == 4 and levels[-1][0] <= 256, levels   # the coarsest level fits one virtual block


def test_channel_flow_msh_from_rest_diverges_in_iteration_1_on_both_sides(oracle):
    """From rest the v and w right-hand sides are ~1e-26; in the fast mode's summation order the lockstep Multigrid solve meets 0 / 0
    and its residual check fails in iteration 1, on the GPU and in the model alike (the oracle's sequential order survives)."""
    pm, om, ps, os_ = channel_flow_pair(oracle)
    z = [np.zeros(pm.n_cells) for _ in range(4)]
    with pytest.raises(fm.ModelDiverged, match=fm.MG_DIVERGED):
        fs.simple_iterations(om, os_, RHO, MU, z, 1, fs.model_solve(os_), pos=fm.Positions(om.export()["cell_centroid"]))
    solver = orc_b200.SteadySolver(pm, ps, RHO, MU)
    solver.set_fields(*z)
    with pytest.raises(orc_b200.OrcError) as e:
        solver.iterate(1)
    assert e.value.code == _lib.E_MG_DIVERGED


# ---- 128^3 bench mesh: iteration 2 of the benchmark, modelled from the GPU's fields after iteration 1 ------------------------
_JOB = {}


def _solve_one(k):
    """System k of the lockstep call in _JOB (set before the fork, so the workers share the matrices instead of pickling them)."""
    j = _JOB
    return fm.iterative_solve(j["A"], j["B"][k:k + 1], j["X"][k:k + 1], j["s"].iterations, fm.MULTIGRID, relaxation=j["s"].relaxation,
                              threshold=j["s"].threshold, levels=j["levels"], pos=j["pos"], mg_levels=j["s"].mg_levels)[0]


def parallel_model_solve(settings):
    """fs.model_solve for the benchmark's settings (Multigrid, BiCGSTAB smoother, Jacobi preconditioner) with the K systems of a
    lockstep call in K processes: the K = 3 arithmetic is the K = 1 arithmetic of each system, so splitting them changes no bit."""
    import multiprocessing as mp
    one = fs.model_solve(settings)
    assert settings.solver_type == fs.po.MULTIGRID and settings.mg_smoother == fs.po.BICGSTAB
    assert settings.preconditioner == fs.po.PC_JACOBI

    def solve(a, B, X, pos=None):
        if B.shape[0] == 1:
            return one(a, B, X, pos)
        A = fm.Mat.from_handle(a)
        _, lev = fs.po.multigrid_trace(a, np.ones(A.nrows), np.zeros(A.nrows), iterations=1)
        _JOB.update(A=A, B=B, X=X, s=settings, levels=[(fm.Mat.from_handle(r), fm.Mat.from_handle(c)) for r, c in lev], pos=pos)
        try:
            with mp.get_context("fork").Pool(B.shape[0]) as pool:
                return np.stack(pool.map(_solve_one, range(B.shape[0])))
        finally:
            _JOB.clear()
    return solve


def test_bench_mesh_iteration_2(oracle):
    """The benchmark's per-step computation (128^3, bench settings, 50 inner iterations, lockstep momentum solve, four-level
    Multigrid on both systems), pinned: the model starts from the GPU's fields after iteration 1 and the oracle's matrix state
    after one replayed momentum assembly (on the fields iteration 1 started from: rest)."""
    import resource
    t0 = time.perf_counter()
    pm, om = hex_pair(oracle, 128, 128, 128)
    ps, os_ = settings_pair(oracle, pressure_relaxation=bench.P_RELAX)
    ps.reduction_mode = ReductionMode.Auto
    n = pm.n_cells
    solver = orc_b200.SteadySolver(pm, ps, RHO, MU)
    solver.set_fields(*[np.zeros(n)] * 4)
    solver.iterate(1)
    after1 = solver.get_fields()
    rep = solver.iterate(1)
    got = solver.get_fields()
    batched, levels = solver.batched, solver.level_sizes()
    solver.close()
    print(f"128^3: GPU iteration 2: batched() = {batched}, levels {levels}")
    state = fs.State(om, MU)
    state.replay(om, os_, RHO, [np.zeros(n)] * 4)
    t1, c1 = time.perf_counter(), time.process_time()
    rec = fs.simple_iterations(om, os_, RHO, MU, after1, 1, parallel_model_solve(os_), state=state, first=2,
                               pos=fm.Positions(om.export()["cell_centroid"]))[0]
    me, kids = resource.getrusage(resource.RUSAGE_SELF), resource.getrusage(resource.RUSAGE_CHILDREN)
    print(f"128^3: model iteration 2: {time.perf_counter() - t1:.0f} s wall, {time.process_time() - c1 + kids.ru_utime + kids.ru_stime:.0f} s "
          f"CPU ({os.cpu_count()} cores; the three momentum systems in three processes); peak RSS {me.ru_maxrss / 2 ** 20:.1f} GB in the "
          f"test process, {kids.ru_maxrss / 2 ** 20:.1f} GB in the largest worker")
    errs = [mismatch(g, rec[c], f"128^3 iteration 2 {c}") for g, c in zip(got, "uvwp")]
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)
    assert batched and rec["batched"]
    bites = check_report(rep, rec, rec["p_prime"], n, peclet_cell_means(state))
    print("128^3: bite margins (smallest block partial / bound):", {k: f"{v:.2e}" for k, v in bites.items()})
    assert bites["u_avg"] > 2 and bites["pressure_correction"] > 2 and bites["peclet_avg"] > 2, bites
    print(f"128^3: {time.perf_counter() - t0:.0f} s")
