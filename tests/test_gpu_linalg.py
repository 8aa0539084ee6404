"""GPU parity of the linear-algebra kernels against the oracle, through the C ABI. Integer/index work (patterns,
aggregates) must be bit-exact; SpMV / scaling / Galerkin values are bit-exact too (same operation order, no FMA);
anything that contains a global dot product is compared at a stated tolerance."""
import numpy as np
import pytest
import scipy.sparse as sp

import fast_model as fm
import orc_b200
from orc_b200 import linear_algebra as la
from orc_b200.settings import SolutionMethod, PreconditionMethod, RestrictionMethods
from conftest import rel_l2, max_rel

pytestmark = pytest.mark.gpu


def random_spd_like(n, density, seed, sym=True):
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=density, random_state=rng, format="csr", data_rvs=lambda k: -rng.random(k))
    if sym:
        a = a + a.T
    a = a.tolil()
    a.setdiag(0)
    a = a.tocsr()
    a.eliminate_zeros()
    d = np.asarray(-a.sum(axis=1)).ravel() + 0.5 + rng.random(n)
    a = (a + sp.diags(d)).tocsr()
    a.sort_indices()
    return a


def kat_matrix(n=100):
    """The reference's own solver test system (src/linear_algebra.rs:309-378)."""
    rows, cols, vals = [], [], []
    for i in range(n):
        for j in range(n):
            if i == j:
                rows.append(i); cols.append(j); vals.append(1.0)
            elif j not in (0, n - 1) and abs(i - j) == 1:
                rows.append(i); cols.append(j); vals.append(-0.25)
    a = sp.csr_matrix((vals, (rows, cols)), shape=(n, n))
    a.sort_indices()
    xs = 2.0 * np.arange(n)
    return a, xs


def both(oracle, ctx, a):
    return la.CsrMatrix.from_scipy(a, ctx), oracle.Csr.from_arrays(a.shape[0], a.shape[1], a.indptr, a.indices, a.data)


def assert_csr_equal(g, o, exact_values=True, tol=0.0):
    grp, gco, gva = g.arrays()
    orp, oco, ova = o.arrays()
    assert g.dims == o.dims
    assert np.array_equal(grp, orp), "row pointers differ"
    assert np.array_equal(gco, oco), "column indices differ"
    if exact_values:
        assert np.array_equal(gva, ova), f"values differ: max rel {max_rel(gva, ova):.3e}"
    else:
        assert max_rel(gva, ova) <= tol


def assert_spmv(a, y, yo, x):
    """Rows shorter than 10 on average go through the thread-per-row kernel whose in-row sums run in ascending column order:
    bit-exact. Longer rows (AMG coarse levels) use G lanes per row and a fixed shuffle tree: equal to rounding, measured
    against the row's own magnitude sum |a_ik x_k| (model-free), and bit-exact against that tree in tests/fast_model.py."""
    if a.nnz < 10 * a.shape[0]:
        assert np.array_equal(y, yo)
    else:
        mag = abs(a) @ np.abs(x)
        assert np.all(np.abs(y - yo) <= 1e-14 * np.maximum(mag, 1e-300))
        assert np.array_equal(y, fm.spmv(fm.Mat.from_scipy(a), x)[0])


@pytest.mark.parametrize("n,density", [(1, 1.0), (37, 0.2), (1000, 0.004), (5000, 0.001), (1000, 0.01), (5000, 0.004), (300, 0.5), (2000, 0.03)])
def test_spmv_matches_oracle(oracle, ctx, n, density):
    a = random_spd_like(n, density, seed=n)
    g, o = both(oracle, ctx, a)
    x = np.random.default_rng(1).standard_normal(n)
    assert_spmv(a, g.spmv(x), o.spmv(x), x)


def test_spmv_long_rows_and_empty_rows(oracle, ctx):
    rng = np.random.default_rng(3)
    a = sp.random(700, 700, density=0.6, random_state=rng, format="lil")
    a[5, :] = 0
    a[699, :] = 0
    a = a.tocsr(); a.eliminate_zeros(); a.sort_indices()
    g, o = both(oracle, ctx, a)
    x = rng.standard_normal(700)
    y = g.spmv(x)
    assert y[5] == 0.0 and y[699] == 0.0
    assert_spmv(a, y, o.spmv(x), x)


def test_spmv_short_rows_spanning_staging_chunks(oracle, ctx):
    """A few very long rows (4000 and 2000 entries) inside a short-row matrix: the thread-per-row kernel sums each of them
    alone, in ascending column order, however long it is."""
    rng = np.random.default_rng(9)
    a = random_spd_like(4000, 0.0005, seed=77).tolil()
    a[100, :] = rng.standard_normal(4000)
    a[2049, ::2] = 1.5
    a = a.tocsr(); a.sort_indices()
    assert a.nnz < 10 * a.shape[0]
    g, o = both(oracle, ctx, a)
    x = rng.standard_normal(4000)
    assert np.array_equal(g.spmv(x), o.spmv(x))


def test_jacobi_scale_bit_exact(oracle, ctx):
    a = random_spd_like(2000, 0.005, seed=5)
    b = np.random.default_rng(2).standard_normal(2000)
    g, o = both(oracle, ctx, a)
    gs, gb = g.jacobi_scale(b)
    os_, ob = o.jacobi_scale(b)
    assert_csr_equal(gs, os_)
    assert np.array_equal(gb, ob)


def test_jacobi_scale_missing_diagonal_rows(oracle, ctx):
    a = random_spd_like(200, 0.05, seed=6).tolil()
    for i in (0, 17, 199):
        a[i, i] = 0
    a = a.tocsr(); a.eliminate_zeros(); a.sort_indices()
    b = np.random.default_rng(2).standard_normal(200)
    g, o = both(oracle, ctx, a)
    gs, gb = g.jacobi_scale(b)
    os_, ob = o.jacobi_scale(b)
    assert_csr_equal(gs, os_)
    assert np.array_equal(gb, ob)


def test_reference_unit_test_jacobi_then_bicgstab(oracle, ctx):
    """validate_iterative_solvers (src/linear_algebra.rs:309-378): Jacobi then BiCGSTAB, |Ax-b| < 1e-3."""
    a, xs = kat_matrix()
    g, o = both(oracle, ctx, a)
    b = a @ xs
    thr = 1e-3 / 100 ** 3
    for method in (SolutionMethod.Jacobi, SolutionMethod.BiCGSTAB):
        x = np.zeros(100)
        la.iterative_solve(g, b, x, 50, method, 0.5, thr, PreconditionMethod.Jacobi)
        xo = oracle.iterative_solve(o, b, np.zeros(100), 50, int(method), 0.5, thr, 1)
        if method == SolutionMethod.BiCGSTAB:
            assert np.linalg.norm(a @ x - b) < 1e-3
        # tolerance: dot products are summed in a different (fixed) order than nalgebra's 8 accumulators
        assert rel_l2(x, xo) < 1e-9, (method, rel_l2(x, xo))


@pytest.mark.parametrize("precond", [0, 1])
def test_bicgstab_matches_oracle(oracle, ctx, precond):
    a = random_spd_like(3000, 0.003, seed=11)
    g, o = both(oracle, ctx, a)
    rng = np.random.default_rng(4)
    b, x0 = rng.standard_normal(3000), rng.standard_normal(3000)
    x = x0.copy()
    la.iterative_solve(g, b, x, 12, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod(precond))
    xo = oracle.iterative_solve(o, b, x0, 12, oracle.BICGSTAB, 0.5, 1e-3, precond)
    assert rel_l2(x, xo) < 1e-9


def test_jacobi_matches_oracle_and_converges(oracle, ctx):
    a = random_spd_like(1500, 0.004, seed=12)
    g, o = both(oracle, ctx, a)
    rng = np.random.default_rng(5)
    b = rng.standard_normal(1500)
    for iters, thr in ((7, 1e-30), (200, 1e-3)):
        x = np.zeros(1500)
        la.iterative_solve(g, b, x, iters, SolutionMethod.Jacobi, 0.5, thr, PreconditionMethod.Jacobi)
        xo = oracle.iterative_solve(o, b, np.zeros(1500), iters, oracle.JACOBI, 0.5, thr, 1)
        assert rel_l2(x, xo) < 1e-12


@pytest.mark.parametrize("sym", [True, False])
def test_gauss_seidel_lexicographic_matches_intended_formula(oracle, ctx, sym):
    a = random_spd_like(900, 0.01, seed=13, sym=sym)
    g, o = both(oracle, ctx, a)
    b = np.random.default_rng(6).standard_normal(900)
    x = np.zeros(900)
    la.iterative_solve(g, b, x, 5, SolutionMethod.GaussSeidel, 0.7, 1e-3, PreconditionMethod.Jacobi)
    xo = oracle.iterative_solve(o, b, np.zeros(900), 5, oracle.GAUSS_SEIDEL, 0.7, 1e-3, 1, gs_intended=1)
    assert np.array_equal(x, xo)  # same row order, same in-row summation order: bit-exact


def test_gauss_seidel_reference_mode_reports_the_panic(ctx):
    from orc_b200.settings import GaussSeidelMode
    a = random_spd_like(50, 0.1, seed=14)
    g = la.CsrMatrix.from_scipy(a, ctx)
    with pytest.raises(orc_b200.OrcError) as e:
        la.iterative_solve(g, np.ones(50), np.zeros(50), 2, SolutionMethod.GaussSeidel, 0.5, 1e-3, PreconditionMethod.NONE,
                           gs_mode=GaussSeidelMode.ReferencePanic)
    assert e.value.code == orc_b200._lib.E_GS_MAINTENANCE


@pytest.mark.parametrize("n,density,sym", [(2, 1.0, True), (33, 0.3, True), (1001, 0.006, True), (4000, 0.002, True), (500, 0.02, False)])
def test_restriction_strongest_bit_exact(oracle, ctx, n, density, sym):
    a = random_spd_like(n, density, seed=20 + n, sym=sym)
    g, o = both(oracle, ctx, a)
    assert_csr_equal(la.build_restriction_matrix(g, RestrictionMethods.Strongest), o.build_restriction(oracle.STRONGEST))


def test_restriction_with_ties_and_positive_offdiagonals(oracle, ctx):
    # uniform Laplacian: every off-diagonal ties, so the FIRST minimum must win; plus a few positive couplings
    n = 12
    lap = sp.diags([-1, -1, 4, -1, -1], [-n, -1, 0, 1, n], shape=(n * n, n * n)).tolil()
    lap[3, 4] = 0.5; lap[4, 3] = 0.5
    a = lap.tocsr(); a.sort_indices()
    g, o = both(oracle, ctx, a)
    assert_csr_equal(la.build_restriction_matrix(g), o.build_restriction(oracle.STRONGEST))


def test_restriction_injection(oracle, ctx):
    for n in (7, 8):
        a = random_spd_like(n, 0.5, seed=n)
        g, o = both(oracle, ctx, a)
        assert_csr_equal(la.build_restriction_matrix(g, RestrictionMethods.Injection), o.build_restriction(oracle.INJECTION))


@pytest.mark.parametrize("n,density", [(40, 0.2), (1500, 0.004), (600, 0.08)])
def test_galerkin_pattern_and_values(oracle, ctx, n, density):
    a = random_spd_like(n, density, seed=30 + n)
    g, o = both(oracle, ctx, a)
    gr = la.build_restriction_matrix(g)
    orr = o.build_restriction(oracle.STRONGEST)
    assert_csr_equal(la.galerkin(gr, g), oracle.galerkin(orr, o))


def test_multigrid_levels_and_solution(oracle, ctx):
    """Three coarse levels: every R_l bit-exact, every A_l pattern bit-exact; values of deeper levels depend on the
    level above only through exact arithmetic, so they are bit-exact too. The solution carries dot-product reordering."""
    a = random_spd_like(3000, 0.002, seed=41)
    g, o = both(oracle, ctx, a)
    rng = np.random.default_rng(8)
    b = rng.standard_normal(3000)
    x, glev = la.multigrid_trace(g, b, np.zeros(3000), iteration_count=6)
    xo, olev = oracle.multigrid_trace(o, b, np.zeros(3000), iterations=6)
    assert len(glev) == len(olev) == 3
    for (gr, ga), (orr, oa) in zip(glev, olev):
        assert_csr_equal(gr, orr)
        assert_csr_equal(ga, oa)
    assert rel_l2(x, xo) < 1e-8


@pytest.mark.parametrize("method", [SolutionMethod.BiCGSTAB, SolutionMethod.Jacobi, SolutionMethod.Multigrid])
def test_reference_order_reductions_make_solves_bit_identical(oracle, ctx, method):
    """ORC_REDUCE_REFERENCE_ORDER: dot products and norms follow nalgebra's 8-accumulator order, SpMV sums stay in ascending
    column order for every row length -> the solution vector is bit-identical to the reference's CPU path."""
    from orc_b200.settings import ReductionMode
    a = random_spd_like(2500, 0.004, seed=51)
    g, o = both(oracle, ctx, a)
    rng = np.random.default_rng(9)
    b, x0 = rng.standard_normal(2500), rng.standard_normal(2500)
    x = x0.copy()
    la.iterative_solve(g, b, x, 40, method, 0.5, 1e-3, PreconditionMethod.Jacobi, reduction_mode=ReductionMode.ReferenceOrder)
    xo = oracle.iterative_solve(o, b, x0, 40, int(method), 0.5, 1e-3, 1)
    assert np.array_equal(x, xo), rel_l2(x, xo)


@pytest.mark.parametrize("method", [SolutionMethod.BiCGSTAB, SolutionMethod.Multigrid])
@pytest.mark.parametrize("n,density", [(3000, 0.002), (4000, 0.012), (2048, 0.03)])   # thread-per-row, 4 and 8 lanes per row
def test_three_systems_in_lockstep_equal_three_single_solves(ctx, method, n, density):
    """orc_iterative_solve3 (the u, v, w momentum solves sharing one matrix, src/solver.rs:99-136): every system must get
    the bits of its own orc_iterative_solve call — same in-row order, same reduction trees, own scalars."""
    a = random_spd_like(n, density, seed=61)
    g = la.CsrMatrix.from_scipy(a, ctx)
    rng = np.random.default_rng(10)
    bs = [rng.standard_normal(n) for _ in range(3)]
    x0 = [rng.standard_normal(n) for _ in range(3)]
    singles = []
    for b, x in zip(bs, x0):
        xs = x.copy()
        la.iterative_solve(g, b, xs, 8, method, 0.5, 1e-3, PreconditionMethod.Jacobi)
        singles.append(xs)
    xb = [x.copy() for x in x0]
    la.iterative_solve3(g, bs, xb, 8, method, 0.5, 1e-3, PreconditionMethod.Jacobi)
    for k in range(3):
        assert np.isfinite(xb[k]).all()
        assert np.array_equal(xb[k], singles[k]), (k, rel_l2(xb[k], singles[k]))


def test_three_systems_need_a_lockstep_solver(ctx):
    a = random_spd_like(500, 0.01, seed=62)
    g = la.CsrMatrix.from_scipy(a, ctx)
    v = [np.ones(500) for _ in range(3)]
    with pytest.raises(orc_b200.OrcError) as e:
        la.iterative_solve3(g, v, [q.copy() for q in v], 5, SolutionMethod.Jacobi, 0.5, 1e-3, PreconditionMethod.Jacobi)
    assert e.value.code == orc_b200._lib.E_UNSUPPORTED


def test_galerkin_with_64_bit_keys_in_a_fresh_process():
    """The Galerkin kernel sorts 32-bit keys (column << log2(2 cap) | position) whenever the columns fit, 64-bit keys otherwise.
    The choice is made once per process; ORC_B200_GALERKIN_KEY64=1 forces the wide keys: same bit-exact results."""
    import os, subprocess, sys
    env = dict(os.environ, ORC_B200_GALERKIN_KEY64="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_linalg.py"), "-m", "gpu", "-x", "-q", "-k",
                          "test_galerkin_pattern_and_values or test_multigrid_levels_and_solution"], capture_output=True, text=True, env=env,
                         timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "passed" in out.stdout


@pytest.mark.parametrize("n,density", [(700, 0.01), (4999, 0.001), (5001, 0.001), (12000, 0.0005)])
def test_single_launch_bicgstab_is_bit_identical_to_the_reference(oracle, ctx, n, density):
    """small.cu: in reference-order mode a system of at most ORC_AUTO_EXACT_MAX_ROWS rows runs its whole BiCGSTAB loop in ONE
    launch (work vectors in shared memory up to 5000 rows, in global scratch above). Same arithmetic as the multi-launch
    reference-order path, so the result is bit-identical to the oracle (src/linear_algebra.rs:247-269)."""
    from orc_b200.settings import ReductionMode
    a = random_spd_like(n, density, seed=70 + n)
    g, o = both(oracle, ctx, a)
    rng = np.random.default_rng(11)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    for precond in (0, 1):
        x = x0.copy()
        l0 = ctx.launch_count()
        la.iterative_solve(g, b, x, 30, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod(precond), reduction_mode=ReductionMode.ReferenceOrder)
        launches = ctx.launch_count() - l0
        xo = oracle.iterative_solve(o, b, x0, 30, oracle.BICGSTAB, 0.5, 1e-3, precond)
        assert np.array_equal(x, xo), rel_l2(x, xo)
        assert launches <= 4, launches   # scaling + the one solver launch (the multi-launch path needs ~300)


def test_single_launch_gauss_seidel_on_a_mesh_like_matrix(oracle, ctx):
    """All sweeps of the lexicographic Gauss-Seidel in one launch (ready flags in shared memory): the 2-D five-point pattern of the
    reference's couette mesh (y-fastest numbering, neighbours i +- 1 and i +- 63), 8001 rows, 50 sweeps — bit-identical."""
    ny, nx = 63, 127
    n = nx * ny
    rng = np.random.default_rng(12)
    idx = np.arange(n).reshape(nx, ny)
    rows = np.concatenate([idx[:, :-1].ravel(), idx[:, 1:].ravel(), idx[:-1, :].ravel(), idx[1:, :].ravel()])
    cols = np.concatenate([idx[:, 1:].ravel(), idx[:, :-1].ravel(), idx[1:, :].ravel(), idx[:-1, :].ravel()])
    off = sp.csr_matrix((-rng.random(rows.size), (rows, cols)), shape=(n, n))
    a = (off + sp.diags(np.asarray(-off.sum(axis=1)).ravel() + 0.3)).tocsr()
    a.sort_indices()
    g, o = both(oracle, ctx, a)
    b = rng.standard_normal(n)
    x = np.zeros(n)
    l0 = ctx.launch_count()
    la.iterative_solve(g, b, x, 50, SolutionMethod.GaussSeidel, 0.8, 1e-3, PreconditionMethod.Jacobi)
    assert ctx.launch_count() - l0 <= 8
    xo = oracle.iterative_solve(o, b, np.zeros(n), 50, oracle.GAUSS_SEIDEL, 0.8, 1e-3, 1, gs_intended=1)
    assert np.array_equal(x, xo)


def test_multi_launch_small_system_paths_in_a_fresh_process():
    """ORC_B200_SMALL=0 switches the one-block kernels off: the multi-launch reference-order BiCGSTAB, the ticketed Gauss-Seidel
    dataflow sweep and the grid-wide restriction kernel (what larger systems run) must give the same bit-exact results on the
    same tests."""
    import os, subprocess, sys
    env = dict(os.environ, ORC_B200_SMALL="0")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_linalg.py"), "-m", "gpu", "-x", "-q", "-k",
                          "test_reference_order_reductions_make_solves_bit_identical or test_gauss_seidel_lexicographic_matches_intended_formula "
                          "or test_restriction_strongest_bit_exact or test_multigrid_levels_and_solution"],
                         capture_output=True, text=True, env=env, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "passed" in out.stdout
