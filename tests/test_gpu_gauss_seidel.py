"""Gauss-Seidel (linalg.cu: gauss_seidel) bit for bit on every kernel path, against the oracle's `gs_intended` sweep (lexicographic
mode) and against a plain NumPy model of the multicolour mode.

The paths: `k_gs_levels` (small.cu; symmetric pattern, 20 n bytes of shared memory fit, n <= 10 239), the ticketed dataflow sweep
`k_gs_sweep` (symmetric, larger n), `k_gs_serial` (pattern not structurally symmetric) and `k_colour_round` + `k_gs_colour`
(ORC_GS_MULTICOLOUR). The matrices reach the edges where those kernels go wrong: a level wider than the block of `k_gs_levels`
(GSL_T = 512 rows), rows with more than GSL_LOWER = 4 lower neighbours, rows longer than the 32 lanes of the ordered warp sum of
`k_gs_sweep`, dependency chains far deeper than 4 096 levels, an assembled tet momentum matrix, and the error flags of every path.

Rules of the model (as in tests/fast_model.py): no np.sum, `@` or np.dot; every row sums its off-diagonal products sequentially in
CSR order, sum = 0 then sum += a_ik x_k, and updates x_i = x_i (1 - w) + w (b_i - sum) / a_ii, the oracle's `gs_intended` expression
(oracle/orc_oracle.cpp, GaussSeidel arm) and the one every GPU kernel evaluates. The kernels are built with -fmad=false."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import fast_model as fm
from orc_b200 import synthetic as syn

MISSING = "Tried to access CsrMatrix element that hasn't been stored yet."
DIVERGED = "****** Solution diverged ******"
GSL_T, GSL_LOWER = 512, 4           # small.cu: block size and the lower neighbours a thread of k_gs_levels keeps in registers
SMALL_MAX_ROWS = 10239              # small.cu: gs_levels_smem(n) = 20 n + 8 <= SMALL_SMEM_MAX = 200 KiB
# (relaxation, Jacobi preconditioner, sweeps) of every case
SETTINGS = [(1.0, False, 3), (0.7, False, 4), (1.0, True, 5), (0.7, True, 3)]


# =============================================================================================================================
# the model
# =============================================================================================================================
class ModelPanic(RuntimeError):
    """The model met what makes the oracle panic (and the GPU raise its status): a missing a_ii or a NaN."""


def greedy_colours(A):
    """colour(i) = the smallest c >= 0 that no stored neighbour j < i has: the greedy colouring in row order."""
    if "colours" not in A.cache:
        colour = np.empty(A.nrows, np.int64)
        for i in range(A.nrows):
            cols = A.col[A.rowptr[i]:A.rowptr[i + 1]]
            used = set(colour[cols[cols < i]].tolist())
            c = 0
            while c in used:
                c += 1
            colour[i] = c
        A.cache["colours"] = colour
    return A.cache["colours"]


def _update_rows(A, d, b, x, rows, w, one_minus_w):
    """The new x of `rows` from the x given: per row sum = 0; sum += a_ik x_k over the stored k != i in CSR order."""
    if (d[rows] < 0).any():
        raise ModelPanic(MISSING)
    lo, ln = A.rowptr[rows], A.lengths[rows]
    s = np.zeros(rows.size)
    for k in range(int(ln.max()) if rows.size else 0):
        live = np.nonzero(ln > k)[0]
        e = lo[live] + k
        j = A.col[e]
        off = j != rows[live]
        live, e, j = live[off], e[off], j[off]
        s[live] = s[live] + A.val[e] * x[j]
    return x[rows] * one_minus_w + w * (b[rows] - s) / A.val[d[rows]]


def gauss_seidel(A, b, x, sweeps, w, jacobi, multicolour):
    """iterative_solve(..., GaussSeidel): optional Jacobi scaling (fast_model.jacobi_scale, pinned to k_jacobi_scale), then `sweeps`
    sweeps. Lexicographic: rows 0, 1, ... each with the newest x. Multicolour: the colours of greedy_colours in ascending order, all
    rows of a colour reading x as it stood when the colour started. A is a fast_model.Mat or a scipy matrix."""
    A = A if isinstance(A, fm.Mat) else fm.Mat.from_scipy(A)
    b = np.asarray(b, dtype=np.float64)
    x = np.array(x, dtype=np.float64)
    if jacobi:
        A, pinv, has = fm.jacobi_scale(A)
        b = fm.jacobi_scale_rhs(pinv, has, b)
    if sweeps == 0 or A.nrows == 0:
        return x
    d = A.diag_index()
    one_minus_w = 1.0 - w
    if multicolour:
        colour = greedy_colours(A)
        groups = [np.nonzero(colour == c)[0] for c in range(int(colour.max()) + 1)]
    for _ in range(sweeps):
        if multicolour:
            for rows in groups:
                x[rows] = _update_rows(A, d, b, x, rows, w, one_minus_w)
                if np.isnan(x[rows]).any():
                    raise ModelPanic(DIVERGED)
            continue
        rp, col, val = A.rowptr, A.col, A.val
        for i in range(A.nrows):   # plain Python floats: IEEE doubles, one rounding per operation
            s = 0.0
            for k in range(rp[i], rp[i + 1]):
                if col[k] != i:
                    s += float(val[k]) * float(x[col[k]])
            if d[i] < 0:
                raise ModelPanic(MISSING)
            x[i] = float(x[i]) * one_minus_w + w * (float(b[i]) - s) / float(val[d[i]])
            if np.isnan(x[i]):
                raise ModelPanic(DIVERGED)
    return x


# =============================================================================================================================
# matrices: diagonally dominant values on the patterns the kernels care about
# =============================================================================================================================
def with_values(pattern, seed):
    """Values on a pattern (the diagonal must be stored): off-diagonals -U(0, 1), a_ii = sum |a_ij| + 0.5 + U(0, 1)."""
    p = sp.csr_matrix(pattern, dtype=np.float64)
    p.sum_duplicates()
    p.sort_indices()
    n = p.shape[0]
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n), np.diff(p.indptr))
    off = p.indices != rows
    val = np.empty(p.nnz)
    val[off] = -rng.random(int(off.sum()))
    dom = np.bincount(rows[off], weights=-val[off], minlength=n)
    val[~off] = dom[rows[~off]] + 0.5 + rng.random(int((~off).sum()))
    return sp.csr_matrix((val, p.indices.copy(), p.indptr.copy()), shape=(n, n))


def symmetric_pattern(n, pairs_i, pairs_j):
    i, j = np.asarray(pairs_i), np.asarray(pairs_j)
    keep = i != j
    i, j = i[keep], j[keep]
    r = np.concatenate([i, j, np.arange(n)])
    c = np.concatenate([j, i, np.arange(n)])
    return sp.csr_matrix((np.ones(r.size), (r, c)), shape=(n, n))


def dense(n, seed):
    return with_values(np.ones((n, n)), seed)


def two_by_two_blocks(nblocks=3000):
    """3 000 independent 2 x 2 blocks: the first dependency level holds 3 000 rows, wider than GSL_T."""
    return with_values(sp.kron(sp.identity(nblocks), np.ones((2, 2))), 3)


def random_rows(n=9000, seed=4):
    """A random symmetric pattern with row lengths from 1 to about 90: rows longer than 32 and with more than GSL_LOWER lower
    neighbours; every 97th row is alone (length 1)."""
    rng = np.random.default_rng(seed)
    alone = np.arange(n) % 97 == 0
    others = np.nonzero(~alone)[0]
    m = rng.integers(0, 45, size=n)
    m[alone] = 0
    src = np.repeat(np.arange(n), m)
    return with_values(symmetric_pattern(n, src, rng.choice(others, size=src.size)), seed)


def box_pattern(oracle, nx, ny, nz):
    """The seven-point pattern of syn.hex_box (the mesh's own cell numbering), as initialize_momentum_matrix stores it."""
    om = oracle.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(nx, ny, nz)))
    rp, co, _ = om.init_momentum_matrix().arrays()
    n = rp.size - 1
    return sp.csr_matrix((np.ones(co.size), co, rp), shape=(n, n))


def chain(n=20000):
    """Tridiagonal: one dependency chain of depth n."""
    return with_values(sp.diags([np.ones(n - 1), np.ones(n), np.ones(n - 1)], [-1, 0, 1]), 5)


def long_rows(n=12000, seed=6):
    """A sparse symmetric pattern in which every 60th row couples to 40-200 others: rows longer than the 32 lanes of one pass of
    the ordered warp sum of k_gs_sweep (two to seven passes)."""
    rng = np.random.default_rng(seed)
    src = [np.arange(n - 1)]
    dst = [np.arange(1, n)]
    hubs = np.arange(0, n, 60)
    k = rng.integers(40, 200, size=hubs.size)
    src.append(np.repeat(hubs, k))
    dst.append(rng.integers(0, n, size=int(k.sum())))
    extra = rng.integers(0, n, size=(2, n))
    src.append(extra[0])
    dst.append(extra[1])
    return with_values(symmetric_pattern(n, np.concatenate(src), np.concatenate(dst)), seed)


def nonsymmetric(n=15000, seed=7):
    rng = np.random.default_rng(seed)
    r = rng.integers(0, n, size=4 * n)
    c = rng.integers(0, n, size=4 * n)
    keep = r != c
    pat = sp.csr_matrix((np.ones(int(keep.sum()) + n), (np.concatenate([r[keep], np.arange(n)]), np.concatenate([c[keep], np.arange(n)]))),
                        shape=(n, n))
    return with_values(pat, seed)


def is_symmetric_pattern(a):
    p = (a != 0).astype(np.int8)
    return (p != p.T).nnz == 0


def both(oracle, ctx, a):
    from orc_b200 import linear_algebra as la
    a = a.tocsr()
    a.sort_indices()
    return la.CsrMatrix.from_scipy(a, ctx), oracle.Csr.from_arrays(a.shape[0], a.shape[1], a.indptr, a.indices, a.data)


def inputs(n, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(n), rng.standard_normal(n)


# =============================================================================================================================
# CPU: the model against the oracle, and the properties of the colouring
# =============================================================================================================================
@pytest.mark.parametrize("name", ["dense1", "dense2", "dense40", "blocks", "chain300", "random300", "nonsym300"])
def test_lexicographic_model_is_the_oracle(oracle, name):
    a = {"dense1": lambda: dense(1, 1), "dense2": lambda: dense(2, 2), "dense40": lambda: dense(40, 3), "blocks": lambda: two_by_two_blocks(60),
         "chain300": lambda: chain(300), "random300": lambda: random_rows(300, 8), "nonsym300": lambda: nonsymmetric(300, 9)}[name]()
    o = oracle.Csr.from_arrays(a.shape[0], a.shape[1], a.indptr, a.indices, a.data)
    b, x0 = inputs(a.shape[0], 11)
    for w, jac, sweeps in SETTINGS:
        want = oracle.iterative_solve(o, b, x0, sweeps, oracle.GAUSS_SEIDEL, w, 1e-3, int(jac), gs_intended=1)
        got = gauss_seidel(a, b, x0, sweeps, w, jac, multicolour=False)
        assert np.array_equal(got, want), (name, w, jac, sweeps)


def _without_diagonal(a, i):
    a = a.tolil()
    a[i, i] = 0
    a = a.tocsr()
    a.eliminate_zeros()
    a.sort_indices()
    return a


@pytest.mark.parametrize("n", [1, 2, 3, 17, 64])
def test_multicolour_model_on_a_dense_pattern_is_the_oracle(oracle, n):
    """Every row of a dense pattern neighbours every other: n colours, one row each, swept in row order."""
    a = dense(n, n)
    assert np.array_equal(greedy_colours(fm.Mat.from_scipy(a)), np.arange(n))
    o = oracle.Csr.from_arrays(n, n, a.indptr, a.indices, a.data)
    b, x0 = inputs(n, 12)
    for w, jac, sweeps in SETTINGS:
        want = oracle.iterative_solve(o, b, x0, sweeps, oracle.GAUSS_SEIDEL, w, 1e-3, int(jac), gs_intended=1)
        assert np.array_equal(gauss_seidel(a, b, x0, sweeps, w, jac, multicolour=True), want), (n, w, jac, sweeps)


@pytest.mark.parametrize("build", [lambda: random_rows(2000, 13), lambda: long_rows(3000, 14), lambda: two_by_two_blocks(500), lambda: chain(1000)])
def test_greedy_colouring_is_proper(build):
    A = fm.Mat.from_scipy(build())
    colour = greedy_colours(A)
    rows = np.repeat(np.arange(A.nrows), A.lengths)
    off = A.col != rows
    assert not (colour[rows[off]] == colour[A.col[off]]).any()
    # greedy: each row's colour is the smallest its lower neighbours leave free, so every smaller colour is taken by one of them
    lower = off & (A.col < rows)
    for i in np.random.default_rng(0).choice(A.nrows, 200, replace=False):
        seen = set(colour[A.col[(rows == i) & lower]].tolist())
        assert set(range(colour[i])) <= seen


def test_seven_point_box_gets_two_colours(oracle):
    """A hex box numbers its cells lexicographically, so the greedy colouring of the seven-point pattern is a checkerboard."""
    p = box_pattern(oracle, 12, 10, 8)
    colour = greedy_colours(fm.Mat.from_scipy(with_values(p, 0)))
    assert colour.max() == 1
    assert 0 < np.count_nonzero(colour) < p.shape[0]


def test_multicolour_model_converges():
    a = with_values(symmetric_pattern(800, *np.random.default_rng(15).integers(0, 800, size=(2, 3200))), 15)
    xs = np.random.default_rng(7).standard_normal(800)
    b = a @ xs
    x = gauss_seidel(a, b, np.zeros(800), 60, 1.0, False, multicolour=True)
    assert np.linalg.norm(x - xs) / np.linalg.norm(xs) < 1e-6


# =============================================================================================================================
# GPU: every path against the oracle (lexicographic) and the model (multicolour)
# =============================================================================================================================
_MATS = {}
CASES = ["dense1", "dense2", "blocks3000", "random9000", "box48x40x30", "chain20000", "long_rows12000", "tet16_momentum", "nonsym15000"]


def tet_momentum(ctx):
    """The x-momentum matrix the GPU assembles on syn.tet_box(16, 16, 16) (24 576 cells), as in test_gpu_assembly.py."""
    import orc_b200
    from orc_b200 import discretization as disc
    from cases import smooth_fields
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.tet_box(16, 16, 16)))
    syn.channel_bcs(pm, fully_3d=True)
    u, v, w, p = smooth_fields(pm.export())
    g_di, *_ = disc.build_momentum_diffusion_matrix(pm, 1e-3, ctx)
    g_a = [disc.initialize_momentum_matrix(pm, ctx) for _ in range(3)]
    disc.build_momentum_advection_matrices(*g_a, g_di, pm, u, v, w, p, orc_b200.NumericalSettings(), 1000.0)
    return g_a[0].to_scipy()


def matrix(name, oracle, ctx):
    if name not in _MATS:
        a = {"dense1": lambda: dense(1, 1), "dense2": lambda: dense(2, 2), "blocks3000": two_by_two_blocks, "random9000": random_rows,
             "box48x40x30": lambda: with_values(box_pattern(oracle, 48, 40, 30), 9), "chain20000": chain, "long_rows12000": long_rows,
             "tet16_momentum": lambda: tet_momentum(ctx), "nonsym15000": nonsymmetric}[name]()
        a = a.tocsr()
        a.sort_indices()
        _MATS[name] = a
    return _MATS[name]


def expected_path(a):
    if not is_symmetric_pattern(a):
        return "k_gs_serial"
    return "k_gs_levels" if a.shape[0] <= SMALL_MAX_ROWS else "k_gs_sweep"


def test_the_cases_reach_the_kernel_edges(oracle):
    """What each matrix is for (the paths with ORC_B200_SMALL unset). The tet momentum matrix needs the GPU to assemble: it is a
    mesh matrix (structurally symmetric) of 24 576 rows, so it runs k_gs_sweep."""
    ctx = None
    cpu_cases = [c for c in CASES if c != "tet16_momentum"]
    paths = {n: expected_path(matrix(n, oracle, ctx)) for n in cpu_cases}
    assert paths == {"dense1": "k_gs_levels", "dense2": "k_gs_levels", "blocks3000": "k_gs_levels", "random9000": "k_gs_levels",
                     "box48x40x30": "k_gs_sweep", "chain20000": "k_gs_sweep", "long_rows12000": "k_gs_sweep", "nonsym15000": "k_gs_serial"}
    lens = {n: np.diff(matrix(n, oracle, ctx).indptr) for n in cpu_cases}
    assert lens["random9000"].min() == 1 and 32 < lens["random9000"].max() <= 100
    a = matrix("random9000", oracle, ctx).tocoo()
    assert np.bincount(a.row[a.col < a.row], minlength=a.shape[0]).max() > GSL_LOWER
    assert 32 < lens["long_rows12000"].max() and (lens["long_rows12000"] > 64).sum() > 50
    assert matrix("box48x40x30", oracle, ctx).shape[0] == 57600


gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("name", CASES)
def test_lexicographic_matches_the_oracle(oracle, ctx, name):
    from orc_b200 import linear_algebra as la
    from orc_b200.settings import SolutionMethod, PreconditionMethod
    a = matrix(name, oracle, ctx)
    g, o = both(oracle, ctx, a)
    b, x0 = inputs(a.shape[0], 21)
    for w, jac, sweeps in SETTINGS:
        x = x0.copy()
        la.iterative_solve(g, b, x, sweeps, SolutionMethod.GaussSeidel, w, 1e-3, PreconditionMethod(int(jac)))
        want = oracle.iterative_solve(o, b, x0, sweeps, oracle.GAUSS_SEIDEL, w, 1e-3, int(jac), gs_intended=1)
        bad = np.flatnonzero(x != want)
        assert bad.size == 0, (name, w, jac, sweeps, f"{bad.size} rows differ, first {bad[:5]}")


@gpu
@pytest.mark.parametrize("name", [c for c in CASES if c != "nonsym15000"])
def test_multicolour_matches_the_model(oracle, ctx, name):
    from orc_b200 import linear_algebra as la
    from orc_b200.settings import SolutionMethod, PreconditionMethod, GaussSeidelMode
    a = matrix(name, oracle, ctx)
    g = la.CsrMatrix.from_scipy(a, ctx)
    A = fm.Mat.from_scipy(a)
    b, x0 = inputs(a.shape[0], 22)
    for w, jac, sweeps in SETTINGS:
        x = x0.copy()
        la.iterative_solve(g, b, x, sweeps, SolutionMethod.GaussSeidel, w, 1e-3, PreconditionMethod(int(jac)), gs_mode=GaussSeidelMode.Multicolour)
        want = gauss_seidel(A, b, x0, sweeps, w, jac, multicolour=True)
        bad = np.flatnonzero(x != want)
        assert bad.size == 0, (name, w, jac, sweeps, f"{bad.size} rows differ, first {bad[:5]}")


@gpu
def test_multicolour_launches_once_per_colour_and_sweep(oracle, ctx):
    """On the 48 x 40 x 30 box: one colouring launch per dependency level (nx + ny + nz - 2 = 116), then 2 colours per sweep."""
    from orc_b200 import linear_algebra as la
    from orc_b200.settings import SolutionMethod, PreconditionMethod, GaussSeidelMode
    a = matrix("box48x40x30", oracle, ctx)
    g = la.CsrMatrix.from_scipy(a, ctx)
    b, x0 = inputs(a.shape[0], 23)
    launches = {}
    for sweeps in (1, 3, 5):   # the first call also locates the diagonal of g (k_find_diag, cached on the handle): not counted
        l0 = ctx.launch_count()
        la.iterative_solve(g, b, x0.copy(), sweeps, SolutionMethod.GaussSeidel, 1.0, 1e-3, PreconditionMethod.Jacobi,
                           gs_mode=GaussSeidelMode.Multicolour)
        launches[sweeps] = ctx.launch_count() - l0
    assert launches[5] - launches[3] == 2 * 2, launches
    assert 0 <= launches[3] - (116 + 2 * 3) <= 3, launches   # + the Jacobi scaling and the symmetry check of the scaled copy


@gpu
def test_multicolour_refuses_a_nonsymmetric_pattern(oracle, ctx):
    """Row 0 = {0, 1}, row 1 = {1}: both rows would get colour 0, and the sweep would write x_1 while row 0 reads it."""
    import orc_b200
    from orc_b200 import linear_algebra as la
    from orc_b200.settings import SolutionMethod, PreconditionMethod, GaussSeidelMode
    for a in (sp.csr_matrix(np.array([[2.0, -1.0], [0.0, 2.0]])), matrix("nonsym15000", oracle, ctx)):
        g = la.CsrMatrix.from_scipy(a, ctx)
        b, x0 = inputs(a.shape[0], 24)
        x = x0.copy()
        with pytest.raises(orc_b200.OrcError) as e:
            la.iterative_solve(g, b, x, 3, SolutionMethod.GaussSeidel, 1.0, 1e-3, PreconditionMethod.NONE, gs_mode=GaussSeidelMode.Multicolour)
        assert e.value.code == orc_b200._lib.E_UNSUPPORTED and "structurally symmetric" in e.value.message
        assert np.array_equal(x, x0)


MODES = ["levels", "sweep", "serial", "multicolour"]


def path_matrix(mode, oracle, ctx):
    return {"levels": lambda: random_rows(3000, 30), "sweep": lambda: matrix("long_rows12000", oracle, ctx),
            "serial": lambda: nonsymmetric(3000, 31), "multicolour": lambda: random_rows(3000, 32)}[mode]()


def _gpu_solve(ctx, a, b, x, sweeps, mode, jac=False):
    from orc_b200 import linear_algebra as la
    from orc_b200.settings import SolutionMethod, PreconditionMethod, GaussSeidelMode
    g = la.CsrMatrix.from_scipy(a, ctx)
    gs = GaussSeidelMode.Multicolour if mode == "multicolour" else GaussSeidelMode.Lexicographic
    return la.iterative_solve(g, b, x, sweeps, SolutionMethod.GaussSeidel, 0.7, 1e-3, PreconditionMethod(int(jac)), gs_mode=gs)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_zero_sweeps_leave_x_unchanged(oracle, ctx, mode):
    a = path_matrix(mode, oracle, ctx)
    b, x0 = inputs(a.shape[0], 25)
    for jac in (False, True):
        x = x0.copy()
        _gpu_solve(ctx, a, b, x, 0, mode, jac)
        assert np.array_equal(x, x0), (mode, jac)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_errors_on_every_path(oracle, ctx, mode):
    """A symmetric stored pair (i, j), (j, i) whose row i stores no a_ii, without the Jacobi scaling (which would drop the row):
    the reference's `get` panic, ORC_E_MISSING_ENTRY. A NaN in b: ORC_E_GS_DIVERGED. The oracle panics with the same messages."""
    import orc_b200
    a = path_matrix(mode, oracle, ctx)
    n = a.shape[0]
    i = int(np.flatnonzero(np.diff(a.indptr) > 3)[n // 100])
    j = int(next(c for c in a.indices[a.indptr[i]:a.indptr[i + 1]] if c != i))
    assert a[j, i] != 0 or mode == "serial"
    holed = _without_diagonal(a, i)
    b, x0 = inputs(n, 26)
    nan_b = b.copy()
    nan_b[n // 2] = np.nan
    for m, rhs, code, msg in ((holed, b, orc_b200._lib.E_MISSING_ENTRY, MISSING), (a, nan_b, orc_b200._lib.E_GS_DIVERGED, DIVERGED)):
        with pytest.raises(orc_b200.OrcError) as e:
            _gpu_solve(ctx, m, rhs, x0.copy(), 3, mode)
        assert e.value.code == code and e.value.message == msg, (mode, e.value.code, e.value.message)
        o = oracle.Csr.from_arrays(n, n, m.indptr, m.indices, m.data)
        with pytest.raises(oracle.OraclePanic, match=msg.replace("*", r"\*")):
            oracle.iterative_solve(o, rhs, x0, 3, oracle.GAUSS_SEIDEL, 0.7, 1e-3, 0, gs_intended=1)
        with pytest.raises(ModelPanic, match=msg.replace("*", r"\*")):
            gauss_seidel(m, rhs, x0, 3, 0.7, False, multicolour=mode == "multicolour")


@gpu
def test_lexicographic_cases_through_the_dataflow_sweep_in_a_fresh_process():
    """ORC_B200_SMALL=0 (read once per process) switches k_gs_levels off: the small lexicographic cases then run k_gs_sweep."""
    env = dict(os.environ, ORC_B200_SMALL="0")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_gauss_seidel.py"), "-m", "gpu", "-x", "-q", "-k",
                          "test_lexicographic_matches_the_oracle or test_zero_sweeps_leave_x_unchanged or test_errors_on_every_path"],
                         capture_output=True, text=True, env=env, timeout=900, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "passed" in out.stdout


# =============================================================================================================================
# GPU: two multicolour SIMPLE iterations against tests/fast_simple.py with the model as its solve
# =============================================================================================================================
@gpu
def test_simple_iterations_with_multicolour_gauss_seidel(oracle):
    import bench
    import fast_simple as fs
    import orc_b200
    from orc_b200.settings import GaussSeidelMode
    from cases import make_pair, settings_pair
    pm, om = make_pair(oracle, syn.hex_box(24, 24, 24))
    for m in (pm, om):
        syn.channel_bcs(m)
    ps, os_ = settings_pair(oracle, solver_type=oracle.GAUSS_SEIDEL)
    ps.gs_mode = GaussSeidelMode.Multicolour
    n = pm.n_cells

    def solve(a, B, X, pos=None):
        A = fm.Mat.from_handle(a)
        return np.stack([gauss_seidel(A, b, x, os_.iterations, os_.relaxation, os_.preconditioner == oracle.PC_JACOBI, multicolour=True)
                         for b, x in zip(B, X)])

    model = fs.simple_iterations(om, os_, bench.RHO, bench.MU, [np.zeros(n)] * 4, 2, solve)
    u, v, w, p = (np.zeros(n) for _ in range(4))
    orc_b200.solve_steady(pm, u, v, w, p, ps, bench.RHO, bench.MU, 2, 1, on_report=lambda d: None)
    for name, got in zip("uvwp", (u, v, w, p)):
        want = model[-1][name]
        assert np.isfinite(want).all() and np.abs(want).max() > 0, name
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (name, f"{bad.size} of {n} cells differ")
