"""The fast-mode (ORC_REDUCE_FAST) kernels bit for bit against tests/fast_model.py, the NumPy restatement of their summation
order, at the sizes and launch regimes the benchmark runs. Every comparison is np.array_equal: the fast mode's order depends on
the matrix and its size only, so even 50 unguarded BiCGSTAB iterations on 2.1 M rows, where no tolerance against the oracle
means anything (DESIGN.md §5), are pinned exactly.

Launch regimes: the fused reductions work in nv = min(tiles, 3552) virtual blocks. nv beyond the resident blocks (888 for three
systems, 1184 for one on a B200) makes a real block park several virtual blocks (vb_park / vb_publish with lv > 0); more than
3552 tiles makes every thread walk several tiles. Each case prints its SpMV class (lanes per row G), nv and tiles per virtual
block, so the coverage can be read off the log (pytest -s).

The Multigrid section runs the 128^3 benchmark mesh: 5 inner iterations (one K = 1 and one K = 3 Multigrid solve, with and without
the locality ordering of the coarse levels) and the benchmark's 50-iteration K = 3 momentum BiCGSTAB on the fine matrix."""
import numpy as np
import pytest

import fast_model as fm
import orc_b200
from orc_b200 import discretization as disc
from orc_b200 import linear_algebra as la
from orc_b200 import synthetic as syn
from orc_b200.settings import PreconditionMethod, ReductionMode, SolutionMethod
from cases import settings_pair, smooth_fields
from test_fast_model import lengths_with_average

pytestmark = pytest.mark.gpu
RHO, MU = 1000.0, 1e-3


def describe(A, what=""):
    G, nv, per = fm.spmv_launch(A)
    line = f"{what} rows={A.nrows} nnz/row={A.nnz / max(A.nrows, 1):.2f} G={G} nv={nv} tiles/vb={per}"
    print(line)
    return line


def mismatch(got, want, what):
    """None if bit-identical, else a line that says where."""
    got, want = np.asarray(got), np.asarray(want)
    if got.shape == want.shape and np.array_equal(got, want):
        return None
    if got.shape != want.shape:
        return f"{what}: shape {got.shape} != {want.shape}"
    bad = np.argwhere(got != want)
    first = tuple(int(v) for v in bad[0])
    scale = np.abs(want).max() or 1.0
    return (f"{what}: {len(bad)} of {want.size} differ, first at {first}: {got[first]!r} vs {want[first]!r}, "
            f"max |diff| / max |model| = {np.nanmax(np.abs(got - want)) / scale:.3e}")


def random_pattern(lengths, ncols, seed, anchor_diagonal=False):
    """Sorted unique columns per row with random gaps of 1-3 (vectorised). With anchor_diagonal (square, ncols = n) every row
    stores (i, i) and its columns wrap around the matrix edge."""
    rng = np.random.default_rng(seed)
    n = lengths.size
    rp = np.zeros(n + 1, np.int64)
    rp[1:] = np.cumsum(lengths)
    nnz = int(rp[-1])
    rows = np.repeat(np.arange(n), lengths)
    cs = np.cumsum(rng.integers(1, 4, nnz))
    base = np.where(rp[:-1] > 0, cs[np.maximum(rp[:-1] - 1, 0)], 0)
    within = cs - np.repeat(base, lengths)            # 1 .. 3 len, increasing within a row
    span = np.where(lengths > 0, within[np.maximum(rp[1:] - 1, 0)], 0)
    assert span.max() < ncols
    if not anchor_diagonal:
        start = (rng.random(n) * (ncols - span)).astype(np.int64)
        return rp, np.repeat(start, lengths) + within - 1, rows
    anchor = rp[:-1] + rng.integers(0, lengths)
    col = (rows + within - np.repeat(within[anchor], lengths)) % ncols
    order = np.lexsort((col, rows))
    return rp, col[order], rows


def spmv_matrix(n, avg, ncols, seed):
    lengths = lengths_with_average(n, avg, seed)
    rp, col, _ = random_pattern(lengths, ncols, seed)
    rng = np.random.default_rng(seed + 1)
    val = rng.standard_normal(col.size) * 10.0 ** rng.uniform(-3, 3, col.size)
    return rp, col, val


def solve_matrix(n, avg, seed, dominance):
    """Square, every diagonal stored, negative off-diagonals, diagonal = (1 + dominance) * sum |off| + dominance * U(0, 1)."""
    lengths = lengths_with_average(n, avg, seed, long_row=0, empty_row=False)
    rp, col, rows = random_pattern(lengths, n, seed, anchor_diagonal=True)
    rng = np.random.default_rng(seed + 2)
    val = -rng.random(col.size)
    diag = col == rows
    assert diag.sum() == n
    off = np.bincount(rows[~diag], weights=-val[~diag], minlength=n)
    val[diag] = (1.0 + dominance) * off + dominance * rng.random(n)
    return rp, col, val


# ---- SpMV: every dispatch class x every virtual-block regime ------------------------------------------------------------
TILES = {"nv1": 1, "nv37": 37, "nv600": 600, "nv1000": 1000, "nv2000": 2000, "nv3552": 3552, "2perVB": 7104, "9perVB": 8 * 3552 + 1}
SPMV_CASES = [(avg, r) for avg in (7, 10, 17, 32, 107) for r in TILES if not (r == "9perVB" and avg in (10, 107))]


@pytest.mark.parametrize("avg,regime", SPMV_CASES, ids=[f"avg{a}-{r}" for a, r in SPMV_CASES])
def test_spmv_bit_exact(ctx, avg, regime):
    rpb = fm.SPMV_BLOCK // (1 if avg < 10 else 4 if avg < 32 else 8)
    tiles = TILES[regime]
    n = tiles * rpb - (0 if regime == "nv3552" else 3)   # a partial last tile, except for the exact 3552
    ncols = max(n, 3 * (4 * avg + 70) + 1)
    rp, col, val = spmv_matrix(n, avg, ncols, seed=avg * 7 + tiles)
    A = fm.Mat(rp, col, val, ncols)
    describe(A, f"spmv avg={avg} {regime}:")
    assert fm.spmv_launch(A)[1] == min(tiles, 3552)
    g = la.CsrMatrix.from_arrays(n, ncols, rp, col, val, ctx)
    x = np.random.default_rng(tiles).standard_normal(ncols)
    err = mismatch(g.spmv(x), fm.spmv(A, x)[0], f"spmv avg={avg} {regime}")
    assert err is None, err


def test_spmv_class_does_not_depend_on_an_earlier_solve(ctx):
    """A reference-order solve on the context must not switch a later standalone SpMV of long rows to the thread-per-row kernel."""
    rp, col, val = solve_matrix(3000, 7, seed=1, dominance=0.5)
    small = la.CsrMatrix.from_arrays(3000, 3000, rp, col, val, ctx)
    la.iterative_solve(small, np.ones(3000), np.zeros(3000), 3, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod.Jacobi,
                       reduction_mode=ReductionMode.ReferenceOrder)
    rp, col, val = spmv_matrix(5000, 107, 5000, seed=2)
    A = fm.Mat(rp, col, val, 5000)
    x = np.random.default_rng(3).standard_normal(5000)
    err = mismatch(la.CsrMatrix.from_arrays(5000, 5000, rp, col, val, ctx).spmv(x), fm.spmv(A, x)[0], "spmv after a reference-order solve")
    assert err is None, err


# ---- BiCGSTAB, K = 1 and K = 3, both preconditioners --------------------------------------------------------------------
# (average row length, rows, longest solve): nv from 1 over the resident-block limits to 3552 with two tiles per virtual block
BICG_CASES = [(7, 200, 50), (7, 37 * 256 - 5, 50), (7, 1000 * 256 - 7, 50), (7, 2000 * 256 + 3, 5), (7, 3552 * 256, 5),
              (7, 7104 * 256 - 100, 5), (17, 37 * 64 - 1, 50), (17, 1100 * 64 + 5, 50), (17, 3 * 3552 * 64 + 9, 5),
              (107, 37 * 32 - 3, 50), (107, 1100 * 32 + 1, 50), (107, 2 * 3552 * 32 + 7, 5)]


@pytest.mark.parametrize("avg,n,iters", BICG_CASES, ids=[f"avg{a}-n{n}" for a, n, _ in BICG_CASES])
@pytest.mark.parametrize("pc", [1, 0], ids=["jacobi", "none"])
def test_bicgstab_bit_exact(ctx, avg, n, iters, pc):
    """Iteration 1 isolates EP_RESID_INIT, EP_SUM_ALPHA, EP_DOTS_OMEGA and k_bicg_xr; iteration 2 adds beta; 5 and 50 the rest.
    The K = 1 solve is system 0 of the K = 3 batch."""
    rp, col, val = solve_matrix(n, avg, seed=n, dominance=1e-3)
    A = fm.Mat(rp, col, val, n)
    Ap, pinv, has = fm.jacobi_scale(A) if pc else (A, None, None)
    describe(Ap, f"bicgstab pc={pc}:")
    print(f"  k_bicg_xr nv={fm.nv_for(-(-n // 256))}")
    rng = np.random.default_rng(n + pc)
    B = rng.standard_normal((3, n))
    X0 = rng.standard_normal((3, n))
    snaps = {k: None for k in (1, 2, 5, 50) if k <= iters}
    fm.bicgstab(Ap, fm.jacobi_scale_rhs(pinv, has, B) if pc else B, X0, max(snaps), snapshots=snaps)
    g = la.CsrMatrix.from_arrays(n, n, rp, col, val, ctx)
    errs = []
    for it, want in snaps.items():
        x1 = X0[0].copy()
        la.iterative_solve(g, B[0], x1, it, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod(pc))
        errs.append(mismatch(x1, want[0], f"K=1 {it} iterations"))
        xs = [q.copy() for q in X0]
        la.iterative_solve3(g, list(B), xs, it, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod(pc))
        errs.append(mismatch(np.stack(xs), want, f"K=3 {it} iterations"))
        assert np.isfinite(want).all()
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)


# ---- Jacobi, K = 1, in the lv > 0 regime -------------------------------------------------------------------------------
@pytest.mark.parametrize("avg,n", [(7, 2000 * 256 + 3), (17, 2000 * 64 + 5)], ids=["avg7", "avg17"])
def test_jacobi_bit_exact(ctx, avg, n):
    rp, col, val = solve_matrix(n, avg, seed=n + 1, dominance=1.0)
    A = fm.Mat(rp, col, val, n)
    Ap, pinv, has = fm.jacobi_scale(A)
    describe(Ap, "jacobi:")
    g = la.CsrMatrix.from_arrays(n, n, rp, col, val, ctx)
    b = np.random.default_rng(n).standard_normal(n)
    bp = fm.jacobi_scale_rhs(pinv, has, b[None])[0]
    errs = []
    for iters, thr in ((7, 1e-30), (200, 1e-3)):
        want, ran, r = fm.jacobi(Ap, bp, np.zeros(n), iters, 0.5, thr)
        print(f"  {iters} iterations, threshold {thr}: the model ran {ran}, last residual {r:.3e}")
        if iters == 200:
            assert 2 < ran < 200      # the convergence latch fired
        x = np.zeros(n)
        la.iterative_solve(g, b, x, iters, SolutionMethod.Jacobi, 0.5, thr, PreconditionMethod.Jacobi)
        errs.append(mismatch(x, want, f"jacobi {iters}"))
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)


# ---- Multigrid and the momentum BiCGSTAB on the 128^3 benchmark mesh ----------------------------------------------------
@pytest.fixture(scope="module")
def bench_mesh(oracle, ctx):
    """The x-momentum matrix the GPU assembles on the 128^3 bench mesh (as in test_gpu_scale's AMG set-up test), its arrays, the
    cell centroids that drive the locality ordering, and the Multigrid hierarchy of the 5-iteration traced solve."""
    arrays = syn.hex_box(128, 128, 128)
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    del arrays
    syn.channel_bcs(pm)
    ps, _ = settings_pair(oracle)
    ex = pm.export()
    u, v, w, p = smooth_fields(ex)
    g_di, *_ = disc.build_momentum_diffusion_matrix(pm, MU, ctx)
    g_a = [disc.initialize_momentum_matrix(pm, ctx) for _ in range(3)]
    disc.build_momentum_advection_matrices(*g_a, g_di, pm, u, v, w, p, ps, RHO)
    g = g_a[0]
    n = g.dims[0]
    A = fm.Mat.from_handle(g)
    rng = np.random.default_rng(128)
    B = rng.standard_normal((3, n))
    x_trace, glev = la.multigrid_trace(g, B[0], np.zeros(n), iteration_count=5)
    levels = [(fm.Mat.from_handle(r), fm.Mat.from_handle(a)) for r, a in glev]
    return dict(pm=pm, g=g, A=A, n=n, B=B, x_trace=x_trace, levels=levels, pos=fm.Positions(ex["cell_centroid"]))


def test_bench_mesh_spmv_bit_exact(bench_mesh):
    s = bench_mesh
    describe(s["A"], "128^3 momentum matrix:")
    x = np.random.default_rng(1).standard_normal(s["n"])
    err = mismatch(s["g"].spmv(x), fm.spmv(s["A"], x)[0], "128^3 spmv")
    assert err is None, err


def test_bench_mesh_multigrid_bit_exact(bench_mesh, monkeypatch):
    """Multigrid, 5 inner iterations: with the locality ordering (the benchmark's path; K = 1 traced and K = 3), and without it
    through ORC_B200_REORDER=0 and through a hint-free re-upload of the same arrays."""
    s = bench_mesh
    n, B, levels, pos = s["n"], s["B"], s["levels"], s["pos"]
    for l, (_, a) in enumerate(levels):
        S = fm.jacobi_scale(a)[0]
        describe(S, f"level {l + 1} (reordered: {fm.reorder_applies(a, l + 1, pos)}):")
    assert fm.reorder_applies(levels[0][1], 1, pos)
    errs = []
    want = fm.iterative_solve(s["A"], B, np.zeros((3, n)), 5, fm.MULTIGRID, levels=levels, pos=pos)
    errs.append(mismatch(s["x_trace"], want[0], "multigrid K=1, ordering on (traced)"))
    xs = [np.zeros(n) for _ in range(3)]
    la.iterative_solve3(s["g"], list(B), xs, 5, SolutionMethod.Multigrid, 0.5, 1e-3, PreconditionMethod.Jacobi)
    errs.append(mismatch(np.stack(xs), want, "multigrid K=3, ordering on"))
    want_off = fm.iterative_solve(s["A"], B[:1], np.zeros((1, n)), 5, fm.MULTIGRID, levels=levels)[0]
    assert not np.array_equal(want_off, want[0])
    monkeypatch.setenv("ORC_B200_REORDER", "0")
    x = np.zeros(n)
    la.iterative_solve(s["g"], B[0], x, 5, SolutionMethod.Multigrid, 0.5, 1e-3, PreconditionMethod.Jacobi)
    errs.append(mismatch(x, want_off, "multigrid K=1, ORC_B200_REORDER=0"))
    monkeypatch.delenv("ORC_B200_REORDER")
    A = s["A"]
    bare = la.CsrMatrix.from_arrays(n, n, A.rowptr, A.col, A.val)
    x = np.zeros(n)
    la.iterative_solve(bare, B[0], x, 5, SolutionMethod.Multigrid, 0.5, 1e-3, PreconditionMethod.Jacobi)
    errs.append(mismatch(x, want_off, "multigrid K=1, matrix without positions"))
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)


def test_bench_mesh_momentum_bicgstab_50_iterations_bit_exact(bench_mesh):
    """The benchmark's momentum solve: Jacobi-preconditioned BiCGSTAB, K = 3 in lockstep, the reference's 50 unguarded iterations
    on the fine 128^3 matrix (8192 tiles: nv = 3552, three tiles per virtual block)."""
    s = bench_mesh
    n, B = s["n"], s["B"]
    Ap, pinv, has = fm.jacobi_scale(s["A"])
    describe(Ap, "128^3 momentum BiCGSTAB:")
    rng = np.random.default_rng(7)
    X0 = 1e-3 * rng.standard_normal((3, n))
    snaps = {5: None, 50: None}
    fm.bicgstab(Ap, fm.jacobi_scale_rhs(pinv, has, B), X0, 50, snapshots=snaps)
    errs = []
    for it, want in snaps.items():
        xs = [q.copy() for q in X0]
        la.iterative_solve3(s["g"], list(B), xs, it, SolutionMethod.BiCGSTAB, 0.5, 1e-3, PreconditionMethod.Jacobi)
        errs.append(mismatch(np.stack(xs), want, f"K=3 {it} iterations"))
    errs = [e for e in errs if e]
    assert not errs, "\n".join(errs)
