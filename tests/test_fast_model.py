"""The NumPy model of the fast-mode arithmetic (tests/fast_model.py) is the right arithmetic, not just a copy of the kernels:

* its trees and virtual-block reductions stay within the rigorous error bound of their own summation order against exact sums
  (math.fsum) on adversarial data, and that bound is tight enough that a dropped or doubled virtual block breaks it;
* its SpMV classes, BiCGSTAB, Jacobi and Multigrid agree with the oracle (the CPU restatement of the reference) to the
  tolerances the GPU parity tests use;
* its Morton permutation matches a key computation done bit by bit;
* the constants it restates are the ones in the CUDA sources.

No GPU code runs here."""
import math
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

import fast_model as fm
from conftest import rel_l2
from orc_b200 import synthetic as syn

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "orc_b200", "csrc")
U = 2.0 ** -53
RHO, MU = 1000.0, 1e-3


def random_spd_like(n, density, seed, sym=True):
    """Same construction as test_gpu_linalg.random_spd_like: negative off-diagonals, dominant diagonal."""
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


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constexpr(text, name):
    m = re.search(r"constexpr\s+(?:int|int64_t)\s+(?:[A-Za-z_]\w*\s*=\s*[^,;]+,\s*)*" + name + r"\s*=\s*(\d+)", text)
    assert m, f"constexpr {name} not found in the sources: tests/fast_model.py must follow the kernel change"
    return int(m.group(1))


def test_constants_match_the_sources():
    linalg, common = _source("linalg.cu"), _source("common.cuh")
    for text, name, model in ((linalg, "SPMV_BLOCK", fm.SPMV_BLOCK), (common, "kVirtualBlocks", fm.VIRTUAL_BLOCKS),
                              (common, "kMaxLocalVb", fm.MAX_LOCAL_VB), (common, "kWarpsPerBlock", fm.WARPS_PER_BLOCK),
                              (linalg, "kReorderMinRows", fm.REORDER_MIN_ROWS), (linalg, "RO_CAP", fm.RO_CAP)):
        assert _constexpr(text, name) == model, f"{name} changed in the CUDA sources: update tests/fast_model.py"
    # the lanes-per-row choice of launch_spmv_k
    m = re.search(r"if \(avg < ([\d.]+) \|\| c\.exact_order\) \{\s*launch_virtual<k_spmv<EPI, K>>.*?"
                  r"\} else if \(avg < ([\d.]+)\) \{\s*launch_virtual<k_spmv_vec<EPI, (\d+), UN, K>>.*?"
                  r"\} else \{\s*launch_virtual<k_spmv_vec<EPI, (\d+), UN, K>>", linalg, re.S)
    assert m, "launch_spmv_k's dispatch changed shape: update fast_model.lanes_per_row"
    assert (float(m.group(1)), float(m.group(2)), int(m.group(3)), int(m.group(4))) == \
        (fm.THREAD_PER_ROW_BELOW, fm.FOUR_LANES_BELOW, 4, 8), "SpMV class thresholds moved: update fast_model.lanes_per_row"
    # the shuffle offsets of the trees
    assert "for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);" in common
    assert "for (int o = G / 2; o > 0; o >>= 1) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], o, G);" in linalg


# ---- trees and reductions against exact sums ------------------------------------------------------------------------------
def _adversarial(n, kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "mixed":      # mixed signs over a 1e-150 .. 1e150 dynamic range
        return rng.standard_normal(n) * 10.0 ** rng.uniform(-150, 150, n)
    if kind == "cancel":     # pairs that cancel to rounding noise plus small terms
        a = rng.standard_normal(n) * 1e8
        a[1::2] = -a[0::2][: n // 2]
        return a + rng.standard_normal(n)
    return rng.standard_normal(n) ** 2 * 10.0 ** rng.uniform(-8, 8, n)   # all-positive sums of squares


@pytest.mark.parametrize("kind", ["mixed", "cancel", "square"])
@pytest.mark.parametrize("n", [0, 1, 2, 17, 31, 32])
def test_warp_tree_bound(n, kind):
    v = _adversarial(n, kind, seed=n)
    exact = math.fsum(v)
    got = fm.warp_tree(v) if n else fm.warp_tree(np.zeros(0))
    assert abs(got - exact) <= 5 * U * math.fsum(np.abs(v)) * (1 + 1e-10)
    if n:
        assert fm.warp_tree_max(v) == v.max()


def test_warp_tree_is_the_shuffle_order():
    """Offsets W/2, ..., 1: with 1 in lane 0 and two halves of an ulp elsewhere, the result is 1 when each half meets the 1 on
    its own (1 + u/2 rounds back to 1) and 1 + u when the halves meet each other first (lanes 1 and 1 + W/2)."""
    h = 2.0 ** -53
    for W, tree in ((32, fm.warp_tree), (4, lambda v: fm.segment_tree(v, 4)), (8, lambda v: fm.segment_tree(v, 8))):
        v = np.zeros(W)
        v[0], v[1], v[W // 2] = 1.0, h, h
        assert tree(v) == 1.0, W
        v = np.zeros(W)
        v[0], v[1], v[1 + W // 2] = 1.0, h, h
        assert tree(v) == 1.0 + 2 * h, W
        v = np.zeros(W)
        v[0], v[W - 1], v[W // 2 - 1] = 1.0, h, h        # the last two lanes meet at offset W/2 as well
        assert tree(v) == 1.0 + 2 * h, W


def _depth(n, G, nv):
    rpb = fm.SPMV_BLOCK // G
    chain = max(1, -(-(-(-n // rpb)) // nv))
    return chain + 10 + max(1, -(-nv // fm.SPMV_BLOCK)) + 10


# lengths at the tree edges and row counts that put nv at 1, 37, 3552 with 1, 2 and >= 8 tiles per virtual block
REDUCE_SIZES = [0, 1, 31, 32, 33, 255, 257, 37 * 256, 3552 * 256, 2 * 3552 * 256 - 5, 9 * 3552 * 256 + 3]


@pytest.mark.parametrize("kind", ["mixed", "square"])
@pytest.mark.parametrize("n", REDUCE_SIZES)
def test_virtual_block_sum_bound(n, kind):
    c = _adversarial(n, kind, seed=n + 1)
    for G in (1, 4, 8):
        nv = fm.nv_for(-(-n // (fm.SPMV_BLOCK // G)))
        got = fm.vb_sum(c[None], G, nv)[0]
        exact = math.fsum(c)
        h = _depth(n, G, nv)
        mag = math.fsum(np.abs(c))
        assert abs(got - exact) <= h * U / (1 - h * U) * mag, (n, G, nv, got, exact)
        if n:
            assert fm.vb_max(np.abs(c)[None], G, nv)[0] == np.abs(c).max()


def test_a_dropped_or_doubled_virtual_block_breaks_the_bound():
    """For positive terms the bound is tight: losing or repeating one of 3552 virtual-block partials moves the total by ~1/3552,
    orders of magnitude beyond (chain + depth) u."""
    n = 2 * 3552 * 256 - 5
    c = _adversarial(n, "square", seed=3)
    nv = fm.nv_for(-(-n // fm.SPMV_BLOCK))
    parts = fm.block_tree(fm._thread_chains(c[None], 1, nv))
    exact, mag = math.fsum(c), math.fsum(c)
    h = _depth(n, 1, nv)
    assert abs(fm.sum_partials(parts)[0] - exact) <= h * U * mag
    k = int(np.argmax(parts[0]))
    for bad in (np.delete(parts, k, axis=1), np.concatenate([parts, parts[:, k:k + 1]], axis=1)):
        assert abs(fm.sum_partials(bad)[0] - exact) > 100 * h * U * mag


# ---- SpMV classes -------------------------------------------------------------------------------------------------------
def lengths_with_average(n, avg, seed, long_row=70, empty_row=True):
    """n row lengths (>= 1 except row 0) with mean exactly `avg`: random +- pairs around it, row 0 empty and row 2 longer than
    UN * G (= 32 for G = 8), both compensated elsewhere."""
    rng = np.random.default_rng(seed)
    lengths = np.full(n, avg, np.int64)
    d = rng.integers(-(avg - 1), avg, n // 2)
    lengths[0:2 * (n // 2):2] += d
    lengths[1:2 * (n // 2):2] -= d
    if empty_row:
        lengths[1] += lengths[0]
        lengths[0] = 0
    extra = max(0, long_row - lengths[2])
    lengths[2] += extra
    while extra > 0:                             # one entry less on the longest other rows, as often as needed
        take = np.argsort(-lengths[3:], kind="stable")[:extra] + 3
        take = take[lengths[take] > 1]
        assert take.size, "rows too short to make up for the long row"
        lengths[take] -= 1
        extra -= take.size
    assert lengths.sum() == avg * n and lengths.min() >= (0 if empty_row else 1)
    return lengths


def rows_with_lengths(lengths, ncols, seed):
    """Random matrix with the given row lengths (0 allowed), sorted unique columns, mixed-sign values."""
    rng = np.random.default_rng(seed)
    lengths = np.asarray(lengths, np.int64)
    rp = np.zeros(lengths.size + 1, np.int64)
    rp[1:] = np.cumsum(lengths)
    col = np.concatenate([np.sort(rng.choice(ncols, size=l, replace=False)) for l in lengths]) if lengths.sum() else np.zeros(0, np.int64)
    val = rng.standard_normal(int(rp[-1])) * 10.0 ** rng.uniform(-3, 3, int(rp[-1]))
    return sp.csr_matrix((val, col, rp), shape=(lengths.size, ncols))


@pytest.mark.parametrize("avg,G", [(7, 1), (10, 4), (17, 4), (32, 8), (107, 8)])
def test_spmv_classes_against_exact_row_sums(oracle, avg, G):
    """The model's SpMV class follows nnz / nrows; every row stays within (ceil(len / G) + log2 G) u of its exact sum, and the
    thread-per-row class is the oracle's ascending-k sum bit for bit. Includes empty rows and rows longer than UN * G."""
    n = 600
    a = rows_with_lengths(lengths_with_average(n, avg, seed=avg), 900, seed=avg)
    lengths = np.diff(a.indptr)
    A = fm.Mat.from_scipy(a)
    assert fm.lanes_per_row(A) == G
    x = np.random.default_rng(1).standard_normal(900)
    y = fm.spmv(A, x)[0]
    o = oracle.Csr.from_arrays(n, 900, a.indptr, a.indices, a.data)
    if G == 1:
        assert np.array_equal(y, o.spmv(x))
    depth = -(-lengths // G) + int(math.log2(G))
    for i in range(n):
        terms = a.data[a.indptr[i]:a.indptr[i + 1]] * x[a.indices[a.indptr[i]:a.indptr[i + 1]]]
        assert abs(y[i] - math.fsum(terms)) <= depth[i] * U * math.fsum(np.abs(terms)) * (1 + 1e-12), i
    assert y[0] == 0.0


# ---- solvers against the oracle ------------------------------------------------------------------------------------------
_mom = {}


def momentum_matrix(oracle, n=16):
    """The x-momentum matrix of an n^3 hex channel, assembled by the oracle on smooth fields."""
    if n not in _mom:
        from cases import smooth_fields
        om = oracle.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(n, n, n)))
        syn.channel_bcs(om)
        u, v, w, p = smooth_fields(om.export())
        di, *_ = om.build_momentum_diffusion(MU)
        a = [om.init_momentum_matrix() for _ in range(3)]
        om.build_momentum_advection(*a, di, u, v, w, p, oracle.Settings(), RHO)
        _mom[n] = (a[0], om.export()["cell_centroid"])
    return _mom[n]


def _cases(oracle):
    yield "spd3000", oracle.Csr.from_arrays(3000, 3000, *_arr(random_spd_like(3000, 0.003, seed=11)))
    yield "spd2048_long", oracle.Csr.from_arrays(2048, 2048, *_arr(random_spd_like(2048, 0.03, seed=61)))
    yield "hex16", momentum_matrix(oracle)[0]


def _arr(a):
    return a.indptr, a.indices, a.data


def _mat(o):
    rp, co, va = o.arrays()
    return fm.Mat(rp, co, va, o.dims[1])


@pytest.mark.parametrize("case", ["spd3000", "spd2048_long", "hex16"])
def test_model_solvers_agree_with_the_oracle(oracle, case):
    """BiCGSTAB (both preconditioners), Jacobi and Multigrid at 5 iterations: the model differs from the oracle only in the
    order of its dot products, so it must meet the GPU parity tolerances: 1e-10 per preconditioned BiCGSTAB / Jacobi solve
    (test_gpu_scale), 1e-9 without the preconditioner (test_gpu_linalg), 1e-8 for Multigrid."""
    o = dict(_cases(oracle))[case]
    A = _mat(o)
    n = A.nrows
    rng = np.random.default_rng(5)
    b, x0 = rng.standard_normal(n), rng.standard_normal(n)
    for pc in (0, 1):
        x = fm.iterative_solve(A, b, x0, 5, fm.BICGSTAB, preconditioner=bool(pc))[0]
        xo = oracle.iterative_solve(o, b, x0, 5, oracle.BICGSTAB, 0.5, 1e-3, pc)
        assert rel_l2(x, xo) <= (1e-10 if pc else 1e-9), (case, "bicgstab", pc, rel_l2(x, xo))
    for iters, thr in ((7, 1e-30), (200, 1e-3)):
        x = fm.iterative_solve(A, b, np.zeros(n), iters, fm.JACOBI, 0.5, thr)[0]
        xo = oracle.iterative_solve(o, b, np.zeros(n), iters, oracle.JACOBI, 0.5, thr, 1)
        assert rel_l2(x, xo) <= 1e-10, (case, "jacobi", iters, rel_l2(x, xo))
    xo, olev = oracle.multigrid_trace(o, b, np.zeros(n), iterations=5)
    levels = [(_mat(r), _mat(a)) for r, a in olev]
    x = fm.iterative_solve(A, b, np.zeros(n), 5, fm.MULTIGRID, levels=levels)[0]
    assert rel_l2(x, xo) <= 1e-8, (case, "multigrid", rel_l2(x, xo))


def test_model_multigrid_with_the_locality_ordering_agrees_with_the_oracle(oracle):
    """32^3 momentum matrix: coarse level 1 has 16384 rows, so the model stores it (and only it) along the Morton curve. The
    ordering changes summation orders only: still 1e-8 of the oracle, and different from the unordered model."""
    o, cc = momentum_matrix(oracle, 32)
    A = _mat(o)
    n = A.nrows
    b = np.random.default_rng(11).standard_normal(n)
    xo, olev = oracle.multigrid_trace(o, b, np.zeros(n), iterations=5)
    levels = [(_mat(r), _mat(a)) for r, a in olev]
    pos = fm.Positions(cc)
    assert [fm.reorder_applies(a, l + 1, pos) for l, (_, a) in enumerate(levels)] == [True, False, False]
    x_on = fm.iterative_solve(A, b, np.zeros(n), 5, fm.MULTIGRID, levels=levels, pos=pos)[0]
    x_off = fm.iterative_solve(A, b, np.zeros(n), 5, fm.MULTIGRID, levels=levels)[0]
    assert rel_l2(x_on, xo) <= 1e-8 and rel_l2(x_off, xo) <= 1e-8
    assert 0 < rel_l2(x_on, x_off) <= 1e-8


# ---- locality ordering ---------------------------------------------------------------------------------------------------
def test_morton_permutation_against_brute_force_keys():
    arrays = syn.hex_box(10, 6, 5, jitter=1e-5)
    from oracle import pyoracle
    cc = pyoracle.Mesh.from_arrays(*syn.mesh_args(arrays)).export()["cell_centroid"]
    pos = fm.Positions(cc)
    for shift in (0, 1, 2):
        n = (cc.shape[0] >> shift) + 3          # rows past the end clamp to the last cell
        keys = []
        for i in range(n):
            f = min(i << shift, cc.shape[0] - 1)
            key = 0
            for a in range(3):
                q = (cc[f, a] - pos.lo[a]) * pos.inv[a]
                v = 1023 if q >= 1023.0 else (int(q) if q > 0.0 else 0)
                for bit in range(10):
                    key |= ((v >> bit) & 1) << (3 * bit + a)
            keys.append(key)
        assert np.array_equal(fm.morton_keys(n, pos, shift), np.array(keys, np.uint32))
        assert np.array_equal(fm.morton_perm(n, pos, shift), np.array(sorted(range(n), key=lambda i: keys[i])))


def test_reordered_system_is_the_permuted_scaled_matrix():
    a = random_spd_like(500, 0.02, seed=3).tolil()
    a[7, 7] = 0.0                                # a row without a stored diagonal: empty in the stored system
    a = a.tocsr()
    a.eliminate_zeros()
    a.sort_indices()
    A = fm.Mat.from_scipy(a)
    perm = np.random.default_rng(0).permutation(500)
    S, pinv, has = fm.reordered_system(A, perm)
    assert S.nnz == A.nnz and S.rowptr[-1] == A.nnz - a.indptr[8] + a.indptr[7]
    d = np.where(has, pinv, 0.0)
    ref = (sp.diags(d) @ a).tocsr()[perm][:, perm].tocsr()
    ref.sort_indices()
    assert np.array_equal(S.rowptr, ref.indptr) and np.array_equal(S.col, ref.indices)
    Sd, _, _ = fm.jacobi_scale(A)
    assert np.array_equal(np.sort(S.val), np.sort(Sd.val))
    assert np.allclose(S.val, ref.data, rtol=1e-15, atol=0)
