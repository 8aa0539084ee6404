"""NumPy restatement of the fast-mode (ORC_REDUCE_FAST) arithmetic of orc_b200/csrc/linalg.cu and common.cuh, operation for
operation, so that a GPU solve can be compared with it bit for bit (np.array_equal) at any size and any iteration count.

The fast mode is deterministic by construction: its summation order depends on the matrix and its size only, never on the
grid, the SM count or the number of systems per launch (common.cuh, Ctx::kVirtualBlocks). Every kernel is built with
-fmad=false and uses IEEE `/` and `sqrt`, so each product, quotient and sum below rounds exactly like its device twin.

Rules of this file: no np.sum / np.add.reduce / `@` / np.dot anywhere (NumPy sums pairwise and BLAS reorders). Every sum is an
explicit sequential loop over entry positions or partials, vectorised across rows / virtual blocks / systems, or an explicit
shuffle tree. Vectors of K systems are arrays of shape (K, n); system k is the K = 1 arithmetic on row k (linalg.cu, Cell<K>).

An intentional change of a kernel's summation order must update this model in the same change (DESIGN.md §5).
"""
import os

import numpy as np

# ---- constants of the kernels (tests/test_fast_model.py reads them back from the sources) ----------------------------------
SPMV_BLOCK = 256          # linalg.cu: constexpr int SPMV_BLOCK
VIRTUAL_BLOCKS = 3552     # common.cuh: Ctx::kVirtualBlocks
MAX_LOCAL_VB = 24         # common.cuh: kMaxLocalVb (virtual blocks per real block; no effect on the order)
WARPS_PER_BLOCK = 8       # common.cuh: kWarpsPerBlock
THREAD_PER_ROW_BELOW = 10.0   # linalg.cu launch_spmv_k: avg < 10 -> k_spmv
FOUR_LANES_BELOW = 32.0       # avg < 32 -> k_spmv_vec<G = 4>, else G = 8
REORDER_MIN_ROWS = 16384  # linalg.cu: kReorderMinRows
RO_CAP = 512              # linalg.cu: RO_CAP (longest row the locality ordering takes)


# =============================================================================================================================
# shuffle trees and virtual-block reductions (common.cuh:257-385)
# =============================================================================================================================
def _tree(v, width, op):
    """Lane 0 of the __shfl_down_sync tree over the last axis (`width` lanes, missing lanes 0 / -inf padded by the caller):
    offsets width/2, ..., 1; lane l takes op(v_l, v_{l+o}). Lane 0 only depends on lanes < 2o at each step."""
    o = width // 2
    while o > 0:
        v = op(v[..., :o], v[..., o:2 * o])
        o //= 2
    return v[..., 0]


def _pad_last(v, width, fill):
    v = np.asarray(v, dtype=np.float64)
    if v.shape[-1] == width:
        return v
    assert v.shape[-1] < width
    out = np.full(v.shape[:-1] + (width,), fill, dtype=np.float64)
    out[..., :v.shape[-1]] = v
    return out


def warp_tree(v):
    """warp_sum (common.cuh:257-261) over the last axis: up to 32 lanes, missing lanes 0.0."""
    return _tree(_pad_last(v, 32, 0.0), 32, np.add)


def warp_tree_max(v):
    """warp_max (common.cuh:262-266): the fmax twin; missing lanes -inf."""
    return _tree(_pad_last(v, 32, -np.inf), 32, np.fmax)


def segment_tree(v, G):
    """The in-row tree of k_spmv_vec (linalg.cu:507-511): __shfl_down_sync(..., o, G) for o = G/2 ... 1 over the G lanes of a
    row (last axis)."""
    assert v.shape[-1] == G
    return _tree(v, G, np.add)


def block_tree(v):
    """block_sum / block_sum_n / vb_park + vb_publish over a 256-thread block (common.cuh:268-300, 347-366): a warp tree per
    warp, then the 8 warp results in lanes 0..7 of one more 32-lane tree (lanes 8..31 zero). v: (..., 256)."""
    w = warp_tree(v.reshape(v.shape[:-1] + (WARPS_PER_BLOCK, 32)))
    return warp_tree(w)


def block_tree_max(v):
    """block_max (common.cuh:301-313)."""
    w = warp_tree_max(v.reshape(v.shape[:-1] + (WARPS_PER_BLOCK, 32)))
    return warp_tree_max(w)


def _chain(arr, op=np.add, start=0.0):
    """Sequential per-thread chain over axis -2 of arr (..., M, T): acc = start; acc = op(acc, arr[m]) in ascending m."""
    acc = np.full(arr.shape[:-2] + arr.shape[-1:], start)
    for m in range(arr.shape[-2]):
        acc = op(acc, arr[..., m, :])
    return acc


def sum_partials(p):
    """sum_partials / sum_partials_n (common.cuh:329-333, 369-385): thread t adds partials t, t+256, ... in ascending order
    (the batches of eight loads do not change it), then one block tree. p: (..., nv)."""
    nv = p.shape[-1]
    m = max(1, -(-nv // SPMV_BLOCK))
    q = _pad_last(p, m * SPMV_BLOCK, 0.0).reshape(p.shape[:-1] + (m, SPMV_BLOCK))
    return block_tree(_chain(q))


def max_partials(p):
    """max_partials (common.cuh:334-338)."""
    nv = p.shape[-1]
    m = max(1, -(-nv // SPMV_BLOCK))
    q = _pad_last(p, m * SPMV_BLOCK, -np.inf).reshape(p.shape[:-1] + (m, SPMV_BLOCK))
    return block_tree_max(_chain(q, np.fmax, -np.inf))


def _thread_chains(c, G, nv, op=np.add, start=0.0):
    """Per-thread serial chains of a fused reduction: c (..., n) holds one contribution per row, (..., nv, 256) comes back.
    Rows form groups of RPB = 256 / G; thread t of virtual block vb visits the rows grp * RPB + t / G for grp = vb, vb + nv, ...
    and only lanes with t % G == 0 add (k_spmv: G = 1, i = vb * 256 + t + m * nv * 256, linalg.cu:437; k_spmv_vec: linalg.cu:480-512;
    k_bicg_xr: G = 1, linalg.cu:613). Padding rows contribute `start`, which leaves every chain unchanged."""
    rpb = SPMV_BLOCK // G
    n = c.shape[-1]
    ngroups = -(-n // rpb)
    m = max(1, -(-ngroups // nv))
    q = _pad_last(c, m * nv * rpb, start).reshape(c.shape[:-1] + (m, nv, rpb))
    acc = np.full(c.shape[:-1] + (nv, rpb), start)
    for j in range(m):
        acc = op(acc, q[..., j, :, :])
    if G == 1:
        return acc
    out = np.full(c.shape[:-1] + (nv, SPMV_BLOCK), start)
    out[..., ::G] = acc
    return out


def vb_sum(c, G, nv):
    """Total of a fused sum: thread chains -> block tree per virtual block (the published partial) -> sum_partials."""
    return sum_partials(block_tree(_thread_chains(c, G, nv)))


def vb_max(c, G, nv, start=0.0):
    """Total of the fused maximum of EP_JACOBI_RES (acc1 starts at 0, linalg.cu:326): block_max, then max_partials."""
    return max_partials(block_tree_max(_thread_chains(c, G, nv, np.fmax, start)))


def nv_for(tiles):
    """Virtual blocks of a launch (linalg.cu:534, grid_for(n, 256, kVirtualBlocks) at :778): clamp(tiles, 1, 3552)."""
    return int(max(1, min(tiles, VIRTUAL_BLOCKS)))


# =============================================================================================================================
# matrices and SpMV (linalg.cu:421-573)
# =============================================================================================================================
class Mat:
    """CSR with ascending columns per row. `nnz` is what the kernels read as A.nnz for the lanes-per-row choice; it can exceed
    the stored entries (linalg.cu:2176: the locality-ordered copy keeps the uncompacted count)."""

    def __init__(self, rowptr, col, val, ncols, nnz=None):
        self.rowptr = np.asarray(rowptr, dtype=np.int64)
        self.col = np.asarray(col, dtype=np.int32)
        self.val = np.asarray(val, dtype=np.float64)
        self.nrows = self.rowptr.size - 1
        self.ncols = int(ncols)
        self.nnz = int(self.rowptr[-1]) if nnz is None else int(nnz)
        self._plan = None
        self._diag = None
        self.cache = {}

    @classmethod
    def from_scipy(cls, a):
        a = a.tocsr()
        a.sort_indices()
        return cls(a.indptr, a.indices, a.data, a.shape[1])

    @classmethod
    def from_handle(cls, h):
        """From an orc_b200 CsrMatrix handle (downloaded)."""
        rp, co, va = h.arrays()
        return cls(rp, co, va, h.dims[1])

    @property
    def lengths(self):
        return np.diff(self.rowptr)

    @property
    def max_row(self):
        return int(self.lengths.max()) if self.nrows else 0

    def diag_index(self):
        """Index of the stored (i, i) entry or -1 (k_find_diag)."""
        if self._diag is None:
            n = self.nrows
            rows = np.repeat(np.arange(n), self.lengths)
            hit = np.nonzero(self.col == rows[:self.col.size] if self.col.size else np.zeros(0, bool))[0]
            d = np.full(n, -1, dtype=np.int64)
            d[rows[hit]] = hit
            self._diag = d
        return self._diag

    def plan(self):
        """(order, slots): `order` lists the rows by descending length (stable), and slot s holds entry rowptr[i] + s of every row
        longer than s, i.e. of the first k_s rows of `order`: (k_s, values, columns) in that order. Working in `order` turns every
        slot's rows into a prefix (contiguous slices instead of a scatter); each row still adds its entries in ascending position."""
        if self._plan is None:
            lens = self.lengths
            order = np.argsort(-lens, kind="stable").astype(np.int64)
            counts = np.bincount(lens, minlength=1) if self.nrows else np.zeros(1, np.int64)
            longer = self.nrows - np.cumsum(counts)   # rows with more than s entries, s = 0, 1, ...
            start = self.rowptr[:-1][order]
            slots = []
            for s in range(self.max_row):
                k = int(longer[s])
                idx = start[:k] + s
                slots.append((k, self.val[idx], self.col[idx]))
            self._plan = (order, slots)
        return self._plan


def lanes_per_row(A, exact_order=False):
    """launch_spmv_k (linalg.cu:553-564): avg = nnz / nrows; < 10 (or reference order): one thread per row; < 32: G = 4; else 8."""
    avg = A.nnz / A.nrows if A.nrows > 0 else 0.0
    if avg < THREAD_PER_ROW_BELOW or exact_order:
        return 1
    return 4 if avg < FOUR_LANES_BELOW else 8


def spmv_launch(A, exact_order=False):
    """(G, nv, tiles per virtual block) of an SpMV launch on A."""
    G = lanes_per_row(A, exact_order)
    tiles = -(-A.nrows // (SPMV_BLOCK // G))
    nv = nv_for(tiles)
    return G, nv, -(-tiles // nv)


def spmv(A, X, exact_order=False):
    """Row sums of A X in the kernel's order; X: (K, ncols) -> (K, nrows).
    G = 1 (k_spmv, linalg.cu:437-448): acc = 0; acc += a_ik x_k in ascending k.
    G = 4 / 8 (k_spmv_vec, :485-511): lane gl adds entries lo+gl, lo+gl+G, ... in ascending order (UN only batches the loads),
    then the width-G shuffle tree."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    K = X.shape[0]
    G = lanes_per_row(A, exact_order)
    order, slots = A.plan()
    # K = 1: plain vectors; K > 1: (ncols, K), one gather fetches the K values of a column
    XT = X[0] if K == 1 else np.ascontiguousarray(X.T)
    shape = (A.nrows,) if K == 1 else (A.nrows, K)
    lanes = np.zeros((G,) + shape)                          # rows in `order`

    def rows(lo, hi):   # every slot over the rows [lo, hi) of `order`: no row is shared, so the chunks are independent
        tmp = np.empty((hi - lo,) + shape[1:])
        for s, (k, v, c) in enumerate(slots):
            e = min(hi, k)
            if e <= lo:
                break
            prod = tmp[:e - lo]
            np.take(XT, c[lo:e], axis=0, out=prod, mode="clip")   # the columns are in range: "clip" only skips a buffer
            np.multiply(v[lo:e] if K == 1 else v[lo:e, None], prod, out=prod)
            acc = lanes[s % G, lo:e]
            np.add(acc, prod, out=acc)

    chunks = _row_chunks(A.nrows, len(A.col))
    if len(chunks) == 1:
        rows(*chunks[0])
    else:   # NumPy releases the GIL inside take / multiply / add
        list(_pool().map(lambda c: rows(*c), chunks))
    out = np.empty(shape)
    out[order] = lanes[0] if G == 1 else segment_tree(np.moveaxis(lanes, 0, -1), G)
    return out[None] if K == 1 else np.ascontiguousarray(out.T)


_POOL = {}


def _pool():
    """The SpMV threads of this process (a forked worker starts its own)."""
    pid = os.getpid()
    if pid not in _POOL:
        from concurrent.futures import ThreadPoolExecutor
        _POOL.clear()
        _POOL[pid] = ThreadPoolExecutor(max_workers=os.cpu_count() or 1)
    return _POOL[pid]


def _row_chunks(n, entries):
    """Row ranges of `order` for the threads of one SpMV: one range for small matrices, else one per core."""
    parts = 1 if entries < 1 << 20 else (os.cpu_count() or 1)
    edges = np.linspace(0, n, parts + 1).astype(np.int64)
    return [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a] or [(0, 0)]


def fused_sum(A, c):
    """Total of per-row contributions c (K, nrows) fused into an SpMV on A (spmv_block_partials + spmv_finalize)."""
    G, nv, _ = spmv_launch(A)
    return vb_sum(c, G, nv)


# =============================================================================================================================
# Jacobi scaling (linalg.cu:829-910)
# =============================================================================================================================
def jacobi_scale(A):
    """A' = P^-1 A: a'_ij = 0 + (1 * (1 / a_ii)) * a_ij (k_jacobi_scale, :844, :859). Rows without a stored diagonal become empty and
    the matrix is compacted (:892-909): the kernel choice then reads the compacted nnz. Returns (A', pinv, has_diag)."""
    if "scaled" not in A.cache:
        d = A.diag_index()
        has = d >= 0
        pinv = np.zeros(A.nrows)
        pinv[has] = 1.0 / A.val[d[has]]
        rows = np.repeat(np.arange(A.nrows), A.lengths)
        sval = 0.0 + (1.0 * pinv[rows]) * A.val
        if has.all():
            S = Mat(A.rowptr, A.col, sval, A.ncols)
        else:
            keep = has[rows]
            rp = np.zeros(A.nrows + 1, np.int64)
            rp[1:] = np.cumsum(np.where(has, A.lengths, 0))
            S = Mat(rp, A.col[keep], sval[keep], A.ncols)
        A.cache["scaled"] = (S, pinv, has)
    return A.cache["scaled"]


def jacobi_scale_rhs(pinv, has, B):
    """b'_i = 0 + pinv_i * b_i, 0 where the diagonal is missing (:850)."""
    return np.where(has, 0.0 + pinv * B, 0.0)


# =============================================================================================================================
# BiCGSTAB (linalg.cu:586-663, 773-809) and Jacobi (:912-953)
# =============================================================================================================================
def bicgstab(A, B, X, iterations, snapshots=None):
    """bicgstab_k: unguarded, r_hat_0 = 1, exactly `iterations` iterations. B, X: (K, n); returns the new X. The solve is the same
    for every iteration count up to the last one, so `snapshots` ({iteration count: None}) collects the X of shorter solves."""
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    X = np.atleast_2d(np.array(X, dtype=np.float64))
    n = A.nrows
    if n == 0:
        return X
    nvx = nv_for(-(-n // 256))                                  # k_bicg_xr: grid_for(n, 256, kVirtualBlocks)
    r = B - spmv(A, X)                                          # EP_RESID_INIT: r = b - A x; p = r; rho = sum(r)
    p = r.copy()
    rho = fused_sum(A, r)
    for it in range(iterations):
        nu = spmv(A, p)                                         # EP_SUM_ALPHA: alpha = rho / sum(nu)
        alpha = rho / fused_sum(A, nu)
        s = r - alpha[:, None] * nu                             # k_bicg_s
        t = spmv(A, s)                                          # EP_DOTS_OMEGA: omega = (t.s) / (t.t)
        omega = fused_sum(A, t * s) / fused_sum(A, t * t)
        h = X + alpha[:, None] * p                              # k_bicg_xr
        X = h + omega[:, None] * s
        r = s - omega[:, None] * t
        rho_prev = rho
        rho = vb_sum(r, 1, nvx)
        beta = rho / rho_prev * alpha / omega
        p = r + beta[:, None] * (p - omega[:, None] * nu)       # k_bicg_p
        if snapshots is not None and it + 1 in snapshots:
            snapshots[it + 1] = X.copy()
    return X


def jacobi(A, b, x, iterations, relaxation, threshold):
    """jacobi (linalg.cu:928-953), one system: a0_ij = a_ij / a_ii off the diagonal, 0 on it; b0 = b / a_ii (k_jacobi_prepare);
    per iteration xn = w (b0 - A0 x) + x (1 - w) (EP_JACOBI on A0), then EP_JACOBI_RES on A: r = sqrt(sum (b - A xn)^2), x = xn, and
    the convergence latch: `initial` is 0 at iteration 0 (so r / 0 never passes), it is set at iteration 1, and from iteration 2
    on r / initial < threshold stops the loop after x = xn has been stored. Returns (x, iterations run, last r)."""
    b = np.asarray(b, dtype=np.float64)[None]
    x = np.array(x, dtype=np.float64)[None]
    n = A.nrows
    d = A.diag_index()
    if (d < 0).any():
        raise ValueError("Tried to access CsrMatrix element that hasn't been stored yet.")
    aii = A.val[d]
    rows = np.repeat(np.arange(n), A.lengths)
    val0 = np.where(A.col == rows, 0.0, A.val / aii[rows])
    A0 = Mat(A.rowptr, A.col, val0, A.ncols)
    b0 = b / aii
    w = relaxation
    one_minus_w = 1.0 - relaxation
    G, nv, _ = spmv_launch(A)
    initial = 0.0
    r = np.nan
    it = 0
    for it in range(iterations):
        xn = w * (b0 - spmv(A0, x)) + x * one_minus_w
        res = b - spmv(A, xn)
        r = float(np.sqrt(vb_sum(res * res, G, nv))[0])
        x = xn
        if it == 1:
            initial = r
        elif it > 1 and np.float64(r) / initial < threshold:
            return x[0], it + 1, r
    return x[0], iterations if iterations else 0, r


# =============================================================================================================================
# locality ordering of the coarse levels (linalg.cu:2057-2196)
# =============================================================================================================================
def morton_spread10(v):
    v = np.asarray(v, dtype=np.uint32) & np.uint32(0x3FF)
    v = (v | (v << np.uint32(16))) & np.uint32(0x030000FF)
    v = (v | (v << np.uint32(8))) & np.uint32(0x0300F00F)
    v = (v | (v << np.uint32(4))) & np.uint32(0x030C30C3)
    v = (v | (v << np.uint32(2))) & np.uint32(0x09249249)
    return v


class Positions:
    """PosHint of a mesh matrix (assembly.cu:215-220): cell centroids, lo = min, inv = 1024 / (max - min) (0 for a flat axis)."""

    def __init__(self, centroids):
        c = np.asarray(centroids, dtype=np.float64)
        self.xyz = [np.ascontiguousarray(c[:, a]) for a in range(3)]
        self.n = c.shape[0]
        self.lo = [float(p.min()) for p in self.xyz]
        self.inv = []
        for a in range(3):
            ext = float(self.xyz[a].max()) - self.lo[a]
            self.inv.append(1024.0 / ext if (ext > 0.0 and np.isfinite(ext)) else 0.0)


def morton_keys(n, pos, shift):
    """k_morton_keys (:2072-2085): row I sits at f = min(I << shift, n_fine - 1); q = (c - lo) * inv, truncated into [0, 1023]
    (NaN -> 0); key = interleave(qx, qy, qz) with x in bit 0."""
    f = np.minimum(np.arange(n, dtype=np.int64) << shift, pos.n - 1)
    key = np.zeros(n, dtype=np.uint32)
    for a in range(3):
        q = (pos.xyz[a][f] - pos.lo[a]) * pos.inv[a]
        with np.errstate(invalid="ignore"):
            v = np.where(q >= 1023.0, 1023.0, np.where(q > 0.0, np.trunc(q), 0.0)).astype(np.uint32)
        key |= morton_spread10(v) << np.uint32(a)
    return key


def morton_perm(n, pos, shift):
    """Stable radix sort of the keys (:2169-2171): row r of the stored system is row perm[r] of the level."""
    return np.argsort(morton_keys(n, pos, shift), kind="stable")


def reorder_applies(A, level, pos, min_level=1):
    """reorder_applies (:2147-2151) for a BiCGSTAB smoother with the Jacobi preconditioner in the fast mode."""
    return (min_level > 0 and level >= min_level and pos is not None and A.nrows == A.ncols and A.nrows >= REORDER_MIN_ROWS
            and 0 < A.max_row <= RO_CAP)


def reordered_system(A, perm):
    """P (D^-1 A) P^T with columns ascending (k_scale_permute_rows, :2094-2132), keeping A.nnz as the declared nnz (:2176).
    Returns (stored matrix, pinv, has_diag) of the level's own numbering."""
    S, pinv, has = jacobi_scale(A)
    n = A.nrows
    iperm = np.empty(n, np.int64)
    iperm[perm] = np.arange(n)
    lens = S.lengths[perm]          # S is A's scaled copy, rows without a diagonal already empty
    rp = np.zeros(n + 1, np.int64)
    rp[1:] = np.cumsum(lens)
    idx = np.repeat(S.rowptr[perm], lens) + (np.arange(int(rp[-1])) - np.repeat(rp[:-1], lens))
    newcol = iperm[S.col[idx]]
    order = np.lexsort((newcol, np.repeat(np.arange(n), lens)))
    return Mat(rp, newcol[order], S.val[idx][order], n, nnz=A.nnz), pinv, has


# =============================================================================================================================
# iterative_solve and Multigrid (linalg.cu:2200-2289)
# =============================================================================================================================
BICGSTAB, JACOBI, MULTIGRID = "bicgstab", "jacobi", "multigrid"
MG_DIVERGED, DIVERGED = "Multigrid diverged", "solution diverged"   # ORC_E_MG_DIVERGED, ORC_E_DIVERGED


class ModelDiverged(RuntimeError):
    """A divergence exit of the GPU path, taken by the model. str() is the GPU's message; `code` names its status
    (orc_b200._lib.E_MG_DIVERGED or E_DIVERGED)."""

    @property
    def code(self):
        from orc_b200 import _lib
        return _lib.E_MG_DIVERGED if str(self) == MG_DIVERGED else _lib.E_DIVERGED


def check_field_sums(*fields):
    """The `u_avg != u_avg` exit of steady_iterate (capi.cu, solver.rs:217-221). A sum is NaN in every order exactly when a term is
    NaN or the terms hold both infinities (finite terms that overflow are the one order-dependent case; the kernels' fields never
    come near DBL_MAX before they turn NaN)."""
    for f in fields:
        f = np.asarray(f)
        if np.isnan(f).any() or (np.isposinf(f).any() and np.isneginf(f).any()):
            raise ModelDiverged(DIVERGED)


def transpose(R):
    """R^T with ascending columns."""
    nnz = R.rowptr[-1]
    rows = np.repeat(np.arange(R.nrows), R.lengths)
    order = np.lexsort((rows, R.col[:nnz]))
    rp = np.zeros(R.ncols + 1, np.int64)
    rp[1:] = np.cumsum(np.bincount(R.col[:nnz], minlength=R.ncols))
    return Mat(rp, rows[order], R.val[:nnz][order], R.nrows)


def iterative_solve(A, B, X, iterations, method, relaxation=0.5, threshold=1e-3, preconditioner=True, levels=None, pos=None,
                    reorder_min_level=1, mg_smoother=BICGSTAB, mg_levels=3):
    """iterative_solve (:2255-2289) in the fast mode. B, X: (K, n) (Jacobi: K = 1). `levels`: [(R_l, A_l)] of the Multigrid
    hierarchy as the GPU built it (la.multigrid_trace; pinned bit-exactly against the oracle elsewhere). `pos`: Positions of
    the fine matrix's unknowns (mesh matrices), which switch the locality ordering on."""
    B = np.atleast_2d(np.asarray(B, dtype=np.float64))
    X = np.atleast_2d(np.array(X, dtype=np.float64))
    Ap, bp = A, B
    if preconditioner:
        Ap, pinv, has = jacobi_scale(A)
        bp = jacobi_scale_rhs(pinv, has, B)
    if method == BICGSTAB:
        return bicgstab(Ap, bp, X, iterations)
    if method == JACOBI:
        assert X.shape[0] == 1
        return jacobi(Ap, bp[0], X[0], iterations, relaxation, threshold)[0][None]
    assert method == MULTIGRID
    kw = dict(relaxation=relaxation, preconditioner=preconditioner)
    X = iterative_solve(Ap, bp, X, iterations, mg_smoother, threshold=threshold, **kw)     # preconditions AGAIN (Q7)
    r = bp - spmv(Ap, X)                                                                 # residual: EP_RESID
    corr = _multigrid_level(Ap, r, 1, levels, iterations, threshold, kw, pos, reorder_min_level, mg_smoother, mg_levels)
    return X + corr                                                                      # dev_axpy_inplace


def _multigrid_level(A, r, level, levels, iterations, threshold, kw, pos, min_level, smoother, mg_levels):
    """multigrid_solve (:2200-2245)."""
    R, Ac = levels[level - 1]
    if "RT" not in R.cache:
        R.cache["RT"] = transpose(R)
    RT = R.cache["RT"]
    rp = spmv(R, r)                                                                      # r' = R r
    ep = np.zeros_like(rp)
    ro = None
    if smoother == BICGSTAB and kw["preconditioner"] and reorder_applies(Ac, level, pos, min_level):
        key = ("ro", level)
        if key not in Ac.cache:
            perm = morton_perm(Ac.nrows, pos, level)
            Ac.cache[key] = (perm,) + reordered_system(Ac, perm)
        perm, S, pinv, has = Ac.cache[key]
        bs = jacobi_scale_rhs(pinv, has, rp)[:, perm]                                    # P D^-1 r'
        ro = (perm, S, bs)

    def smooth(e, thr):
        if ro is None:
            return iterative_solve(Ac, rp, e, iterations, smoother, threshold=thr, **kw)
        perm, S, bs = ro
        y = bicgstab(S, bs, e[:, perm], iterations)                                       # reordered_smooth
        out = np.empty_like(y)
        out[:, perm] = y
        return out

    ep = smooth(ep, threshold)
    # residual_norm_check (EP_RESID_NORM on the unscaled level matrix, :97-105): sqrt(sum r_i^2) is NaN exactly when some r_i is
    # NaN (squares are >= 0 or +inf), whatever the order of the sum; r_i itself comes from the kernel's row order
    if np.isnan(rp - spmv(Ac, ep)).any():
        raise ModelDiverged(MG_DIVERGED)
    if level < mg_levels and Ac.nrows > 16:
        corr = _multigrid_level(Ac, rp, level + 1, levels, iterations, threshold, kw, pos, min_level, smoother, mg_levels)
        ep = ep + corr
        ep = smooth(ep, threshold / 10.0)
    return spmv(RT, ep)                                                                  # out = R^T e'
