"""Whole SIMPLE iterations of the fast mode, composed from parts that are already pinned bit for bit: the oracle's assemblies and
correction (bit-exact with the GPU kernels, test_gpu_scale.py), the oracle's Multigrid hierarchies (bit-exact with the GPU's) and
fast_model's solves (bit-exact with every fast-mode solve, test_gpu_fast_model.py). Put together in the order of steady_iterate
(capi.cu; src/solver.rs:60-222; oracle solve_steady) they predict every bit of a fast-mode SIMPLE iteration on the GPU.

Nothing is restated here: every step is an oracle or fast_model call. The solve is a parameter, so that the same driver run with
the oracle's own solver can be checked against oracle.solve_steady."""
import math

import numpy as np

import fast_model as fm
from oracle import pyoracle as po

_METHOD = {po.BICGSTAB: fm.BICGSTAB, po.JACOBI: fm.JACOBI, po.MULTIGRID: fm.MULTIGRID}


def batchable(settings):
    """solve_batchable (linalg.cu) in the fast mode: BiCGSTAB, or Multigrid with the BiCGSTAB smoother."""
    return settings.solver_type == po.BICGSTAB or (settings.solver_type == po.MULTIGRID and settings.mg_smoother == po.BICGSTAB)


def values_identical(a, b):
    """csr_values_identical: the value arrays equal bit for bit."""
    va, vb = a.arrays()[2], b.arrays()[2]
    return va.shape == vb.shape and np.array_equal(va.view(np.int64), vb.view(np.int64))


def oracle_solve(settings):
    """solve(a, B, X, pos) with the oracle's iterative_solve, one system at a time (pos is ignored)."""
    def solve(a, B, X, pos=None):
        return np.stack([po.iterative_solve(a, b, x, settings.iterations, settings.solver_type, settings.relaxation, settings.threshold,
                                            settings.preconditioner, settings.gs_intended, settings.mg_smoother, settings.mg_levels)
                         for b, x in zip(B, X)])
    return solve


def model_solve(settings, levels_log=None):
    """solve(a, B, X, pos) with fast_model.iterative_solve: K = len(B) systems on one matrix. Multigrid rebuilds the hierarchy on every
    call, as the GPU does: oracle.multigrid_trace of the unscaled matrix (its levels are those of the Jacobi-scaled copy, which is what
    Multigrid coarsens). `levels_log` (a list) collects the (rows, nnz) of every hierarchy."""
    method = _METHOD[settings.solver_type]

    def solve(a, B, X, pos=None):
        A = fm.Mat.from_handle(a)
        levels = None
        if method == fm.MULTIGRID:
            _, lev = po.multigrid_trace(a, np.ones(A.nrows), np.zeros(A.nrows), iterations=1, relaxation=settings.relaxation,
                                        threshold=settings.threshold, preconditioner=settings.preconditioner,
                                        mg_smoother=settings.mg_smoother, mg_levels=settings.mg_levels)
            levels = [(fm.Mat.from_handle(r), fm.Mat.from_handle(c)) for r, c in lev]
            if levels_log is not None:
                levels_log.append([(A.nrows, A.nnz)] + [(c.nrows, c.nnz) for _, c in levels])
        return fm.iterative_solve(A, B, X, settings.iterations, method, relaxation=settings.relaxation, threshold=settings.threshold,
                                  preconditioner=settings.preconditioner == po.PC_JACOBI, levels=levels, pos=pos,
                                  mg_smoother=_METHOD[settings.mg_smoother], mg_levels=settings.mg_levels)
    return solve


class State:
    """The locals of solve_steady that live across iterations (src/solver.rs:41-49): the diffusion matrix and sources, the three
    momentum matrices (their diagonals feed the next assembly and the correction) and p'."""

    def __init__(self, om, mu):
        self.a_di, *self.b_di = om.build_momentum_diffusion(mu)
        self.a = [om.init_momentum_matrix() for _ in range(3)]
        self.p_prime = np.zeros(om.n_cells)

    def replay(self, om, settings, rho, fields):
        """The momentum assembly of an iteration that started from `fields` (u, v, w, p): brings the matrices to the state that
        iteration leaves behind, without its solves. With the GPU's field snapshots this starts the model at any iteration."""
        om.build_momentum_advection(*self.a, self.a_di, *fields, settings, rho)


def simple_iterations(om, settings, rho, mu, fields, iterations, solve, state=None, pos=None, first=1, on_iteration=None):
    """`iterations` SIMPLE iterations from `fields` (u, v, w, p) and `state` (a fresh State: the start of solve_steady).
    solve(a, B, X, pos) -> X solves a X_k = B_k for the K rows of B. `pos`: fm.Positions of the cell centroids (both the momentum and
    the pressure-correction matrices carry them on the GPU). Returns one dict per iteration: u, v, w, p, `batched` (the lockstep
    choice), `report` (the 9 columns of oracle.solve_steady's reports: iteration, u/v/w averages as sequential sums / n, Peclet
    avg / min / max, velocity and pressure correction norms), `sums` (math.fsum of u, v, w) and the iteration's `p_prime`. A
    divergence exit raises fm.ModelDiverged (or the solver's own exception) before on_iteration sees that iteration."""
    state = state or State(om, mu)
    n = om.n_cells
    u, v, w, p = (np.array(f, dtype=np.float64) for f in fields)
    out = []
    for it in range(first, first + iterations):
        bu, bv, bw, pe = om.build_momentum_advection(*state.a, state.a_di, u, v, w, p, settings, rho)           # :61-79
        B = np.stack([bu + state.b_di[0], bv + state.b_di[1], bw + state.b_di[2]])                             # :80-82
        a_u, a_v, a_w = state.a
        batched = batchable(settings) and values_identical(a_u, a_v) and values_identical(a_u, a_w)         # capi.cu lockstep
        if batched:
            u, v, w = solve(a_u, B, np.stack([u, v, w]), pos)
        else:
            u, v, w = (solve(a, b[None], x[None], pos)[0] for a, b, x in zip(state.a, B, (u, v, w)))          # :99-136
        pa, pb = om.build_pressure_correction(*state.a, u, v, w, p, settings, rho)                          # :137-148
        state.p_prime = solve(pa, pb[None], (state.p_prime * 0.)[None], pos)[0]                              # :167-179
        u, v, w, p, (pp_norm, vc_norm) = om.apply_pressure_correction(*state.a, state.p_prime, u, v, w, p, settings)  # :193-204
        report = np.array([it, np.cumsum(u)[-1] / n, np.cumsum(v)[-1] / n, np.cumsum(w)[-1] / n, *pe, vc_norm, pp_norm])
        fm.check_field_sums(u, v, w)                                                                         # :217-221
        rec = dict(iteration=it, u=u, v=v, w=w, p=p, p_prime=state.p_prime, batched=batched, report=report,
                   sums=tuple(math.fsum(f) for f in (u, v, w)))
        out.append(rec)
        if on_iteration:
            on_iteration(rec)
    return out
