"""Mirror of the reference's discretization module (src/discretization.rs) + the solver.rs helpers that tests compare."""
import ctypes as C

import numpy as np

from . import _lib
from .context import default_context
from .linear_algebra import CsrMatrix
from .mesh import _f64, _p


def build_momentum_diffusion_matrix(mesh, mu, ctx=None):  # src/discretization.rs:39-131 -> (a_di, b_u, b_v, b_w)
    ctx = ctx or default_context()
    mesh._bind(ctx)
    n = mesh.n_cells
    out = C.c_void_p()
    bu, bv, bw = np.zeros(n), np.zeros(n), np.zeros(n)
    _lib.check(_lib.lib().orc_build_momentum_diffusion(ctx.handle, mesh.handle, C.c_double(mu), C.byref(out), _p(bu), _p(bv), _p(bw)))
    return CsrMatrix(out, ctx), bu, bv, bw


def initialize_momentum_matrix(mesh, ctx=None):  # src/discretization.rs:450-472
    ctx = ctx or default_context()
    mesh._bind(ctx)
    out = C.c_void_p()
    _lib.check(_lib.lib().orc_init_momentum_matrix(ctx.handle, mesh.handle, C.byref(out)))
    return CsrMatrix(out, ctx)


def build_momentum_advection_matrices(a_u, a_v, a_w, a_di, mesh, u, v, w, p, settings, rho):
    """src/discretization.rs:134-356. a_u/a_v/a_w are updated in place; returns (b_u, b_v, b_w, (pe_avg, pe_min, pe_max))."""
    mesh._bind(a_u.ctx)
    n = mesh.n_cells
    s = settings.to_c()
    u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
    bu, bv, bw, pe = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(3)
    _lib.check(_lib.lib().orc_build_momentum_advection(a_u.ctx.handle, mesh.handle, a_u.handle, a_v.handle, a_w.handle, a_di.handle, _p(u),
                                                       _p(v), _p(w), _p(p), C.byref(s), C.c_double(rho), _p(bu), _p(bv), _p(bw), _p(pe)))
    return bu, bv, bw, tuple(pe)


def build_pressure_correction_matrices(mesh, u, v, w, p, a_u, a_v, a_w, settings, rho):  # src/discretization.rs:359-448 -> (a, b)
    mesh._bind(a_u.ctx)
    n = mesh.n_cells
    s = settings.to_c()
    u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
    out = C.c_void_p()
    b = np.zeros(n)
    _lib.check(_lib.lib().orc_build_pressure_correction(a_u.ctx.handle, mesh.handle, a_u.handle, a_v.handle, a_w.handle, _p(u), _p(v), _p(w),
                                                        _p(p), C.byref(s), C.c_double(rho), C.byref(out), _p(b)))
    return CsrMatrix(out, a_u.ctx), b


def calculate_pressure_gradient(mesh, p, ctx=None):  # src/solver.rs:874-902 for every cell -> (N, 3)
    ctx = ctx or default_context()
    mesh._bind(ctx)
    p = _f64(p)
    g = np.zeros((mesh.n_cells, 3))
    _lib.check(_lib.lib().orc_pressure_gradient(ctx.handle, mesh.handle, _p(p), _p(g)))
    return g


def apply_pressure_correction(mesh, a_u, a_v, a_w, p_prime, u, v, w, p, settings):  # src/solver.rs:1170-1227
    mesh._bind(a_u.ctx)
    s = settings.to_c()
    pp = _f64(p_prime)
    u, v, w, p = _f64(u).copy(), _f64(v).copy(), _f64(w).copy(), _f64(p).copy()
    norms = np.zeros(2)
    _lib.check(_lib.lib().orc_apply_pressure_correction(a_u.ctx.handle, mesh.handle, a_u.handle, a_v.handle, a_w.handle, _p(pp), _p(u), _p(v),
                                                        _p(w), _p(p), C.byref(s), _p(norms)))
    return u, v, w, p, tuple(norms)


def build_pressure_laplace(mesh, ctx=None):
    """The system initialize_pressure_field assembles (src/solver.rs:437-494) -> (a, b)."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    out = C.c_void_p()
    b = np.zeros(mesh.n_cells)
    _lib.check(_lib.lib().orc_build_pressure_laplace(ctx.handle, mesh.handle, C.byref(out), _p(b)))
    return CsrMatrix(out, ctx), b


def calculate_gradients(mesh, u, v, w, p, gradient_scheme=0, ctx=None):
    """calculate_pressure_gradient / calculate_velocity_gradient (src/solver.rs:774-949) for every cell -> ((N, 3), (N, 3, 3)).
    gradient_scheme: settings.GradientReconstructionMethods (Green-Gauss cell based or LeastSquares)."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    n = mesh.n_cells
    u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
    gp, gu = np.zeros((n, 3)), np.zeros((n, 3, 3))
    _lib.check(_lib.lib().orc_gradients(ctx.handle, mesh.handle, _p(u), _p(v), _p(w), _p(p), C.c_int32(int(gradient_scheme)), _p(gp), _p(gu)))
    return gp, gu


def build_velocity_potential(mesh, ctx=None):
    """The psi system initialize_velocity_field assembles (src/solver.rs:524-590) -> (a, b)."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    out = C.c_void_p()
    b = np.zeros(mesh.n_cells)
    _lib.check(_lib.lib().orc_build_velocity_potential(ctx.handle, mesh.handle, C.byref(out), _p(b)))
    return CsrMatrix(out, ctx), b


def potential_gradient(mesh, psi, ctx=None):
    """Least-squares gradient of psi over the cell neighbours (src/solver.rs:624-693) -> (u, v, w)."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    psi = _f64(psi)
    n = mesh.n_cells
    u, v, w = np.zeros(n), np.zeros(n), np.zeros(n)
    _lib.check(_lib.lib().orc_potential_gradient(ctx.handle, mesh.handle, _p(psi), _p(u), _p(v), _p(w)))
    return u, v, w


def build_scalar_transport(mesh, a_u, a_v, a_w, u, v, w, p, phi, gamma, rho, settings):
    """The system of one passive scalar sweep (DESIGN.md §1: steady div(rho u phi) - div(Gamma grad phi) = 0; not in the reference)
    with the face fluxes of the flow u, v, w, p and the diagonals of a_u, a_v, a_w, for the given phi -> (a, b). Convection scheme:
    settings.momentum (UD, CD1 or TVD with settings.limiter). On a partition mesh every rank calls it together with its local
    vectors (halo cells included) and gets its local rows."""
    mesh._bind(a_u.ctx)
    n = mesh.n_cells
    s = settings.to_c()
    u, v, w, p, phi = _f64(u), _f64(v), _f64(w), _f64(p), _f64(phi)
    out = C.c_void_p()
    b = np.zeros(n)
    _lib.check(_lib.lib().orc_build_scalar_transport(a_u.ctx.handle, mesh.handle, a_u.handle, a_v.handle, a_w.handle, _p(u), _p(v), _p(w),
                                                     _p(p), _p(phi), C.c_double(gamma), C.c_double(rho), C.byref(s), C.byref(out), _p(b)))
    return CsrMatrix(out, a_u.ctx), b
