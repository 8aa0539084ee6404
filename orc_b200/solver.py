"""Mirror of the reference's solver::solve_steady (src/solver.rs:26-244)."""
import ctypes as C

import numpy as np

from . import _lib
from .context import default_context
from .mesh import _f64, _p


def _exposed_cells(mesh):
    """The cells a call exchanges with the caller: the owned cells of a partition mesh, all cells otherwise."""
    try:
        return mesh.partition_info()["n_own"]
    except _lib.OrcError:
        return mesh.n_cells


def solve_steady(mesh, u, v, w, p, numerical_settings, rho, mu, iteration_count, reporting_interval, ctx=None, on_report=None):
    """Same argument order as the reference. u, v, w, p are numpy float64 vectors updated IN PLACE (the reference's
    &mut DVector). Reports (the line printed at src/solver.rs:213-215) go to `on_report(dict)`; default prints them."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    s = numerical_settings.to_c()
    arrs = [u, v, w, p]
    n_expected = _exposed_cells(mesh)
    for a in arrs:
        if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous and a.size == n_expected):
            raise ValueError("u, v, w, p must be contiguous float64 arrays of length n_cells")
    print("Solving...")

    def _cb(rep_ptr, _user):
        r = rep_ptr.contents
        d = {k: getattr(r, k) for k, _ in _lib.Report._fields_}
        if on_report:
            on_report(d)
        else:
            print(f"Iteration {d['iteration']}: avg velocity = ({d['u_avg']:.2e}, {d['v_avg']:.2e}, {d['w_avg']:.2e})\t"
                  f"avg peclet = {d['peclet_avg']:.1e}\tmin peclet = {d['peclet_min']:.1e}\tmax peclet = {d['peclet_max']:.1e}\t"
                  f"velocity correction: {d['velocity_correction']:.2e}\tpressure correction: {d['pressure_correction']:.2e}\t"
                  f"ms/iter: {d['ms_per_iter']:.1e}")

    cb = _lib.REPORT_CB(_cb)
    rc = _lib.lib().orc_solve_steady(ctx.handle, mesh.handle, _p(u), _p(v), _p(w), _p(p), C.byref(s), C.c_double(rho), C.c_double(mu),
                                     C.c_uint64(iteration_count), C.c_uint64(reporting_interval), cb, None)
    _lib.check(rc)
    print("Done solving.")


class SystemConstraintType:   # src/solver.rs:703-708
    PressureOnly, VelocityOnly, Hybrid = 0, 1, 2


def check_boundary_conditions(mesh):
    """src/solver.rs:710-770. Raises OrcError(E_INVALID, "You must set boundary conditions.") like the reference's panic."""
    out = C.c_int32()
    _lib.check(_lib.lib().orc_check_boundary_conditions(mesh.handle, C.byref(out)))
    return out.value


def initialize_flow(mesh, mu, rho, iteration_count, ctx=None, reduction_mode=0):
    """src/solver.rs:246-352, same argument order; returns (u, v, w, p). `reduction_mode`: settings.ReductionMode (the reference
    has no such knob: ReferenceOrder makes the result bit-identical to its CPU path, Fast is the throughput mode). On a partition
    mesh every rank calls it with its own context and gets the fields of its owned cells."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    n = _exposed_cells(mesh)
    u, v, w, p = (np.zeros(n) for _ in range(4))
    print("Initializing pressure field...")
    print("Initializing velocity field...")
    _lib.check(_lib.lib().orc_initialize_flow(ctx.handle, mesh.handle, C.c_double(mu), C.c_double(rho), C.c_uint64(iteration_count),
                                              C.c_int32(int(reduction_mode)), _p(u), _p(v), _p(w), _p(p)))
    print("Done!")
    return u, v, w, p


def initialize_flow_new(mesh, mu, rho, iteration_count, ctx=None, reduction_mode=2):
    """src/solver.rs:354-410, same argument order; returns (u, v, w, p). What the reference's current main() calls before
    solve_steady (src/tests.rs:195-197): the Laplace pressure field for PressureOnly / Hybrid boundary-condition systems (the
    overlapping match arm: a Hybrid system gets no velocity field), initialize_velocity_field (:511-696) for VelocityOnly ones.
    `reduction_mode`: settings.ReductionMode (default Auto). On a partition mesh every rank calls it with its own context and gets
    the fields of its owned cells."""
    ctx = ctx or default_context()
    mesh._bind(ctx)
    n = _exposed_cells(mesh)
    u, v, w, p = (np.zeros(n) for _ in range(4))
    print("Initializing flow...")
    _lib.check(_lib.lib().orc_initialize_flow_new(ctx.handle, mesh.handle, C.c_double(mu), C.c_double(rho), C.c_uint64(iteration_count),
                                                  C.c_int32(int(reduction_mode)), _p(u), _p(v), _p(w), _p(p)))
    print("Done!")
    return u, v, w, p


class SteadySolver:
    """solve_steady with its locals (src/solver.rs:41-49) kept resident on the device between calls."""

    def __init__(self, mesh, numerical_settings, rho, mu, ctx=None):
        self.ctx = ctx or default_context()
        self.mesh = mesh._bind(self.ctx)
        self._s = numerical_settings.to_c()
        self._h = C.c_void_p()
        _lib.check(_lib.lib().orc_steady_create(self.ctx.handle, mesh.handle, C.byref(self._s), C.c_double(rho), C.c_double(mu),
                                                C.byref(self._h)))
        self.n = _exposed_cells(mesh)

    def set_fields(self, u, v, w, p):
        u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
        _lib.check(_lib.lib().orc_steady_set_fields(self._h, _p(u), _p(v), _p(w), _p(p)))

    def get_fields(self):
        u, v, w, p = (np.zeros(self.n) for _ in range(4))
        _lib.check(_lib.lib().orc_steady_get_fields(self._h, _p(u), _p(v), _p(w), _p(p)))
        return u, v, w, p

    def iterate(self, iterations=1):
        rep = _lib.Report()
        _lib.check(_lib.lib().orc_steady_iterate(self._h, C.c_uint64(iterations), C.byref(rep)))
        return {k: getattr(rep, k) for k, _ in _lib.Report._fields_}

    def gradients(self, gradient_scheme=0):
        """discretization.calculate_gradients of the resident fields -> ((n, 3), (n, 3, 3)), n = the exposed (owned) cells. On a
        partition mesh every rank calls it together (the fields' halo cells are exchanged first)."""
        gp, gu = np.zeros((self.n, 3)), np.zeros((self.n, 3, 3))
        _lib.check(_lib.lib().orc_steady_gradients(self._h, C.c_int32(int(gradient_scheme)), _p(gp), _p(gu)))
        return gp, gu

    def write_gradients(self, output_file_name, decimal_precision, gradient_scheme):
        """io.write_gradients of the resident fields. A partition writes the lines of its owned cells: the rank files, concatenated
        in rank order, are the whole mesh's file."""
        from .io import _owned_centroids, _write_gradient_lines
        gp, gu = self.gradients(gradient_scheme)
        _write_gradient_lines(output_file_name, _owned_centroids(self.mesh), gp, gu, decimal_precision)

    def solve_scalar(self, gamma, phi=None, sweeps=1):
        """A passive scalar carried by the resident flow (DESIGN.md §1; not in the reference): `sweeps` assemble + solve sweeps of
        steady div(rho u phi) - div(gamma grad phi) = 0 with the handle's settings (convection scheme settings.momentum, the
        matrix solver of settings.matrix_solver) and the zones' scalar conditions (Mesh.set_zone_scalar). Starts from `phi` (zero by
        default) and returns phi of the exposed cells. The flow state is left as it was. On a partition mesh every rank calls it
        together."""
        x = np.zeros(self.n) if phi is None else _f64(phi).copy()
        if x.size != self.n:
            raise ValueError("phi must have one value per exposed cell")
        _lib.check(_lib.lib().orc_steady_solve_scalar(self._h, C.c_double(gamma), C.c_uint64(sweeps), _p(x)))
        return x

    def couple_scalar(self, gamma, beta, phi_ref, gravity, sweeps=1):
        """Buoyancy-driven flow (Boussinesq, DESIGN.md §1; not in the reference): from now on every iterate() adds the body force
        -rho * beta * (phi - phi_ref) * gravity of the resident scalar to the momentum equations and, after the pressure correction,
        runs `sweeps` sweeps of the scalar transport of solve_scalar(gamma) from the resident phi. p becomes the reduced pressure.
        `gravity` is (g_x, g_y, g_z). reset() zeroes phi and keeps the coupling."""
        gx, gy, gz = (float(g) for g in gravity)
        if sweeps < 1:
            raise ValueError("sweeps must be >= 1 (uncouple_scalar() uncouples)")
        _lib.check(_lib.lib().orc_steady_couple_scalar(self._h, C.c_double(gamma), C.c_double(beta), C.c_double(phi_ref), C.c_double(gx),
                                                       C.c_double(gy), C.c_double(gz), C.c_uint64(sweeps)))

    def uncouple_scalar(self):
        """Back to the plain loop: iterate() neither adds a body force nor solves for phi (the resident phi is kept)."""
        _lib.check(_lib.lib().orc_steady_couple_scalar(self._h, C.c_double(0.0), C.c_double(0.0), C.c_double(0.0), C.c_double(0.0),
                                                       C.c_double(0.0), C.c_double(0.0), C.c_uint64(0)))

    def set_scalar(self, phi):
        """The resident phi of the exposed cells."""
        x = _f64(phi)
        if x.size != self.n:
            raise ValueError("phi must have one value per exposed cell")
        _lib.check(_lib.lib().orc_steady_set_scalar(self._h, _p(x)))

    def get_scalar(self):
        x = np.zeros(self.n)
        _lib.check(_lib.lib().orc_steady_get_scalar(self._h, _p(x)))
        return x

    def scalar_zone_flux(self, name):
        """(diffusive, convective) outward flux of the resident phi through zone `name` on the resident flow (coupled handles only:
        the diffusivity is the coupling's gamma). On a partition mesh every rank calls it together and gets the whole zone's flux."""
        out = np.zeros(2)
        _lib.check(_lib.lib().orc_steady_scalar_zone_flux(self._h, name.encode(), _p(out)))
        return float(out[0]), float(out[1])

    def reset(self):
        """Back to the state solve_steady starts from: zero fields, momentum matrices re-initialised (diag 1)."""
        _lib.check(_lib.lib().orc_steady_reset(self._h))

    def phase_ms(self):
        out = np.zeros(5)
        _lib.check(_lib.lib().orc_steady_phase_ms(self._h, _p(out)))
        return dict(zip(("momentum_assembly", "momentum_solves", "pressure_assembly", "pressure_solve", "correction"), out.tolist()))

    @property
    def batched(self):
        """True if the last iterate() solved u, v, w in lockstep (a_u == a_v == a_w bit for bit; ORC_B200_BATCH=0 disables)."""
        out = C.c_int32()
        _lib.check(_lib.lib().orc_steady_batched(self._h, C.byref(out)))
        return bool(out.value)

    def level_sizes(self):
        out = np.zeros(16, np.int64)
        n = C.c_int32()
        _lib.check(_lib.lib().orc_steady_level_sizes(self._h, _p(out), C.c_int32(8), C.byref(n)))
        return [(int(out[2 * l]), int(out[2 * l + 1])) for l in range(n.value)]

    def close(self):
        if self._h:
            _lib.lib().orc_steady_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
