"""TEST INFRASTRUCTURE ONLY. ctypes driver for tests/scalar_oracle/scalar_oracle.cpp, the sequential model of the passive scalar
transport (DESIGN.md §1). It links against the oracle's library (oracle/_build/liborc_oracle.so) for the mesh, the face flux, the
pressure gradient and iterative_solve, and is compiled on first use into a directory under the system's temporary directory (the
repository tree may be read-only)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "scalar_oracle", "scalar_oracle.cpp")
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")

ZERO_GRADIENT, FIXED = 0, 1
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = po.build()
        po.lib()   # loaded first: the model resolves its oracle symbols (and the partition emulation's state) to this copy
        key = hashlib.sha256(open(_SRC, "rb").read() + open(os.path.join(_ORACLE, "orc_oracle.hpp"), "rb").read()
                             + so.encode()).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"orc_scalar_oracle_{os.getuid()}_{key}")
        out = os.path.join(out_dir, "libscalar_oracle.so")
        if not os.path.exists(out):
            os.makedirs(out_dir, exist_ok=True)
            tmp = out + f".{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", _ORACLE, "-o", tmp, _SRC,
                                   so, "-Wl,-rpath," + os.path.dirname(so)])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.so_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def _chk(rc):
    if rc != 0:
        raise po.OraclePanic(lib().so_last_error().decode())


_f64, _i64, _p = po._f64, po._i64, po._p


class ScalarBcs:
    """Per-zone scalar conditions of an oracle mesh (the oracle's FaceZone has no such field): ZERO_GRADIENT unless set."""

    def __init__(self, mesh):
        self.names = mesh.zones()["names"]
        self.kind = np.zeros(len(self.names), np.int64)
        self.value = np.zeros(len(self.names))

    def set(self, name, kind, value=0.0):
        k = self.names.index(name)
        self.kind[k], self.value[k] = kind, value


def unit_diagonals(mesh):
    """a_u = a_v = a_w with diagonal 1 (the momentum matrices solve_steady starts from, src/solver.rs:43-45)."""
    a = mesh.init_momentum_matrix()
    return a, a, a


def face_flux(mesh, u, v, w, p, a_u, a_v, a_w, vel_interp, gradient, side=0):
    """F_f of every face, from the side of c0 (side 0) or of c1 (side 1)."""
    u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
    out = np.zeros(mesh.counts()["faces"])
    _chk(lib().so_face_flux(mesh.h, _p(u), _p(v), _p(w), _p(p), a_u.h, a_v.h, a_w.h, C.c_int64(vel_interp), C.c_int64(gradient),
                            C.c_int64(side), _p(out)))
    return out


def build(mesh, bcs, u, v, w, p, phi, a_u, a_v, a_w, gamma, rho, scheme, limiter, vel_interp, gradient):
    """The system of one sweep -> (oracle Csr, b)."""
    u, v, w, p, phi = _f64(u), _f64(v), _f64(w), _f64(p), _f64(phi)
    iv = _i64([scheme, limiter, vel_interp, gradient])
    out = C.c_void_p()
    b = np.zeros(mesh.n_cells)
    _chk(lib().so_build(mesh.h, _p(u), _p(v), _p(w), _p(p), _p(phi), a_u.h, a_v.h, a_w.h, C.c_double(gamma), C.c_double(rho), _p(iv),
                        _p(bcs.kind), _p(bcs.value), C.byref(out), _p(b)))
    return po.Csr(out), b


def solve(mesh, bcs, u, v, w, p, phi, a_u, a_v, a_w, gamma, rho, settings, sweeps):
    """`sweeps` assemble + iterative_solve sweeps with a pyoracle.Settings -> phi."""
    s = settings
    u, v, w, p = _f64(u), _f64(v), _f64(w), _f64(p)
    x = _f64(phi).copy()
    iv = _i64([s.momentum, s.limiter, s.velocity_interpolation, s.gradient, s.solver_type, s.iterations, s.preconditioner, s.mg_smoother,
               s.mg_levels])
    dv = _f64([s.relaxation, s.threshold])
    _chk(lib().so_solve(mesh.h, _p(u), _p(v), _p(w), _p(p), a_u.h, a_v.h, a_w.h, C.c_double(gamma), C.c_double(rho), _p(iv), _p(dv),
                        _p(bcs.kind), _p(bcs.value), C.c_int64(sweeps), _p(x)))
    return x


def simple_iterations(mesh, settings, rho, mu, iterations):
    """solve_steady's loop (src/solver.rs:41-222) from rest, step by step over the oracle's entries, keeping the momentum
    matrices: -> (u, v, w, p, a_u, a_v, a_w). Equal to pyoracle.Mesh.solve_steady's fields."""
    s = settings
    n = mesh.n_cells
    a_di, bu_di, bv_di, bw_di = mesh.build_momentum_diffusion(mu)
    a_u, a_v, a_w = mesh.init_momentum_matrix(), mesh.init_momentum_matrix(), mesh.init_momentum_matrix()
    u, v, w, p = (np.zeros(n) for _ in range(4))
    pp = np.zeros(n)
    kw = dict(gs_intended=s.gs_intended, mg_smoother=s.mg_smoother, mg_levels=s.mg_levels)
    for _ in range(iterations):
        bu, bv, bw, _ = mesh.build_momentum_advection(a_u, a_v, a_w, a_di, u, v, w, p, s, rho)
        bu, bv, bw = bu + bu_di, bv + bv_di, bw + bw_di
        u = po.iterative_solve(a_u, bu, u, s.iterations, s.solver_type, s.relaxation, s.threshold, s.preconditioner, **kw)
        v = po.iterative_solve(a_v, bv, v, s.iterations, s.solver_type, s.relaxation, s.threshold, s.preconditioner, **kw)
        w = po.iterative_solve(a_w, bw, w, s.iterations, s.solver_type, s.relaxation, s.threshold, s.preconditioner, **kw)
        pc_a, pc_b = mesh.build_pressure_correction(a_u, a_v, a_w, u, v, w, p, s, rho)
        pp = pp * 0.0
        pp = po.iterative_solve(pc_a, pc_b, pp, s.iterations, s.solver_type, s.relaxation, s.threshold, s.preconditioner, **kw)
        u, v, w, p, _ = mesh.apply_pressure_correction(a_u, a_v, a_w, pp, u, v, w, p, s)
    return u, v, w, p, a_u, a_v, a_w


def split_walls(arrays):
    """hex_box / tet_box arrays with the WALL zone split by face position into WALL (y = 0) and WALL_TOP (y = ly)."""
    m = dict(arrays)
    xyz = m["xyz"].reshape(-1, 3)
    off, nodes = m["face_node_offsets"], m["face_nodes"]
    wall = int(m["zone_ids"][m["zone_names"].index("WALL")])
    top = int(m["zone_ids"].max()) + 1
    fz = m["face_zone"].copy()
    ly = m["extent"][1]
    for f in np.nonzero(fz == wall)[0]:
        if xyz[nodes[off[f]:off[f + 1]], 1].mean() > ly / 2:
            fz[f] = top
    m["face_zone"] = fz
    m["zone_ids"] = np.append(m["zone_ids"], top)
    m["zone_types"] = np.append(m["zone_types"], 3)
    m["zone_names"] = list(m["zone_names"]) + ["WALL_TOP"]
    return m
