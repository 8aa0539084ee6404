"""ctypes loader for liborc_b200.so (the C ABI declared in include/orc_b200.h).

There is no CPU fallback: if the shared library is missing the import fails loudly, and every compute
entry returns ORC_E_CUDA when no sm_100 device is present.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "liborc_b200.so")
CSRC = os.path.join(_HERE, "csrc")

# status codes (include/orc_b200.h)
OK, E_INVALID, E_CUDA, E_NCCL, E_UNSUPPORTED, E_DIVERGED, E_MG_DIVERGED, E_JACOBI_DIVERGED, E_GS_MAINTENANCE, E_GS_DIVERGED, E_IO, \
    E_MISSING_ENTRY, E_INTERNAL = range(13)


class OrcError(RuntimeError):
    """A non-zero status from liborc_b200: the reference would have panicked here (or CUDA failed)."""

    def __init__(self, code, message):
        super().__init__(f"[orc_b200 status {code}] {message}")
        self.code = code
        self.message = message


class Settings(C.Structure):
    """orc_settings: NumericalSettings + MatrixSolverSettings of the reference (src/lib.rs:14-86)."""
    _fields_ = [("momentum", C.c_int32), ("limiter", C.c_int32), ("pressure_interpolation", C.c_int32),
                ("velocity_interpolation", C.c_int32), ("gradient", C.c_int32), ("solver_type", C.c_int32),
                ("preconditioner", C.c_int32), ("mg_smoother", C.c_int32), ("mg_levels", C.c_int32), ("gs_mode", C.c_int32),
                ("assembly_mode", C.c_int32), ("reduction_mode", C.c_int32), ("iterations", C.c_uint64),
                ("pressure_relaxation", C.c_double), ("momentum_relaxation", C.c_double), ("relaxation", C.c_double),
                ("threshold", C.c_double)]


class Report(C.Structure):
    _fields_ = [("iteration", C.c_uint64), ("u_avg", C.c_double), ("v_avg", C.c_double), ("w_avg", C.c_double),
                ("peclet_avg", C.c_double), ("peclet_min", C.c_double), ("peclet_max", C.c_double),
                ("velocity_correction", C.c_double), ("pressure_correction", C.c_double), ("ms_per_iter", C.c_double)]


REPORT_CB = C.CFUNCTYPE(None, C.POINTER(Report), C.c_void_p)

EXPORTS = [
    "orc_settings_default", "orc_ctx_create", "orc_ctx_destroy", "orc_last_error", "orc_version", "orc_ctx_launch_count",
    "orc_ctx_synchronize", "orc_mesh_read", "orc_mesh_from_arrays", "orc_mesh_from_geometry", "orc_mesh_free", "orc_mesh_counts", "orc_mesh_export",
    "orc_mesh_zones", "orc_mesh_geometry_device", "orc_mesh_set_zone", "orc_mesh_pattern", "orc_mesh_levels", "orc_csr_upload", "orc_csr_dims",
    "orc_csr_download", "orc_csr_set_values", "orc_csr_free", "orc_spmv", "orc_jacobi_scale", "orc_iterative_solve",
    "orc_iterative_solve3", "orc_build_restriction", "orc_galerkin", "orc_multigrid_trace", "orc_build_momentum_diffusion", "orc_init_momentum_matrix",
    "orc_build_momentum_advection", "orc_build_pressure_correction", "orc_pressure_gradient", "orc_apply_pressure_correction",
    "orc_solve_steady", "orc_check_boundary_conditions", "orc_build_pressure_laplace", "orc_initialize_flow", "orc_initialize_flow_new", "orc_build_velocity_potential", "orc_potential_gradient", "orc_gradients", "orc_steady_create", "orc_steady_set_fields", "orc_steady_get_fields", "orc_steady_iterate", "orc_steady_reset",
    "orc_steady_phase_ms", "orc_steady_batched", "orc_steady_level_sizes", "orc_steady_gradients", "orc_steady_destroy", "orc_bench_amg_setup", "orc_bench_spmv", "orc_bench_bicgstab", "orc_bench_spmv_batch", "orc_bench_bicgstab_batch", "orc_prof_enable", "orc_prof_config", "orc_prof_get", "orc_prof_get_ref_bytes", "orc_prof_get_spmv_detail", "orc_comm_unique_id", "orc_ctx_comm_init", "orc_ctx_peer_window", "orc_ctx_peer_open", "orc_ctx_peer_disable", "orc_ctx_peer_enabled", "orc_mesh_partition", "orc_mesh_partition_window",
    "orc_mesh_partition_info", "orc_mesh_partition_maps", "orc_mesh_set_zone_scalar", "orc_build_scalar_transport", "orc_steady_solve_scalar",
    "orc_steady_couple_scalar", "orc_steady_set_scalar", "orc_steady_get_scalar", "orc_steady_scalar_zone_flux",
]


def build(force=False):
    """Compile liborc_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    args = ["make", "-C", CSRC, "-s", "-j4"] + (["-B"] if force else [])
    subprocess.check_call(args)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(orc_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.orc_last_error.restype = C.c_char_p
        L.orc_version.restype = C.c_char_p
        L.orc_ctx_launch_count.restype = C.c_uint64
        L.orc_ctx_launch_count.argtypes = [C.c_void_p]
        for name in ("orc_ctx_destroy", "orc_mesh_free", "orc_steady_destroy"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [C.c_void_p]
        L.orc_csr_free.restype = None
        L.orc_csr_free.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_settings_default.restype = None
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise OrcError(rc, lib().orc_last_error().decode(errors="replace"))
