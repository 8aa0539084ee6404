"""orc_b200 — B200-native (sm_100a, fp64) drop-in for the steady SIMPLE inner loop of reidprichard/ORC.

The product is liborc_b200.so (C ABI in include/orc_b200.h, CUDA sources in orc_b200/csrc). This package is
the host-side mirror of the reference's own interface for that path, module for module:

    reference (Rust)                       here
    io::read_mesh                          orc_b200.io.read_mesh
    mesh::{Mesh, FaceZone, ...}            orc_b200.mesh.{Mesh, FaceConditionTypes}
    settings::{NumericalSettings, ...}     orc_b200.settings.{NumericalSettings, MatrixSolverSettings, ...}
    discretization::build_*                orc_b200.discretization.build_*
    linear_algebra::iterative_solve        orc_b200.linear_algebra.iterative_solve
    solver::solve_steady                   orc_b200.solver.solve_steady
    solver::initialize_flow                orc_b200.solver.initialize_flow
    solver::initialize_flow_new            orc_b200.solver.initialize_flow_new
    io::write_gradients                    orc_b200.io.write_gradients
    tests::channel_flow::solve_channel_flow*   orc_b200.channel_flow.solve_channel_flow[_velocity_inlet]   (the validation cases of src/main.rs)
"""
from . import _lib  # noqa: F401
from ._lib import OrcError  # noqa: F401
from .context import Context, default_context  # noqa: F401
from .settings import (NumericalSettings, MatrixSolverSettings, MomentumDiscretization, PressureInterpolation,  # noqa: F401
                       VelocityInterpolation, GradientReconstructionMethods, SolutionMethod, PreconditionMethod,
                       RestrictionMethods, TVD_LUD, TVD_QUICK, TVD_UMIST)
from .mesh import Mesh, FaceConditionTypes, ScalarCondition  # noqa: F401
from .io import read_mesh, read_data, write_data, write_gradients  # noqa: F401
from .linear_algebra import CsrMatrix, iterative_solve  # noqa: F401
from .solver import (solve_steady, SteadySolver, initialize_flow, initialize_flow_new, check_boundary_conditions,  # noqa: F401
                     SystemConstraintType)
