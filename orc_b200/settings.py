"""Mirror of the reference's `settings` module (src/lib.rs:8-202): same names, same defaults."""
import enum

from . import _lib


class MomentumDiscretization(enum.IntEnum):  # src/lib.rs:89-105
    UD = 0
    CD1 = 1
    CD2 = 2
    TVD = 3


class TvdLimiter(enum.IntEnum):  # psi(r) presets, src/lib.rs:107-118 (a bare fn(Float)->Float in the reference)
    UD = 0
    CD1 = 1
    LUD = 2
    QUICK = 3
    UMIST = 4


TVD_LUD, TVD_QUICK, TVD_UMIST = TvdLimiter.LUD, TvdLimiter.QUICK, TvdLimiter.UMIST


class PressureInterpolation(enum.IntEnum):  # src/lib.rs:120-130
    Linear = 0
    LinearWeighted = 1
    Standard = 2
    SecondOrder = 3
    NONE = 4


class VelocityInterpolation(enum.IntEnum):  # src/lib.rs:132-140
    Linear = 0
    LinearWeighted = 1
    RhieChow = 2
    NONE = 3


class GradientReconstructionMethods(enum.IntEnum):  # src/lib.rs:142-162
    GreenGaussCellBased = 0
    GreenGaussNodeBased = 1
    LeastSquares = 2
    NONE = 3


class SolutionMethod(enum.IntEnum):  # src/lib.rs:170-180
    GaussSeidel = 0
    Jacobi = 1
    Multigrid = 2
    BiCGSTAB = 3


class PreconditionMethod(enum.IntEnum):  # src/lib.rs:182-186
    NONE = 0
    Jacobi = 1


class RestrictionMethods(enum.IntEnum):  # src/lib.rs:197-201
    Injection = 0
    Strongest = 1


class GaussSeidelMode(enum.IntEnum):
    ReferencePanic = 0   # what the reference does: "Gauss-Seidel out for maintenance :)" (src/linear_algebra.rs:245)
    Lexicographic = 1    # intended forward SOR sweep, exact
    Multicolour = 2      # greedy colouring in row order, colours swept in ascending order (DESIGN.md §5)


class AssemblyMode(enum.IntEnum):
    Exact = 0    # reproduces the in-place diagonal recurrence of src/discretization.rs:182-197, 340-351
    Frozen = 1


class ReductionMode(enum.IntEnum):
    Fast = 0             # fused deterministic tree reductions (production, large meshes)
    ReferenceOrder = 1   # nalgebra's 8-accumulator dot order: bit-identical solves, for small meshes
    Auto = 2             # default: ReferenceOrder up to 16384 rows (include/orc_b200.h: ORC_AUTO_EXACT_MAX_ROWS), Fast above


class MatrixSolverSettings:  # src/lib.rs:39-56, defaults :76-86
    def __init__(self, solver_type=SolutionMethod.Multigrid, iterations=50, relaxation=0.5, relative_convergence_threshold=1e-3,
                 preconditioner=PreconditionMethod.Jacobi):
        self.solver_type = solver_type
        self.iterations = iterations
        self.relaxation = relaxation
        self.relative_convergence_threshold = relative_convergence_threshold
        self.preconditioner = preconditioner


class NumericalSettings:  # src/lib.rs:14-35, defaults :58-74
    def __init__(self, momentum=MomentumDiscretization.CD1, limiter=TVD_QUICK, pressure_interpolation=PressureInterpolation.SecondOrder,
                 velocity_interpolation=VelocityInterpolation.RhieChow,
                 gradient_reconstruction=GradientReconstructionMethods.GreenGaussCellBased, pressure_relaxation=0.01,
                 momentum_relaxation=0.5, matrix_solver=None, mg_smoother=SolutionMethod.BiCGSTAB, mg_levels=3,
                 gs_mode=GaussSeidelMode.Lexicographic, assembly_mode=AssemblyMode.Exact, reduction_mode=ReductionMode.Auto):
        self.momentum = momentum
        self.limiter = limiter  # psi when momentum == TVD
        self.pressure_interpolation = pressure_interpolation
        self.velocity_interpolation = velocity_interpolation
        self.gradient_reconstruction = gradient_reconstruction
        self.pressure_relaxation = pressure_relaxation
        self.momentum_relaxation = momentum_relaxation
        self.matrix_solver = matrix_solver or MatrixSolverSettings()
        self.mg_smoother = mg_smoother   # compile-time constants in the reference (src/linear_algebra.rs:9-10)
        self.mg_levels = mg_levels
        self.gs_mode = gs_mode
        self.assembly_mode = assembly_mode
        self.reduction_mode = reduction_mode

    def to_c(self):
        s = _lib.Settings()
        s.momentum = int(self.momentum); s.limiter = int(self.limiter)
        s.pressure_interpolation = int(self.pressure_interpolation); s.velocity_interpolation = int(self.velocity_interpolation)
        s.gradient = int(self.gradient_reconstruction); s.solver_type = int(self.matrix_solver.solver_type)
        s.preconditioner = int(self.matrix_solver.preconditioner); s.mg_smoother = int(self.mg_smoother)
        s.mg_levels = int(self.mg_levels); s.gs_mode = int(self.gs_mode); s.assembly_mode = int(self.assembly_mode); s.reduction_mode = int(self.reduction_mode)
        s.iterations = int(self.matrix_solver.iterations); s.pressure_relaxation = float(self.pressure_relaxation)
        s.momentum_relaxation = float(self.momentum_relaxation); s.relaxation = float(self.matrix_solver.relaxation)
        s.threshold = float(self.matrix_solver.relative_convergence_threshold)
        return s
