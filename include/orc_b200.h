/* orc_b200.h — C ABI of liborc_b200.so: a B200-native (sm_100a, fp64, hand-written CUDA) drop-in for
 * the steady SIMPLE inner loop of reidprichard/ORC.
 *
 * ORC has no FFI of its own: the boundary is the set of public Rust functions of the `orc` crate
 * that sit on the hot path (SURVEY.md §8b). Every entry point below names the reference function
 * it replaces (file:line into the reference tree). The Rust-side binding a maintainer would add is
 * shown in INTEGRATION.md (rust/orc-b200-sys).
 *
 * Conventions
 *  - plain C: opaque handles, pointers and sizes. No C++/torch types cross the boundary.
 *  - every function returns an int32 status (ORC_OK == 0). The reference's error channel is
 *    panic!(); each panic site on the path maps to a status code, nothing unwinds across the ABI.
 *    orc_last_error() returns the message of the last failure on the calling thread.
 *  - all `double*` / `int*` arguments are HOST pointers unless the name ends in `_dev`; the
 *    library copies to/from the device inside the call. Matrices live on the device behind
 *    orc_csr handles (the reference's CsrMatrix<f64> locals of solve_steady never leave the call
 *    either, src/solver.rs:41-49).
 *  - one context per device per process, single host thread (the reference is single-threaded).
 *  - there is NO CPU fallback: every compute entry fails with ORC_E_CUDA when no sm_100 device
 *    (or no CUDA driver) is present.
 */
#ifndef ORC_B200_H
#define ORC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------------------------- */
enum {
    ORC_OK = 0,
    ORC_E_INVALID = 1,          /* bad argument / dimension mismatch (nalgebra dimension panics)        */
    ORC_E_CUDA = 2,             /* CUDA runtime failure, or no usable device                            */
    ORC_E_NCCL = 3,             /* NCCL failure (multi-GPU)                                             */
    ORC_E_UNSUPPORTED = 4,      /* scheme/BC the reference panics on: src/discretization.rs:114-117,287;
                                   src/solver.rs:901,993-995,1001,1100,1134-1137,1148                   */
    ORC_E_DIVERGED = 5,         /* "solution diverged"                       src/solver.rs:217-221      */
    ORC_E_MG_DIVERGED = 6,      /* "Multigrid diverged"                      src/linear_algebra.rs:103  */
    ORC_E_JACOBI_DIVERGED = 7,  /* "diverged" / "max solution value > 10^10" src/linear_algebra.rs:192-196,214-216 */
    ORC_E_GS_MAINTENANCE = 8,   /* "Gauss-Seidel out for maintenance :)"     src/linear_algebra.rs:245  */
    ORC_E_GS_DIVERGED = 9,      /* "****** Solution diverged ******"         src/linear_algebra.rs:240  */
    ORC_E_IO = 10,              /* mesh file unreadable / malformed          src/io.rs:32-515 expects   */
    ORC_E_MISSING_ENTRY = 11,   /* CsrMatrix::get on an un-stored entry      src/lib.rs:664-666         */
    ORC_E_INTERNAL = 12         /* a dataflow kernel exceeded its spin bound (never expected)           */
};

/* ---- settings (src/lib.rs:14-201). Enum values are part of the ABI. ------------------------ */
enum { ORC_MOM_UD = 0, ORC_MOM_CD1 = 1, ORC_MOM_CD2 = 2, ORC_MOM_TVD = 3 };                 /* lib.rs:89-105  */
enum { ORC_PSI_UD = 0, ORC_PSI_CD1 = 1, ORC_PSI_LUD = 2, ORC_PSI_QUICK = 3, ORC_PSI_UMIST = 4 }; /* lib.rs:107-118 */
enum { ORC_P_LINEAR = 0, ORC_P_LINEAR_WEIGHTED = 1, ORC_P_STANDARD = 2, ORC_P_SECOND_ORDER = 3, ORC_P_NONE = 4 }; /* lib.rs:120-130 */
enum { ORC_V_LINEAR = 0, ORC_V_LINEAR_WEIGHTED = 1, ORC_V_RHIE_CHOW = 2, ORC_V_NONE = 3 };  /* lib.rs:132-140 */
enum { ORC_G_GREEN_GAUSS_CELL = 0, ORC_G_GREEN_GAUSS_NODE = 1, ORC_G_LEAST_SQUARES = 2, ORC_G_NONE = 3 }; /* lib.rs:142-162 */
enum { ORC_SOLVER_GAUSS_SEIDEL = 0, ORC_SOLVER_JACOBI = 1, ORC_SOLVER_MULTIGRID = 2, ORC_SOLVER_BICGSTAB = 3 }; /* lib.rs:170-180 */
enum { ORC_PC_NONE = 0, ORC_PC_JACOBI = 1 };                                                /* lib.rs:182-186 */
enum { ORC_RESTRICT_INJECTION = 0, ORC_RESTRICT_STRONGEST = 1 };                            /* lib.rs:197-201 */
/* TGRID boundary ids, src/mesh.rs:50-66 */
enum { ORC_BC_INTERIOR = 2, ORC_BC_WALL = 3, ORC_BC_PRESSURE_INLET = 4, ORC_BC_PRESSURE_OUTLET = 5, ORC_BC_SYMMETRY = 7,
       ORC_BC_VELOCITY_INLET = 10 };
/* Gauss-Seidel behaviour. The reference arm always panics (src/linear_algebra.rs:219-246). */
enum { ORC_GS_REFERENCE_PANIC = 0, /* run nothing, return ORC_E_GS_MAINTENANCE                                   */
       ORC_GS_LEXICOGRAPHIC = 1,   /* intended forward SOR sweep in row order, exact (dataflow kernel)           */
       ORC_GS_MULTICOLOUR = 2 };   /* greedy colouring in row order, colours swept in ascending order (DESIGN.md);
                                      structurally symmetric patterns only (else ORC_E_UNSUPPORTED)          */
/* Momentum assembly recurrence (SURVEY.md Q2, src/discretization.rs:182-197 + :340-351). */
enum { ORC_ASSEMBLY_EXACT = 0,  /* cell i sees NEW diagonals of neighbours j<i, OLD of j>i, like the reference     */
       ORC_ASSEMBLY_FROZEN = 1 }; /* every face sees previous-iteration diagonals (documented deviation)            */

/* Global reductions (dot products, norms) of the solvers. */
enum { ORC_REDUCE_FAST = 0,             /* fused, deterministic block-tree sums: equal to the reference up to summation order */
       ORC_REDUCE_REFERENCE_ORDER = 1,  /* nalgebra's 8-accumulator order: the whole solve is bit-identical to the reference's
                                           CPU path; latency bound by construction, meant for small meshes (configs 1-2)   */
       ORC_REDUCE_AUTO = 2 };           /* default: REFERENCE_ORDER for systems of at most ORC_AUTO_EXACT_MAX_ROWS rows (decided once,
                                           on the fine system of the call), FAST above. On the reference's own small, exactly
                                           axis-aligned meshes the v / w right-hand sides are rounding noise and the unguarded
                                           BiCGSTAB (src/linear_algebra.rs:255-268) divides noise by noise: only the reference's
                                           own summation order reproduces its outcome there (channel_flow.msh: FAST ends in
                                           "Multigrid diverged" where the reference converges), and it is cheap at that size.   */
#define ORC_AUTO_EXACT_MAX_ROWS 16384

typedef struct orc_settings {   /* NumericalSettings + MatrixSolverSettings, defaults src/lib.rs:58-86 */
    int32_t momentum;               /* ORC_MOM_*   default CD1                                  */
    int32_t limiter;                /* ORC_PSI_*   psi(r) when momentum == TVD (lib.rs:104)     */
    int32_t pressure_interpolation; /* ORC_P_*     default SECOND_ORDER                         */
    int32_t velocity_interpolation; /* ORC_V_*     default RHIE_CHOW                            */
    int32_t gradient;               /* ORC_G_*     default GREEN_GAUSS_CELL                     */
    int32_t solver_type;            /* ORC_SOLVER_* default MULTIGRID                           */
    int32_t preconditioner;         /* ORC_PC_*    default JACOBI                               */
    int32_t mg_smoother;            /* compile-time const in the reference: BiCGSTAB (linear_algebra.rs:9)  */
    int32_t mg_levels;              /* compile-time const in the reference: 3        (linear_algebra.rs:10) */
    int32_t gs_mode;                /* ORC_GS_*                                                 */
    int32_t assembly_mode;          /* ORC_ASSEMBLY_*                                           */
    int32_t reduction_mode;         /* ORC_REDUCE_*                                             */
    uint64_t iterations;            /* matrix_solver.iterations, default 50                     */
    double pressure_relaxation;     /* default 0.01 */
    double momentum_relaxation;     /* default 0.5  */
    double relaxation;              /* matrix_solver.relaxation, default 0.5                    */
    double threshold;               /* matrix_solver.relative_convergence_threshold, 1e-3       */
} orc_settings;
/* Fills the reference defaults (src/lib.rs:58-86) + {BiCGSTAB smoother, 3 levels, lexicographic GS, exact assembly}. */
void orc_settings_default(orc_settings* s);

/* ---- context ------------------------------------------------------------------------------- */
typedef struct orc_ctx orc_ctx;
typedef struct orc_mesh orc_mesh;
typedef struct orc_csr orc_csr;
typedef struct orc_steady orc_steady;

/* `stream` is a cudaStream_t (0 = the library creates its own). All work of the context is issued on it. */
int32_t orc_ctx_create(int32_t device, void* stream, orc_ctx** out);
void orc_ctx_destroy(orc_ctx* ctx);
const char* orc_last_error(void);
const char* orc_version(void);
/* number of kernels this library has launched on this context since creation (bench.py: gpu_launches) */
uint64_t orc_ctx_launch_count(orc_ctx* ctx);
int32_t orc_ctx_synchronize(orc_ctx* ctx);

/* ---- mesh: src/io.rs:32-515 read_mesh, src/mesh.rs:181-195 Mesh/get_face_zone -------------- */
/* Host-side TGRID ASCII reader + geometry (normals, centroids, areas, volumes: io.rs:289-438),
 * flattening to SoA, CSR pattern + face->nnz scatter maps + assembly level schedule. No GPU needed
 * until the first compute entry uploads the device mirror (lazily). */
int32_t orc_mesh_read(const char* path, orc_mesh** out);
/* Same geometry pass over in-memory TGRID-style connectivity: node ids 0-based; c0/c1 1-based cell ids, 0 = none. */
int32_t orc_mesh_from_arrays(int32_t dimensions, int64_t n_nodes, const double* xyz, int64_t n_faces,
                             const int64_t* face_node_offsets, const int64_t* face_nodes, const int64_t* c0, const int64_t* c1,
                             const int64_t* face_zone, int64_t n_zones, const int64_t* zone_ids, const int64_t* zone_types,
                             const char* const* zone_names, orc_mesh** out);
/* The caller's own Mesh (src/mesh.rs:181-187), flattened WITH the geometry the reference computed (io.rs:289-438): nothing is
 * recomputed, so the coefficients are built from the reference's own areas / normals / volumes. face_c0 / face_c1: 0-based
 * cell_indices[0] / cell_indices[1] (-1 = none); face_zone: zone ids; cell face lists ascending per cell (io.rs:404-411).
 * Meshes made this way have no nodes: orc_mesh_counts reports 0 of them. */
int32_t orc_mesh_from_geometry(int32_t dimensions, int64_t n_cells, int64_t n_faces, const int64_t* face_c0, const int64_t* face_c1,
                               const int64_t* face_zone, const double* face_area, const double* face_normal3, const double* face_centroid3,
                               const double* cell_volume, const double* cell_centroid3, const int64_t* cell_face_offsets,
                               const int64_t* cell_face_indices, int64_t n_zones, const int64_t* zone_ids, const int64_t* zone_types,
                               const char* const* zone_names, orc_mesh** out);
void orc_mesh_free(orc_mesh* m);
/* out[0..7] = cells, faces, nodes, zones, sum of cell face-list lengths, dimensions, nnz, assembly levels */
int32_t orc_mesh_counts(const orc_mesh* m, int64_t* out8);
/* SoA export for parity checks (bit-exact against the oracle's restatement of io.rs geometry). */
int32_t orc_mesh_export(const orc_mesh* m, int64_t* face_c0, int64_t* face_c1, int64_t* face_zone, double* face_area,
                        double* face_normal3, double* face_centroid3, double* cell_volume, double* cell_centroid3,
                        int64_t* cell_face_offsets, int64_t* cell_face_indices);
/* zone table in ascending zone-id order; names into 64-byte slots */
/* The geometry pass of io::read_mesh (src/io.rs:289-438: face normal / centroid / area, cell centroid / volume) recomputed ON THE DEVICE
 * from the mesh's node coordinates, for multi-million-cell meshes: same operator order as the host pass, bit-identical results. Outputs
 * are host arrays (F, 3F, 3F, N, 3N doubles); device_ms (may be NULL) receives the device time of the two kernels. Meshes without nodes
 * (orc_mesh_from_geometry, partitions) return ORC_E_INVALID. */
int32_t orc_mesh_geometry_device(orc_ctx* ctx, const orc_mesh* m, double* face_area, double* face_normal3, double* face_centroid3,
                                 double* cell_volume, double* cell_centroid3, double* device_ms);
int32_t orc_mesh_zones(const orc_mesh* m, int64_t* ids, int64_t* types, double* scalar, double* vector3, char* names64);
/* mesh.get_face_zone(name) + assignment of zone_type/scalar_value/vector_value (src/tests.rs:60-76) */
int32_t orc_mesh_set_zone(orc_mesh* m, const char* name, int64_t zone_type, double scalar, double vx, double vy, double vz);
/* the shared sparsity pattern (diag + face neighbours, sorted columns): rowptr[N+1], col[nnz] */
int32_t orc_mesh_pattern(const orc_mesh* m, int64_t* rowptr, int64_t* col);
/* assembly level schedule (host logic, testable without a GPU): level_of_cell[N] */
int32_t orc_mesh_levels(const orc_mesh* m, int64_t* level_of_cell);

/* ---- CSR handles (nalgebra-sparse CsrMatrix<f64> on the device) ----------------------------- */
int32_t orc_csr_upload(orc_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* rowptr, const int64_t* col, const double* val,
                       orc_csr** out);
int32_t orc_csr_dims(const orc_csr* a, int64_t* out3 /* nrows, ncols, nnz */);
int32_t orc_csr_download(orc_ctx* ctx, const orc_csr* a, int64_t* rowptr, int64_t* col, double* val);
int32_t orc_csr_set_values(orc_ctx* ctx, orc_csr* a, const double* val);
void orc_csr_free(orc_ctx* ctx, orc_csr* a);
/* y = A x   (&CsrMatrix * &DVector, call sites src/linear_algebra.rs:82,97,140,165,199,202,250,256,260,283) */
int32_t orc_spmv(orc_ctx* ctx, const orc_csr* a, const double* x, double* y);
/* A' = diag(1/a_ii) A, b' = diag(1/a_ii) b   (src/linear_algebra.rs:157-168) */
int32_t orc_jacobi_scale(orc_ctx* ctx, const orc_csr* a, const double* b, orc_csr** a_out, double* b_out);

/* ---- linear_algebra.rs ---------------------------------------------------------------------- */
/* iterative_solve (src/linear_algebra.rs:144-299). x is in/out. Uses s->solver_type, iterations, relaxation,
 * threshold, preconditioner, mg_smoother, mg_levels, gs_mode. */
int32_t orc_iterative_solve(orc_ctx* ctx, const orc_csr* a, const double* b, double* x, const orc_settings* s);
/* Three iterative_solve calls that share the matrix (the u, v, w momentum solves of src/solver.rs:99-136 when a_u, a_v, a_w hold
 * the same values) run in lockstep: the matrix and the AMG hierarchy are read / built once. Every system gets the arithmetic
 * of its own orc_iterative_solve call. BiCGSTAB and Multigrid(BiCGSTAB smoother) only, else ORC_E_UNSUPPORTED. */
int32_t orc_iterative_solve3(orc_ctx* ctx, const orc_csr* a, const double* b0, const double* b1, const double* b2, double* x0, double* x1,
                             double* x2, const orc_settings* s);
/* build_restriction_matrix (src/linear_algebra.rs:12-63) */
int32_t orc_build_restriction(orc_ctx* ctx, const orc_csr* a, int32_t method, orc_csr** r_out);
/* a' = R * a * R^T  (src/linear_algebra.rs:84: (R*A)*R.transpose(), symbolic-union pattern) */
int32_t orc_galerkin(orc_ctx* ctx, const orc_csr* r, const orc_csr* a, orc_csr** out);
/* Multigrid solve that keeps R_l and A_l of every coarse level it built (parity tests). Handles are owned by the caller. */
int32_t orc_multigrid_trace(orc_ctx* ctx, const orc_csr* a, const double* b, double* x, const orc_settings* s, int32_t max_out,
                            orc_csr** r_levels, orc_csr** a_levels, int32_t* n_levels);

/* ---- discretization.rs ---------------------------------------------------------------------- */
/* build_momentum_diffusion_matrix (src/discretization.rs:39-131) */
int32_t orc_build_momentum_diffusion(orc_ctx* ctx, orc_mesh* m, double mu, orc_csr** a_di, double* b_u, double* b_v, double* b_w);
/* initialize_momentum_matrix (src/discretization.rs:450-472) */
int32_t orc_init_momentum_matrix(orc_ctx* ctx, orc_mesh* m, orc_csr** out);
/* build_momentum_advection_matrices (src/discretization.rs:134-356): a_u/a_v/a_w in/out, b_* and peclet3 = (avg,min,max) out */
int32_t orc_build_momentum_advection(orc_ctx* ctx, orc_mesh* m, orc_csr* a_u, orc_csr* a_v, orc_csr* a_w, const orc_csr* a_di,
                                     const double* u, const double* v, const double* w, const double* p, const orc_settings* s,
                                     double rho, double* b_u, double* b_v, double* b_w, double* peclet3);
/* build_pressure_correction_matrices (src/discretization.rs:359-448) */
int32_t orc_build_pressure_correction(orc_ctx* ctx, orc_mesh* m, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w,
                                      const double* u, const double* v, const double* w, const double* p, const orc_settings* s,
                                      double rho, orc_csr** a_out, double* b_out);

/* ---- solver.rs ------------------------------------------------------------------------------ */
/* calculate_pressure_gradient for every cell (src/solver.rs:874-902, Green-Gauss cell based, incl. the Float*Vector quirk) */
int32_t orc_pressure_gradient(orc_ctx* ctx, orc_mesh* m, const double* p, double* grad3n);
/* apply_pressure_correction (src/solver.rs:1170-1227); norms2 = (|p'|, sqrt(sum |du|^2)) */
int32_t orc_apply_pressure_correction(orc_ctx* ctx, orc_mesh* m, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w,
                                      const double* p_prime, double* u, double* v, double* w, double* p, const orc_settings* s,
                                      double* norms2);

/* One report per `report_every` iterations: the scalars printed at src/solver.rs:213-215. */
typedef struct orc_report {
    uint64_t iteration;
    double u_avg, v_avg, w_avg, peclet_avg, peclet_min, peclet_max, velocity_correction, pressure_correction, ms_per_iter;
} orc_report;
typedef void (*orc_report_cb)(const orc_report*, void* user);

/* solve_steady (src/solver.rs:26-244): u, v, w, p are host in/out vectors of length n_cells. */
int32_t orc_solve_steady(orc_ctx* ctx, orc_mesh* m, double* u, double* v, double* w, double* p, const orc_settings* s, double rho,
                         double mu, uint64_t iteration_count, uint64_t reporting_interval, orc_report_cb cb, void* user);

/* The same loop with its state kept resident on the device between calls (what solve_steady's locals are,
 * src/solver.rs:41-49): create = lines 41-49, iterate = the body of the loop at :60-222. */
int32_t orc_steady_create(orc_ctx* ctx, orc_mesh* m, const orc_settings* s, double rho, double mu, orc_steady** out);
int32_t orc_steady_set_fields(orc_steady* st, const double* u, const double* v, const double* w, const double* p);
int32_t orc_steady_get_fields(orc_steady* st, double* u, double* v, double* w, double* p);
int32_t orc_steady_iterate(orc_steady* st, uint64_t iterations, orc_report* last /* nullable */);
/* back to the state solve_steady starts from (src/solver.rs:43-49): zero fields, momentum matrices re-initialised */
int32_t orc_steady_reset(orc_steady* st);
/* per-phase device time (ms, CUDA events) accumulated since creation:
 * momentum assembly, 3 momentum solves, pressure assembly, pressure solve, correction */
int32_t orc_steady_phase_ms(orc_steady* st, double* out5);
/* 1 if the last orc_steady_iterate solved u, v, w in lockstep (a_u == a_v == a_w bit for bit, checked on the device; env
 * ORC_B200_BATCH=0 disables it), 0 if they were solved one after the other. */
int32_t orc_steady_batched(orc_steady* st, int32_t* out);
/* per-level sizes of the last Multigrid solve: out[2*l] = rows, out[2*l+1] = nnz, l = 0..levels */
int32_t orc_steady_level_sizes(orc_steady* st, int64_t* out, int32_t cap, int32_t* n_levels);
/* orc_gradients of the handle's resident u, v, w, p, without their round trip through the host: the OWNED rows (n_own of a
 * partition, after a halo exchange of the four fields), same layout, NULL outputs and errors as orc_gradients. */
int32_t orc_steady_gradients(orc_steady* st, int32_t gradient, double* grad_p3n, double* grad_u9n);
void orc_steady_destroy(orc_steady* st);

/* ---- flow initialisation: the step before the loop (src/solver.rs:246-352) ------------------------- */
enum { ORC_CONSTRAINT_PRESSURE_ONLY = 0, ORC_CONSTRAINT_VELOCITY_ONLY = 1, ORC_CONSTRAINT_HYBRID = 2 };  /* src/solver.rs:703-708 */
/* check_boundary_conditions (src/solver.rs:710-770). "You must set boundary conditions." -> ORC_E_INVALID. Host logic. */
int32_t orc_check_boundary_conditions(const orc_mesh* m, int32_t* constraint_type);
/* the Laplace system assembled by initialize_pressure_field (src/solver.rs:437-494); b_out: n_cells doubles */
int32_t orc_build_pressure_laplace(orc_ctx* ctx, orc_mesh* m, orc_csr** a_out, double* b_out);
/* initialize_flow (src/solver.rs:246-352): returns u, v, w, p (n_cells doubles each, host). `reduction_mode` as in orc_settings.
 * Both initialisations also take a partition mesh (all ranks call them together): they write its OWNED cells (n_own doubles), as
 * orc_steady_get_fields does; ORC_REDUCE_REFERENCE_ORDER is single-GPU only (ORC_E_UNSUPPORTED), Auto means Fast there. */
int32_t orc_initialize_flow(orc_ctx* ctx, orc_mesh* m, double mu, double rho, uint64_t iteration_count, int32_t reduction_mode, double* u,
                            double* v, double* w, double* p);
/* initialize_flow_new (src/solver.rs:354-410; the reference's current main() calls it, src/tests.rs:195-197): pressure field for
 * PressureOnly / Hybrid constraint systems, initialize_velocity_field (:511-696) for VelocityOnly ones. mu, rho and iteration_count
 * are accepted and unused, like in the reference. */
int32_t orc_initialize_flow_new(orc_ctx* ctx, orc_mesh* m, double mu, double rho, uint64_t iteration_count, int32_t reduction_mode, double* u,
                                double* v, double* w, double* p);
/* the potential system of initialize_velocity_field (:524-590) and the least-squares gradient of psi over the neighbours (:624-693) */
int32_t orc_build_velocity_potential(orc_ctx* ctx, orc_mesh* m, orc_csr** a_out, double* b_out);
int32_t orc_potential_gradient(orc_ctx* ctx, orc_mesh* m, const double* psi, double* u, double* v, double* w);
/* calculate_pressure_gradient / calculate_velocity_gradient for every cell (src/solver.rs:774-949) with `gradient` = ORC_G_*:
 * Green-Gauss cell based or least squares. grad_p3n: N x 3; grad_u9n: N x 9 row-major tensors; either may be NULL.
 * A singular least-squares system returns ORC_E_INVALID (the reference unwraps a None, :855, :945). */
int32_t orc_gradients(orc_ctx* ctx, orc_mesh* m, const double* u, const double* v, const double* w, const double* p, int32_t gradient,
                      double* grad_p3n, double* grad_u9n);

/* ---- multi-GPU: one process per GPU, the mesh partitioned by contiguous cell ranges (SURVEY.md §8e) ----------- */
/* NCCL communicator of a context. Rank 0 calls orc_comm_unique_id and ships the 128 bytes to the other ranks (the Python
 * host does it with torch.distributed); every rank then calls orc_ctx_comm_init. */
int32_t orc_comm_unique_id(char* out128);
int32_t orc_ctx_comm_init(orc_ctx* ctx, int32_t rank, int32_t nranks, const char* id128);
/* Peer windows: symmetric memory over CUDA IPC (NVLink / NVSwitch, one node). With them the halo exchange and the small allreduces of
 * the distributed BiCGSTAB run as this library's own kernels over peer stores (one-shot allreduce fused with the scalar update, push /
 * wait-and-unpack halo exchange) instead of NCCL calls. Step 1: every rank allocates its window and gets a 64-byte handle; step 2:
 * every rank maps the handles of all ranks (nranks x 64 bytes, by rank). If any rank fails, ALL ranks call orc_ctx_peer_disable. */
int32_t orc_ctx_peer_window(orc_ctx* ctx, char* handle_out64);
int32_t orc_ctx_peer_open(orc_ctx* ctx, const char* all_handles);
int32_t orc_ctx_peer_disable(orc_ctx* ctx);
int32_t orc_ctx_peer_enabled(orc_ctx* ctx, int32_t* out);
/* The rank's share of a (global) mesh: [lower halo | owned cells | upper halo] in ascending global id, every face of an
 * owned cell, geometry copied from the global mesh, plus the halo-exchange plan. Host logic only (no GPU needed).
 * orc_steady_* on a partition mesh exchange halos (ncclSend/Recv), allreduce the BiCGSTAB scalars, and build the AMG
 * hierarchy per partition. set_fields / get_fields then take the OWNED cells (n_own values, global order). */
int32_t orc_mesh_partition(const orc_mesh* global, int32_t rank, int32_t nranks, orc_mesh** out);
/* The same from a WINDOW of the global mesh that holds this rank's cells and all their face neighbours (e.g. a slab of a
 * structured box plus two layers on each side, so that halo cells keep all their faces and hence their exact geometry):
 * rank q owns the window cells [cuts[q], cuts[q+1]) (nranks + 1 ascending entries, clamped to the window); window cell 0 has
 * global id `id_offset`. Lets every rank build only its part of a multi-million-cell mesh. */
int32_t orc_mesh_partition_window(const orc_mesh* window, int32_t rank, int32_t nranks, const int64_t* cuts, int64_t id_offset,
                                  int64_t n_global, orc_mesh** out);
/* out[0..7] = g0, g1 (owned global range), n_lo, n_own, n_hi, neighbours, total send count, global cells */
int32_t orc_mesh_partition_info(const orc_mesh* m, int64_t* out8);
int32_t orc_mesh_partition_maps(const orc_mesh* m, int64_t* local_to_global, int32_t* nbr_rank, int32_t* send_ptr, int32_t* send_idx,
                                int32_t* recv_begin, int32_t* recv_count);

/* ---- measurement hooks (bench.py roofline leg) ---------------------------------------------- */
/* Per-kernel-class device timing: CUDA events on the context stream around every launch of the class.
 * classes: 0 SpMV (all fused epilogues; bytes = 12 nnz + 20 n per launch), 1 BiCGSTAB vector kernels,
 * 2 assembly, 3 restriction build, 4 Galerkin product, 5 Jacobi scaling, 6 other. */
int32_t orc_prof_enable(orc_ctx* ctx, int32_t on);
/* which kernel classes are timed (bit k = class k, in the order of orc_prof_get) and how densely: every `sample_every`-th
 * launch of a class gets its pair of events (an event pair costs a few microseconds, which matters on 10 us kernels) */
int32_t orc_prof_config(orc_ctx* ctx, uint32_t class_mask, uint32_t sample_every);
int32_t orc_prof_get(orc_ctx* ctx, double* ms, double* bytes, uint64_t* count, int32_t n_classes);
/* the timed launches' bytes counted in the reference's units (a lockstep SpMV = three SpMVs of 12*nnz + 20*n bytes) */
int32_t orc_prof_get_ref_bytes(orc_ctx* ctx, double* bytes, int32_t n_classes);
/* the timed SpMV launches broken down by matrix (rows, entries) and systems per launch (1 or 3): ms, algorithmic bytes, launches */
int32_t orc_prof_get_spmv_detail(orc_ctx* ctx, int32_t cap, int64_t* rows, int64_t* nnz, int32_t* systems, double* ms, double* bytes,
                                 uint64_t* count, int32_t* n_out);
/* Times `reps` launches of the production SpMV kernel on `a` with CUDA events on the context stream; x is device-resident. */
/* device time (best of reps) of one AMG level's setup on `a`: build_restriction and the Galerkin product; optionally returns the coarse matrix */
int32_t orc_bench_amg_setup(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_restriction, double* ms_galerkin, orc_csr** coarse_out);
int32_t orc_bench_spmv(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_per_launch);
/* Times `reps` BiCGSTAB iterations (the 5 fused kernels) on `a`. */
int32_t orc_bench_bicgstab(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_per_iteration);
/* the same for `systems` (1 or 3) right-hand sides in lockstep */
int32_t orc_bench_spmv_batch(orc_ctx* ctx, const orc_csr* a, int32_t systems, int32_t reps, double* ms_per_launch);
int32_t orc_bench_bicgstab_batch(orc_ctx* ctx, const orc_csr* a, int32_t systems, int32_t reps, double* ms_per_iteration);

#ifdef __cplusplus
}
#endif
#endif /* ORC_B200_H */
