// linalg.cuh — device linear algebra of the SIMPLE inner loop (src/linear_algebra.rs of the reference).
#pragma once
#include <memory>

#include "common.cuh"

namespace orc {

using CsrPtr = std::unique_ptr<DCsr>;
struct DistEnv;   // dist.cuh: the communicator and halo plan of a partition

// ---- CSR plumbing ----
CsrPtr csr_alloc(Ctx& c, int64_t nrows, int64_t ncols, int64_t nnz);            // owns pattern + values
CsrPtr csr_like(Ctx& c, const DCsr& a);                                         // shares a's pattern, own values
void csr_ensure_diag(Ctx& c, DCsr& a);                                          // builds a.diag, a.full_diag
void csr_check_symmetry(Ctx& c, DCsr& a);                                       // fills a.sym if unknown

// ---- kernels behind the C ABI ----
// Vectors come as batches of K systems: K = 1 plain, K = 3 interleaved 32-byte cells [x0, x1, x2, 0] (linalg.cu: Cell<K>).
void spmv(Ctx& c, const DCsr& a, const double* x, double* y, int K = 1);        // y = A x, ordered in-row sums
// A' = diag(1/a_ii) A ; b' = diag(1/a_ii) b                                       linear_algebra.rs:157-168
CsrPtr jacobi_scale(Ctx& c, DCsr& a, const double* b, double* b_out, int K = 1);
CsrPtr build_restriction(Ctx& c, DCsr& a, int method, CsrPtr* rt_out);          // linear_algebra.rs:12-63 (+ R^T)
CsrPtr spgemm(Ctx& c, const DCsr& a, const DCsr& b);                            // &Csr * &Csr, symbolic-union pattern
CsrPtr galerkin(Ctx& c, const DCsr& r, const DCsr& rt, const DCsr& a);          // (R*A)*R^T  linear_algebra.rs:84

struct SolveParams {
    uint64_t iterations = 50;
    int method = ORC_SOLVER_MULTIGRID;
    double relaxation = 0.5;
    double threshold = 1e-3;
    int preconditioner = ORC_PC_JACOBI;
    int mg_smoother = ORC_SOLVER_BICGSTAB;
    int mg_levels = 3;
    int gs_mode = ORC_GS_LEXICOGRAPHIC;
    bool exact_order = false;  // reductions in nalgebra's accumulation order (bit-identical solves, small meshes)
};
struct MgTrace {  // keeps R_l, A_l of a Multigrid solve (parity tests) and the level sizes (bench byte model)
    bool keep = false;
    std::vector<CsrPtr> restriction, coarse;
    std::vector<int64_t> rows, nnz;
};
// iterative_solve (linear_algebra.rs:144-299). b, x are device vectors. Errors surface through the device
// flag word (checked by the caller with check_solver_flags) so that the solve never syncs with the host
// except where sizes are data dependent (AMG setup).
// On a partition (env->on()) the matrix is row-partitioned (rows = local cells, halo rows empty; columns local ids incl. halo).
// BiCGSTAB and Jacobi run globally (halo exchange before every SpMV, allreduce for every scalar); Multigrid = global BiCGSTAB
// pre-smoothing + the reference's multigrid_solve applied to THIS rank's diagonal block (partition-local aggregates).
void iterative_solve(Ctx& c, DCsr& a, const double* b, double* x, const SolveParams& sp, MgTrace* trace, int K = 1,
                     const DistEnv* env = nullptr);
bool solve_batchable(const SolveParams& sp);   // can three systems that share the matrix run in lockstep (K = 3)?
void pack3(Ctx& c, int64_t n, const double* a, const double* b, const double* c3, double* out);   // -> cells
void unpack3(Ctx& c, int64_t n, const double* in, double* a, double* b, double* c3);
// device-side bitwise comparison of the value arrays of matrices that share a pattern (syncs)
bool csr_values_identical(Ctx& c, const DCsr& a, const DCsr& b);
// out = &a * sa + &b * sb (nalgebra-sparse operator semantics) for matrices that share one pattern      solver.rs:310-311
void csr_blend(Ctx& c, const DCsr& a, double sa, const DCsr& b, double sb, DCsr& out);
void check_solver_flags(Ctx& c);  // throws the mapped ORC_E_* if a device flag is set, and clears the word
void throw_for_flags(int flags);  // the mapping itself (a status word received from a peer rank)
void bicgstab(Ctx& c, const DCsr& a, const double* b, double* x, uint64_t iterations, int K = 1, const DistEnv* env = nullptr);

// single-launch solvers for small systems (small.cu): the whole BiCGSTAB loop / all Gauss-Seidel sweeps in one block
bool small_enabled();                                                            // ORC_B200_SMALL=0 switches the one-block kernels off
bool small_solve_ok(const Ctx& c, const DCsr& a);                                // reference-order mode and <= ORC_AUTO_EXACT_MAX_ROWS rows
void bicgstab_small(Ctx& c, const DCsr& a, const double* b, double* x, uint64_t iterations);
bool gs_small_ok(const Ctx& c, const DCsr& a, uint64_t sweeps);                  // symmetric pattern, x + flags fit into shared memory
void gauss_seidel_small(Ctx& c, const DCsr& a, const double* b, double* x, double w, double one_minus_w, uint64_t sweeps);

// small device helpers used by the assembly / driver code
void dev_axpy_inplace(Ctx& c, double* y, const double* x, int64_t n);            // y += x
void dev_fill(Ctx& c, double* y, double v, int64_t n);
void dev_scale(Ctx& c, double* y, double s, int64_t n);                          // y *= s
double dev_norm_host(Ctx& c, const double* x, int64_t n);                        // sqrt(sum x^2), syncs

}  // namespace orc
