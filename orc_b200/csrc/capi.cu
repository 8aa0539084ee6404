// capi.cu — the C ABI of liborc_b200 (include/orc_b200.h) and the SIMPLE driver behind it
// (solve_steady, src/solver.rs:26-244 of the reference). Nothing unwinds across the boundary: every
// entry point maps exceptions to a status code and a thread-local message.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>

#include "assembly.cuh"
#include "dist.cuh"
#include "linalg.cuh"
#include "mesh_host.hpp"

using namespace orc;

static thread_local std::string g_err;

struct orc_ctx {
    Ctx c;
    Comm comm;  // multi-GPU: one NCCL communicator per context (inactive on one GPU)
};
struct MeshDevice {   // device side of a mesh on ONE context
    std::unique_ptr<DMesh> d;     // device mirror, created lazily on first use with the context
    std::unique_ptr<Halo> halo;   // device side of the partition plan, built with the mirror
};
struct orc_mesh {
    std::unique_ptr<HostMesh> h;
    std::unique_ptr<PartPlan> plan;  // set on partition meshes (orc_mesh_partition)
    // One mirror PER CONTEXT: steady handles and mesh matrices alias the mirror's pattern arrays, so using the mesh with a second
    // context must not tear down the first one's mirror. Map nodes are address-stable. A mesh must be freed before its contexts.
    std::map<Ctx*, MeshDevice> dev;
    bool zones_checked = false;
    uint64_t checked_epoch = 0;
};
struct orc_csr {
    CsrPtr m;
};

#define ORC_TRY(...)                                                                       \
    try {                                                                                  \
        __VA_ARGS__;                                                                       \
        return ORC_OK;                                                                     \
    } catch (const orc::Error& e) { g_err = e.what(); return e.code;                       \
    } catch (const orc::MeshError& e) { g_err = e.what(); return e.code;                   \
    } catch (const std::bad_alloc&) { g_err = "out of host memory"; return ORC_E_INVALID;  \
    } catch (const std::exception& e) { g_err = e.what(); return ORC_E_INTERNAL; }

static void require(bool ok, const char* msg) {
    if (!ok) throw Error(ORC_E_INVALID, msg);
}

// The BC kinds the path handles (discretization.rs:114-117; solver.rs:1001,1100,1148); a zone typed Interior
// must hold two-cell faces (face.cell_indices[1] would be out of bounds otherwise).
static void check_zones(orc_mesh* m) {
    HostMesh& h = *m->h;
    if (m->zones_checked && m->checked_epoch == h.zone_epoch) return;
    for (auto& z : h.zones) {
        switch (z.type) {
            case ORC_BC_INTERIOR: case ORC_BC_WALL: case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: case ORC_BC_SYMMETRY:
            case ORC_BC_VELOCITY_INLET: break;
            default: throw Error(ORC_E_UNSUPPORTED, "BC not supported: zone '" + z.name + "' has type " + std::to_string(z.type));
        }
    }
    for (int64_t f = 0; f < h.n_faces; ++f)
        if (h.zones[h.face_zone[f]].type == ORC_BC_INTERIOR && h.face_c1[f] < 0)
            throw Error(ORC_E_INVALID, "index out of bounds: face of an Interior zone has one cell");
    m->zones_checked = true;
    m->checked_epoch = h.zone_epoch;
}
static DMesh& device_mesh(Ctx& c, orc_mesh* m) {
    require(m && m->h, "null mesh");
    check_zones(m);
    MeshDevice& md = m->dev[&c];
    if (!md.d) {
        md.d = mesh_upload(c, *m->h);
        if (m->plan) { md.halo.reset(new Halo()); md.halo->build(c, *m->plan); }
    }
    mesh_refresh_zones(c, *md.d, *m->h);
    return *md.d;
}
static AsmSettings asm_settings(const orc_settings* s) {
    AsmSettings a;
    a.momentum = s->momentum; a.limiter = s->limiter; a.p_interp = s->pressure_interpolation; a.v_interp = s->velocity_interpolation;
    a.gradient = s->gradient; a.assembly_mode = s->assembly_mode;
    return a;
}
static bool resolve_exact_order(int reduction_mode, int64_t fine_rows) {
    if (reduction_mode == ORC_REDUCE_AUTO) return fine_rows <= ORC_AUTO_EXACT_MAX_ROWS;
    return reduction_mode == ORC_REDUCE_REFERENCE_ORDER;
}
// `fine_rows`: rows of the system the call solves (ORC_REDUCE_AUTO decides once per call, coarse levels inherit the decision)
static SolveParams solve_params(const orc_settings* s, int64_t fine_rows) {
    SolveParams p;
    p.iterations = s->iterations; p.method = s->solver_type; p.relaxation = s->relaxation; p.threshold = s->threshold;
    p.preconditioner = s->preconditioner; p.mg_smoother = s->mg_smoother; p.mg_levels = s->mg_levels; p.gs_mode = s->gs_mode;
    p.exact_order = resolve_exact_order(s->reduction_mode, fine_rows);
    return p;
}

// =================================================================================================
// the SIMPLE driver: state that solve_steady keeps in locals (solver.rs:41-49), resident on the device
// =================================================================================================
struct orc_steady {
    Ctx* c = nullptr;
    orc_ctx* octx = nullptr;
    DistEnv env;
    orc_mesh* mesh = nullptr;
    DMesh* dm = nullptr;  // the mesh's mirror on this handle's context
    orc_settings s;
    double rho = 0., mu = 0.;
    int64_t N = 0, N_global = 0;  // local vector length (owned + halo) and the global cell count
    CsrPtr a_di, a_u, a_v, a_w, pc_a;
    DBuf<double> b_u_di, b_v_di, b_w_di, b_u, b_v, b_w, pc_b, p_prime, du, dv, dw, u, v, w, p, scal;
    AsmWork work;
    MgTrace trace;  // level sizes of the last Multigrid solve
    uint64_t iteration = 0;
    bool batch_momentum = true;   // ORC_B200_BATCH=0 switches the lockstep u/v/w solve off (A/B runs, tests)
    bool last_batched = false;
    double phase_ms[5] = {0, 0, 0, 0, 0};
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // Boussinesq coupling of the scalar (orc_steady_couple_scalar; sweeps == 0: not coupled) and the resident phi with the buffers
    // of its sweeps, all allocated on first use so that a handle that never uses them carries none
    struct Coupling { double gamma = 0., beta = 0., phi_ref = 0., g[3] = {0., 0., 0.}; uint64_t sweeps = 0; } cpl;
    DBuf<double> phi, phi_b;
    CsrPtr phi_a;
    ScalarWork swork;
    ~orc_steady() {
        for (auto& e : ev) if (e) cudaEventDestroy(e);
    }
};

// The DistEnv of a partition mesh whose device mirror exists on ctx: the plan must match the communicator. With several ranks, all
// of them agree on the peer path (collective) and `work`'s assembly exchanges its halo cells.
static DistEnv partition_env(orc_ctx* ctx, orc_mesh* m, AsmWork* work) {
    Ctx& c = ctx->c;
    require(ctx->comm.nranks == m->plan->nranks && ctx->comm.rank == m->plan->rank, "partition mesh does not match the context's communicator");
    DistEnv env;
    env.comm = &ctx->comm; env.halo = m->dev[&c].halo.get();
    if (env.on()) {
        env.halo->agree_on_peer(c, ctx->comm);
        Comm* cm = env.comm; Halo* hl = env.halo; Ctx* cp = &c;
        if (work) work->halo_exchange = [cm, hl, cp](double* const* f, int n) { hl->exchange(*cp, *cm, f, n); };
    }
    return env;
}
// fills the halo cells of up to Halo::kMaxFields vectors from their owners on a partition; nothing on one GPU
static void exchange(Ctx& c, const DistEnv& env, std::initializer_list<double*> fields) {
    if (!env.on()) return;
    double* f[Halo::kMaxFields]; int k = 0;
    for (double* q : fields) f[k++] = q;
    env.halo->exchange(c, *env.comm, f, k);
}
static double allreduce_host(Ctx& c, Comm& cm, double v, int op) {
    if (!cm.active()) return v;
    DBuf<double> d(&c, 1);
    ORC_CUDA(cudaMemcpyAsync(d.p, &v, sizeof(double), cudaMemcpyHostToDevice, c.stream));
    cm.allreduce(c, d.p, 1, op);
    ORC_CUDA(cudaMemcpyAsync(&v, d.p, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    return v;
}

// The three momentum systems (matrices a, b, c3) are independent (solver.rs:99-136 reads only what the assembly wrote) and, unless the
// scheme is TVD, their matrices are bit-identical (a_nb.x == a_nb.y == a_nb.z, discretization.rs:217-232): solve them in lockstep with
// ONE pass over the matrix and ONE AMG hierarchy. Verified on the device on every call; on a partition every rank must take the same
// branch (the solves contain collectives), so the ranks agree on it (min). ORC_B200_BATCH=0 switches it off (A/B runs, tests).
static bool lockstep_enabled() {
    const char* e = getenv("ORC_B200_BATCH");
    return !(e && atoi(e) == 0);
}
static bool lockstep(Ctx& c, const DistEnv& env, bool enabled, const SolveParams& sp, const DCsr& a, const DCsr& b, const DCsr& c3) {
    if (!solve_batchable(sp)) return false;
    double same = (enabled && csr_values_identical(c, a, b) && csr_values_identical(c, a, c3)) ? 1. : 0.;
    if (env.on()) same = allreduce_host(c, *env.comm, same, 3);
    return same == 1.;
}
// the K = 3 solve of a x_k = b_k, k = u, v, w, on interleaved cells (linalg.cu: Cell<3>)
static void solve_lockstep(Ctx& c, const DistEnv& env, DCsr& a, const double* bu, const double* bv, const double* bw, double* u, double* v,
                           double* w, int64_t N, const SolveParams& sp) {
    DBuf<double> b4(&c, (size_t)std::max<int64_t>(N, 1) * 4), x4(&c, (size_t)std::max<int64_t>(N, 1) * 4);
    pack3(c, N, bu, bv, bw, b4);
    pack3(c, N, u, v, w, x4);
    iterative_solve(c, a, b4, x4, sp, nullptr, 3, &env);
    unpack3(c, N, x4, u, v, w);
}

static orc_steady* steady_create(orc_ctx* octx, orc_mesh* m, const orc_settings* s, double rho, double mu) {
    Ctx& c = octx->c;
    require(s != nullptr, "null settings");
    validate_settings(asm_settings(s));
    DMesh& d = device_mesh(c, m);
    std::unique_ptr<orc_steady> st(new orc_steady());
    st->c = &c; st->octx = octx; st->mesh = m; st->dm = &d; st->s = *s; st->rho = rho; st->mu = mu; st->N = d.N; st->N_global = d.N;
    if (m->plan) {
        st->N_global = m->plan->n_global;
        st->env = partition_env(octx, m, &st->work);
        // Gauss-Seidel's sweep is one dependency chain over all rows: it has no partitioned form
        if (st->env.on())
            require(s->solver_type == ORC_SOLVER_JACOBI || s->solver_type == ORC_SOLVER_BICGSTAB || s->solver_type == ORC_SOLVER_MULTIGRID,
                    "multi-GPU solves support Jacobi, BiCGSTAB and Multigrid");
    }
    const size_t N = (size_t)std::max<int64_t>(d.N, 1);
    for (DBuf<double>* b : {&st->b_u_di, &st->b_v_di, &st->b_w_di, &st->b_u, &st->b_v, &st->b_w, &st->pc_b, &st->p_prime, &st->du, &st->dv,
                            &st->dw, &st->u, &st->v, &st->w, &st->p}) {
        b->alloc(&c, N);
        b->zero();  // halo entries of a partition are never written by the assembly kernels
    }
    st->scal.alloc(&c, 16);
    st->batch_momentum = lockstep_enabled();
    st->a_di = mesh_matrix(c, d); st->a_u = mesh_matrix(c, d); st->a_v = mesh_matrix(c, d); st->a_w = mesh_matrix(c, d); st->pc_a = mesh_matrix(c, d);
    build_momentum_diffusion(c, d, mu, *st->a_di, st->b_u_di, st->b_v_di, st->b_w_di);                  // solver.rs:41-42
    init_momentum_matrix(c, d, *st->a_u); init_momentum_matrix(c, d, *st->a_v); init_momentum_matrix(c, d, *st->a_w);  // :43-45
    dev_fill(c, st->du, 1., d.N); dev_fill(c, st->dv, 1., d.N); dev_fill(c, st->dw, 1., d.N);            // their diagonals
    for (DBuf<double>* b : {&st->b_u, &st->b_v, &st->b_w, &st->p_prime, &st->u, &st->v, &st->w, &st->p}) b->zero();  // :46-49
    for (auto& e : st->ev) ORC_CUDA(cudaEventCreate(&e));
    check_solver_flags(c);
    return st.release();
}

// The status word as a double that survives a SUM allreduce over up to 15 ranks flag by flag: bit b of the word goes to the
// hexadecimal digit b (a plain max over the words would mix the flags of different ranks).
__global__ void k_flags_to_double(const int* flags, double* out) {
    const int f = *flags & ~DF_CONVERGED;
    double v = 0., digit = 1.;
    for (int b = 0; b < 12; ++b, digit *= 16.) if ((f >> b) & 1) v += digit;
    *out = v;
}
static int flags_from_double(double v) {
    unsigned long long w = (unsigned long long)v;
    int f = 0;
    for (int b = 0; b < 12; ++b, w >>= 4) if (w & 15ull) f |= 1 << b;
    return f;
}

// what every scalar entry checks first: phi is determined only with a FIXED boundary zone, and Gamma is a diffusivity
static void require_scalar_problem(const HostMesh& h, double gamma, const AsmSettings& as) {
    validate_scalar_settings(as);
    require(gamma >= 0., "the diffusivity gamma must be >= 0 (and not NaN)");
    bool fixed = false;
    for (const HostZone& z : h.zones) fixed = fixed || (z.type != ORC_BC_INTERIOR && z.scalar_bc_kind == ORC_SBC_FIXED);
    require(fixed, "no boundary zone fixes the scalar: phi is undetermined (orc_mesh_set_zone_scalar with ORC_SBC_FIXED)");
}
// `sweeps` assemble + iterative_solve sweeps of the scalar system from phi = x on the flow u, v, w, p with the diagonals du, dv, dw
// (their halo cells filled); x's halo cells are refreshed before every sweep. a shares the mesh pattern, b has N entries.
static void scalar_sweeps(Ctx& c, const DMesh& d, const DistEnv& env, ScalarWork& work, const AsmSettings& as, const SolveParams& sp,
                          double gamma, double rho, uint64_t sweeps, const double* du, const double* dv, const double* dw, const double* u,
                          const double* v, const double* w, const double* p, DCsr& a, double* b, double* x) {
    scalar_face_flux(c, d, work, as, du, dv, dw, u, v, w, p);
    for (uint64_t k = 0; k < sweeps; ++k) {
        exchange(c, env, {x});                                       // the neighbours' phi for the gradient and the face values
        build_scalar_transport(c, d, work, as, gamma, rho, x, a, b);
        iterative_solve(c, a, b, x, sp, nullptr, 1, &env);
    }
}
// the resident phi (zero) and the buffers of the coupled sweeps, on first use
static void ensure_scalar(orc_steady& st) {
    if (st.phi.p) return;
    Ctx& c = *st.c;
    const size_t N = (size_t)std::max<int64_t>(st.N, 1);
    st.phi.alloc(&c, N); st.phi.zero();
    st.phi_b.alloc(&c, N); st.phi_b.zero();
    st.phi_a = mesh_matrix(c, *st.dm);
    st.swork.halo_exchange = st.work.halo_exchange;
}

static void steady_iterate(orc_steady& st, uint64_t iterations, uint64_t report_every, orc_report_cb cb, void* user, orc_report* last) {
    Ctx& c = *st.c;
    DMesh& d = device_mesh(c, st.mesh);
    const AsmSettings as = asm_settings(&st.s);
    // multi-GPU solves always use the fused reductions (ORC_REDUCE_AUTO never picks the single-GPU reference-order kernels there)
    const SolveParams sp = solve_params(&st.s, st.env.on() ? INT64_MAX : st.N_global);
    const int64_t N = st.N;
    const bool coupled = st.cpl.sweeps > 0;
    if (coupled) require_scalar_problem(*st.mesh->h, st.cpl.gamma, as);   // the zones' scalar conditions may have changed since
    cudaEvent_t t_report;
    ORC_CUDA(cudaEventCreate(&t_report));
    struct EvGuard { cudaEvent_t e; ~EvGuard() { cudaEventDestroy(e); } } guard{t_report};
    ORC_CUDA(cudaEventRecord(t_report, c.stream));
    for (uint64_t k = 0; k < iterations; ++k) {
        const uint64_t iter_number = ++st.iteration;
        ORC_CUDA(cudaEventRecord(st.ev[0], c.stream));
        const bool dist = st.env.on();
        exchange(c, st.env, {st.u.p, st.v.p, st.w.p, st.p.p});                                              // C1: neighbours' fields
        int pid = c.prof_begin(PC_ASSEMBLY, 0.);
        build_momentum_advection(c, d, st.work, as, st.rho, *st.a_u, *st.a_v, *st.a_w, *st.a_di, st.du, st.dv, st.dw, st.u, st.v, st.w, st.p,
                                 st.b_u, st.b_v, st.b_w, st.scal.p + 8);                                   // solver.rs:61-79
        if (coupled) {  // b + b_di + the body force of phi as it stood when the iteration started (DESIGN.md §1)
            momentum_source_buoyancy(c, d, st.b_u, st.b_v, st.b_w, st.b_u_di, st.b_v_di, st.b_w_di, st.phi, st.rho * st.cpl.beta, st.cpl.phi_ref,
                                     st.cpl.g);
        } else {
            dev_axpy_inplace(c, st.b_u, st.b_u_di, N); dev_axpy_inplace(c, st.b_v, st.b_v_di, N); dev_axpy_inplace(c, st.b_w, st.b_w_di, N);  // :80-82
        }
        c.prof_end(pid);
        exchange(c, st.env, {st.du.p, st.dv.p, st.dw.p});  // new diagonals for the pressure system; the "old" state of the next assembly (C4)
        ORC_CUDA(cudaEventRecord(st.ev[1], c.stream));
        st.last_batched = lockstep(c, st.env, st.batch_momentum, sp, *st.a_u, *st.a_v, *st.a_w);
        if (st.last_batched) {
            solve_lockstep(c, st.env, *st.a_u, st.b_u, st.b_v, st.b_w, st.u, st.v, st.w, N, sp);
        } else {
            iterative_solve(c, *st.a_u, st.b_u, st.u, sp, nullptr, 1, &st.env);                            // :99-110
            iterative_solve(c, *st.a_v, st.b_v, st.v, sp, nullptr, 1, &st.env);                            // :112-123
            iterative_solve(c, *st.a_w, st.b_w, st.w, sp, nullptr, 1, &st.env);                            // :125-136
        }
        exchange(c, st.env, {st.u.p, st.v.p, st.w.p});
        ORC_CUDA(cudaEventRecord(st.ev[2], c.stream));
        pid = c.prof_begin(PC_ASSEMBLY, 0.);
        build_pressure_correction(c, d, st.work, as, st.rho, st.du, st.dv, st.dw, st.u, st.v, st.w, st.p, *st.pc_a, st.pc_b);  // :137-148
        c.prof_end(pid);
        ORC_CUDA(cudaEventRecord(st.ev[3], c.stream));
        dev_scale(c, st.p_prime, 0., N);                                                                   // p_prime *= 0.  (:167)
        iterative_solve(c, *st.pc_a, st.pc_b, st.p_prime, sp, &st.trace, 1, &st.env);                     // :168-179
        exchange(c, st.env, {st.p_prime.p});
        ORC_CUDA(cudaEventRecord(st.ev[4], c.stream));
        apply_pressure_correction(c, d, st.du, st.dv, st.dw, st.p_prime, st.u, st.v, st.w, st.p, st.s.pressure_relaxation,
                                  st.s.momentum_relaxation, st.scal.p);                                    // :193-204
        if (coupled) {  // the scalar sweeps on the corrected flow and this iteration's diagonals (counted in the correction phase)
            exchange(c, st.env, {st.u.p, st.v.p, st.w.p, st.p.p});
            scalar_sweeps(c, d, st.env, st.swork, as, sp, st.cpl.gamma, st.rho, st.cpl.sweeps, st.du, st.dv, st.dw, st.u, st.v, st.w, st.p,
                          *st.phi_a, st.phi_b, st.phi);
        }
        ORC_CUDA(cudaEventRecord(st.ev[5], c.stream));
        if (dist) {  // C2: iteration scalars; the status word travels along so that every rank takes the same exit
            Comm& cm = *st.env.comm;
            k_flags_to_double<<<1, 1, 0, c.stream>>>(c.d_flags, st.scal.p + 5);
            c.after_launch("k_flags_to_double");
            cm.allreduce(c, st.scal.p, 5, 0);        // sum p'^2, sum |du|^2, sum u, sum v, sum w
            cm.allreduce(c, st.scal.p + 5, 1, 0);    // the status words, one hexadecimal digit per flag
            cm.allreduce(c, st.scal.p + 8, 1, 0);    // Peclet: sum of cell means
            cm.allreduce(c, st.scal.p + 9, 1, 3);    // min
            cm.allreduce(c, st.scal.p + 10, 1, 2);   // max
        }
        double h[16];
        ORC_CUDA(cudaMemcpyAsync(h, st.scal.p, sizeof(double) * 16, cudaMemcpyDeviceToHost, c.stream));
        if (dist) {
            c.sync();
            int local = c.read_flags();
            if (local == 0 && h[5] != 0.) {
                c.clear_flags();
                throw_for_flags(flags_from_double(h[5]));   // another rank failed: fail with the same error
            }
        }
        check_solver_flags(c);  // synchronises
        c.prof_resolve();
        for (int q = 0; q < 5; ++q) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, st.ev[q], st.ev[q + 1]);
            st.phase_ms[q] += ms;
        }
        const double Ng = (double)st.N_global;
        const double u_avg = h[2] / Ng, v_avg = h[3] / Ng, w_avg = h[4] / Ng;                               // :206-208
        orc_report rep;
        rep.iteration = iter_number; rep.u_avg = u_avg; rep.v_avg = v_avg; rep.w_avg = w_avg;
        rep.peclet_avg = h[8] / Ng; rep.peclet_min = h[9]; rep.peclet_max = h[10];
        rep.velocity_correction = sqrt(h[1]); rep.pressure_correction = sqrt(h[0]); rep.ms_per_iter = 0.;
        if (report_every != 0 && iter_number % report_every == 0) {                                         // :209-216
            float ms = 0.f;
            cudaEventElapsedTime(&ms, t_report, st.ev[5]);
            rep.ms_per_iter = ms / (double)report_every;
            ORC_CUDA(cudaEventRecord(t_report, c.stream));
            if (cb) cb(&rep, user);
        }
        if (last) *last = rep;
        if (u_avg != u_avg || v_avg != v_avg || w_avg != w_avg) throw Error(ORC_E_DIVERGED, "solution diverged");  // :217-221
    }
}

// =================================================================================================
extern "C" {

const char* orc_last_error(void) { return g_err.c_str(); }
const char* orc_version(void) { return "orc_b200 0.1 (sm_100a, fp64)"; }

void orc_settings_default(orc_settings* s) {
    if (!s) return;
    memset(s, 0, sizeof(*s));
    s->momentum = ORC_MOM_CD1; s->limiter = ORC_PSI_QUICK; s->pressure_interpolation = ORC_P_SECOND_ORDER;
    s->velocity_interpolation = ORC_V_RHIE_CHOW; s->gradient = ORC_G_GREEN_GAUSS_CELL; s->solver_type = ORC_SOLVER_MULTIGRID;
    s->preconditioner = ORC_PC_JACOBI; s->mg_smoother = ORC_SOLVER_BICGSTAB; s->mg_levels = 3; s->gs_mode = ORC_GS_LEXICOGRAPHIC;
    s->assembly_mode = ORC_ASSEMBLY_EXACT; s->reduction_mode = ORC_REDUCE_AUTO; s->iterations = 50; s->pressure_relaxation = 0.01; s->momentum_relaxation = 0.5;
    s->relaxation = 0.5; s->threshold = 1e-3;
}

int32_t orc_ctx_create(int32_t device, void* stream, orc_ctx** out) {
    ORC_TRY({
        require(out != nullptr, "null out");
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error(ORC_E_CUDA, std::string("no CUDA device: liborc_b200 has no CPU fallback (") + cudaGetErrorString(e) + ")");
        require(device >= 0 && device < ndev, "device index out of range");
        ORC_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        ORC_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) throw Error(ORC_E_CUDA, std::string("device '") + prop.name + "' is not sm_100-class; this library ships sm_100a code only");
        std::unique_ptr<orc_ctx> ctx(new orc_ctx());
        Ctx& c = ctx->c;
        c.device = device;
        c.sm_count = prop.multiProcessorCount;
        if (stream) { c.stream = (cudaStream_t)stream; c.own_stream = false; }
        else { ORC_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking)); c.own_stream = true; }
        ORC_CUDA(cudaMalloc(&c.d_flags, sizeof(int)));
        ORC_CUDA(cudaMalloc(&c.d_scal, sizeof(double) * 64));
        ORC_CUDA(cudaMalloc(&c.d_partials, sizeof(double) * Ctx::kPartialLanes * Ctx::kMaxBlocks));
        ORC_CUDA(cudaMalloc(&c.d_counter, sizeof(unsigned int) * 4));
        ORC_CUDA(cudaMemsetAsync(c.d_flags, 0, sizeof(int), c.stream));
        ORC_CUDA(cudaMemsetAsync(c.d_scal, 0, sizeof(double) * 64, c.stream));
        ORC_CUDA(cudaMemsetAsync(c.d_counter, 0, sizeof(unsigned int) * 4, c.stream));
        c.sync();
        *out = ctx.release();
    });
}
void orc_ctx_destroy(orc_ctx* ctx) {
    if (!ctx) return;
    Ctx& c = ctx->c;
    cudaStreamSynchronize(c.stream);
    c.cache_release_all();
    for (auto& kv : c.cache_live) cudaFree(kv.first);
    cudaFree(c.d_flags); cudaFree(c.d_scal); cudaFree(c.d_partials); cudaFree(c.d_counter);
    if (c.own_stream) cudaStreamDestroy(c.stream);
    ctx->comm.destroy();
    delete ctx;
}
uint64_t orc_ctx_launch_count(orc_ctx* ctx) { return ctx ? ctx->c.launches : 0; }
int32_t orc_ctx_synchronize(orc_ctx* ctx) { ORC_TRY({ require(ctx, "null ctx"); ctx->c.sync(); }); }

// ---- mesh ------------------------------------------------------------------------------------------
int32_t orc_mesh_read(const char* path, orc_mesh** out) {
    ORC_TRY({
        require(path && out, "null argument");
        std::unique_ptr<orc_mesh> m(new orc_mesh());
        m->h.reset(read_tgrid(path));
        *out = m.release();
    });
}
int32_t orc_mesh_from_arrays(int32_t dimensions, int64_t n_nodes, const double* xyz, int64_t n_faces, const int64_t* face_node_offsets,
                             const int64_t* face_nodes, const int64_t* c0, const int64_t* c1, const int64_t* face_zone, int64_t n_zones,
                             const int64_t* zone_ids, const int64_t* zone_types, const char* const* zone_names, orc_mesh** out) {
    ORC_TRY({
        require(xyz && face_node_offsets && face_nodes && c0 && c1 && face_zone && zone_ids && zone_types && zone_names && out, "null argument");
        std::unique_ptr<orc_mesh> m(new orc_mesh());
        m->h.reset(mesh_from_arrays(dimensions, n_nodes, xyz, n_faces, face_node_offsets, face_nodes, c0, c1, face_zone, n_zones, zone_ids,
                                    zone_types, zone_names));
        *out = m.release();
    });
}
int32_t orc_mesh_from_geometry(int32_t dimensions, int64_t n_cells, int64_t n_faces, const int64_t* face_c0, const int64_t* face_c1,
                               const int64_t* face_zone, const double* face_area, const double* face_normal3, const double* face_centroid3,
                               const double* cell_volume, const double* cell_centroid3, const int64_t* cell_face_offsets,
                               const int64_t* cell_face_indices, int64_t n_zones, const int64_t* zone_ids, const int64_t* zone_types,
                               const char* const* zone_names, orc_mesh** out) {
    ORC_TRY({
        require(face_c0 && face_c1 && face_zone && face_area && face_normal3 && face_centroid3 && cell_volume && cell_centroid3 &&
                    cell_face_offsets && cell_face_indices && zone_ids && zone_types && zone_names && out, "null argument");
        std::unique_ptr<orc_mesh> m(new orc_mesh());
        m->h.reset(mesh_from_geometry(dimensions, n_cells, n_faces, face_c0, face_c1, face_zone, face_area, face_normal3, face_centroid3,
                                      cell_volume, cell_centroid3, cell_face_offsets, cell_face_indices, n_zones, zone_ids, zone_types,
                                      zone_names));
        *out = m.release();
    });
}
void orc_mesh_free(orc_mesh* m) {
    if (!m) return;
    for (auto& kv : m->dev) cudaStreamSynchronize(kv.first->stream);
    delete m;
}
int32_t orc_mesh_counts(const orc_mesh* m, int64_t* out8) {
    ORC_TRY({
        require(m && out8, "null argument");
        const HostMesh& h = *m->h;
        out8[0] = h.n_cells; out8[1] = h.n_faces; out8[2] = h.n_nodes; out8[3] = (int64_t)h.zones.size(); out8[4] = (int64_t)h.cf_face.size();
        out8[5] = h.dims; out8[6] = h.nnz(); out8[7] = (int64_t)h.level_ptr.size() - 1;
    });
}
int32_t orc_mesh_export(const orc_mesh* m, int64_t* face_c0, int64_t* face_c1, int64_t* face_zone, double* face_area, double* face_normal3,
                        double* face_centroid3, double* cell_volume, double* cell_centroid3, int64_t* cell_face_offsets,
                        int64_t* cell_face_indices) {
    ORC_TRY({
        require(m != nullptr, "null mesh");
        const HostMesh& h = *m->h;
        for (int64_t f = 0; f < h.n_faces; ++f) {
            face_c0[f] = h.face_c0[f]; face_c1[f] = h.face_c1[f]; face_zone[f] = h.zones[h.face_zone[f]].id; face_area[f] = h.face_area[f];
        }
        memcpy(face_normal3, h.face_normal.data(), sizeof(double) * 3 * h.n_faces);
        memcpy(face_centroid3, h.face_centroid.data(), sizeof(double) * 3 * h.n_faces);
        memcpy(cell_volume, h.cell_volume.data(), sizeof(double) * h.n_cells);
        memcpy(cell_centroid3, h.cell_centroid.data(), sizeof(double) * 3 * h.n_cells);
        for (int64_t c = 0; c <= h.n_cells; ++c) cell_face_offsets[c] = h.cf_ptr[c];
        for (size_t q = 0; q < h.cf_face.size(); ++q) cell_face_indices[q] = h.cf_face[q];
    });
}
int32_t orc_mesh_geometry_device(orc_ctx* ctx, const orc_mesh* m, double* face_area, double* face_normal3, double* face_centroid3,
                                 double* cell_volume, double* cell_centroid3, double* device_ms) {
    ORC_TRY({
        require(ctx && m && m->h && face_area && face_normal3 && face_centroid3 && cell_volume && cell_centroid3, "null argument");
        mesh_geometry_device(ctx->c, *m->h, face_area, face_normal3, face_centroid3, cell_volume, cell_centroid3, device_ms);
    });
}
int32_t orc_mesh_zones(const orc_mesh* m, int64_t* ids, int64_t* types, double* scalar, double* vector3, char* names64) {
    ORC_TRY({
        require(m != nullptr, "null mesh");
        const HostMesh& h = *m->h;
        for (size_t k = 0; k < h.zones.size(); ++k) {
            ids[k] = h.zones[k].id; types[k] = h.zones[k].type; scalar[k] = h.zones[k].scalar;
            for (int q = 0; q < 3; ++q) vector3[3 * k + q] = h.zones[k].vec[q];
            memset(names64 + 64 * k, 0, 64);
            strncpy(names64 + 64 * k, h.zones[k].name.c_str(), 63);
        }
    });
}
int32_t orc_mesh_set_zone(orc_mesh* m, const char* name, int64_t zone_type, double scalar, double vx, double vy, double vz) {
    ORC_TRY({
        require(m && name, "null argument");
        int k = m->h->find_zone(name);
        if (k < 0) throw Error(ORC_E_INVALID, std::string("face zone '") + name + "' should exist in mesh");  // mesh.rs:189-195
        HostZone& z = m->h->zones[k];
        z.type = (int32_t)zone_type; z.scalar = scalar; z.vec[0] = vx; z.vec[1] = vy; z.vec[2] = vz;
        m->h->zone_epoch++;
    });
}
int32_t orc_mesh_pattern(const orc_mesh* m, int64_t* rowptr, int64_t* col) {
    ORC_TRY({
        require(m && rowptr && col, "null argument");
        const HostMesh& h = *m->h;
        for (int64_t i = 0; i <= h.n_cells; ++i) rowptr[i] = h.rowptr[i];
        for (int64_t k = 0; k < h.nnz(); ++k) col[k] = h.col[k];
    });
}
int32_t orc_mesh_levels(const orc_mesh* m, int64_t* level_of_cell) {
    ORC_TRY({
        require(m && level_of_cell, "null argument");
        for (int64_t i = 0; i < m->h->n_cells; ++i) level_of_cell[i] = m->h->level_of_cell[i];
    });
}

// ---- CSR handles ---------------------------------------------------------------------------------------
int32_t orc_csr_upload(orc_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* rowptr, const int64_t* col, const double* val,
                       orc_csr** out) {
    ORC_TRY({
        require(ctx && rowptr && out, "null argument");
        require(nrows >= 0 && ncols >= 0 && rowptr[0] == 0, "bad CSR dimensions");
        const int64_t nnz = rowptr[nrows];
        require(nnz <= INT32_MAX && nrows < INT32_MAX && ncols < INT32_MAX, "matrix exceeds 32-bit indexing");
        std::vector<int> rp((size_t)nrows + 1), cl((size_t)std::max<int64_t>(nnz, 1));
        for (int64_t i = 0; i <= nrows; ++i) { require(i == 0 || rowptr[i] >= rowptr[i - 1], "rowptr must be non-decreasing"); rp[i] = (int)rowptr[i]; }
        for (int64_t i = 0; i < nrows; ++i)
            for (int64_t k = rowptr[i]; k < rowptr[i + 1]; ++k) {
                require(col[k] >= 0 && col[k] < ncols, "column index out of range");
                require(k == rowptr[i] || col[k] > col[k - 1], "columns must be sorted and unique within a row");
                cl[k] = (int)col[k];
            }
        Ctx& c = ctx->c;
        CsrPtr a = csr_alloc(c, nrows, ncols, nnz);
        ORC_CUDA(cudaMemcpyAsync(a->rowptr, rp.data(), sizeof(int) * rp.size(), cudaMemcpyHostToDevice, c.stream));
        if (nnz > 0) {
            ORC_CUDA(cudaMemcpyAsync(a->col, cl.data(), sizeof(int) * nnz, cudaMemcpyHostToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(a->val, val, sizeof(double) * nnz, cudaMemcpyHostToDevice, c.stream));
        }
        c.sync();
        std::unique_ptr<orc_csr> h(new orc_csr());
        h->m = std::move(a);
        *out = h.release();
    });
}
int32_t orc_csr_dims(const orc_csr* a, int64_t* out3) {
    ORC_TRY({ require(a && out3, "null argument"); out3[0] = a->m->nrows; out3[1] = a->m->ncols; out3[2] = a->m->nnz; });
}
int32_t orc_csr_download(orc_ctx* ctx, const orc_csr* a, int64_t* rowptr, int64_t* col, double* val) {
    ORC_TRY({
        require(ctx && a, "null argument");
        Ctx& c = ctx->c;
        const DCsr& m = *a->m;
        std::vector<int> rp((size_t)m.nrows + 1), cl((size_t)std::max<int64_t>(m.nnz, 1));
        ORC_CUDA(cudaMemcpyAsync(rp.data(), m.rowptr, sizeof(int) * rp.size(), cudaMemcpyDeviceToHost, c.stream));
        if (m.nnz > 0) {
            ORC_CUDA(cudaMemcpyAsync(cl.data(), m.col, sizeof(int) * m.nnz, cudaMemcpyDeviceToHost, c.stream));
            if (val) ORC_CUDA(cudaMemcpyAsync(val, m.val, sizeof(double) * m.nnz, cudaMemcpyDeviceToHost, c.stream));
        }
        c.sync();
        if (rowptr) for (int64_t i = 0; i <= m.nrows; ++i) rowptr[i] = rp[i];
        if (col) for (int64_t k = 0; k < m.nnz; ++k) col[k] = cl[k];
    });
}
int32_t orc_csr_set_values(orc_ctx* ctx, orc_csr* a, const double* val) {
    ORC_TRY({
        require(ctx && a && val, "null argument");
        if (a->m->nnz > 0) ORC_CUDA(cudaMemcpyAsync(a->m->val, val, sizeof(double) * a->m->nnz, cudaMemcpyHostToDevice, ctx->c.stream));
        ctx->c.sync();
    });
}
void orc_csr_free(orc_ctx* ctx, orc_csr* a) {
    if (!a) return;
    if (ctx) cudaStreamSynchronize(ctx->c.stream);
    delete a;
}

// host vector <-> device helpers
struct HostVecIn {
    DBuf<double> d;
    HostVecIn(Ctx& c, const double* h, int64_t n) : d(&c, (size_t)std::max<int64_t>(n, 1)) {
        if (n > 0) ORC_CUDA(cudaMemcpyAsync(d.p, h, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
    }
};
static void to_host(Ctx& c, double* h, const double* d, int64_t n) {
    if (n > 0) ORC_CUDA(cudaMemcpyAsync(h, d, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
}

int32_t orc_spmv(orc_ctx* ctx, const orc_csr* a, const double* x, double* y) {
    ORC_TRY({
        require(ctx && a && x && y, "null argument");
        Ctx& c = ctx->c;
        c.exact_order = false;   // the fast kernels, whatever reduction mode the last solve on this context used
        HostVecIn dx(c, x, a->m->ncols);
        DBuf<double> dy(&c, (size_t)std::max<int64_t>(a->m->nrows, 1));
        spmv(c, *a->m, dx.d, dy);
        to_host(c, y, dy, a->m->nrows);
        c.sync();
    });
}
int32_t orc_jacobi_scale(orc_ctx* ctx, const orc_csr* a, const double* b, orc_csr** a_out, double* b_out) {
    ORC_TRY({
        require(ctx && a && b && a_out && b_out, "null argument");
        Ctx& c = ctx->c;
        HostVecIn db(c, b, a->m->nrows);
        DBuf<double> dbo(&c, (size_t)std::max<int64_t>(a->m->nrows, 1));
        CsrPtr s = jacobi_scale(c, *a->m, db.d, dbo);
        if (!s->own_pattern) {  // detach from the input's pattern so that the handle can outlive it
            CsrPtr own = csr_alloc(c, s->nrows, s->ncols, s->nnz);
            ORC_CUDA(cudaMemcpyAsync(own->rowptr, s->rowptr, sizeof(int) * (s->nrows + 1), cudaMemcpyDeviceToDevice, c.stream));
            if (s->nnz > 0) {
                ORC_CUDA(cudaMemcpyAsync(own->col, s->col, sizeof(int) * s->nnz, cudaMemcpyDeviceToDevice, c.stream));
                ORC_CUDA(cudaMemcpyAsync(own->val, s->val, sizeof(double) * s->nnz, cudaMemcpyDeviceToDevice, c.stream));
            }
            s = std::move(own);
        }
        to_host(c, b_out, dbo, a->m->nrows);
        c.sync();
        std::unique_ptr<orc_csr> h(new orc_csr());
        h->m = std::move(s);
        *a_out = h.release();
    });
}

// ---- linear_algebra.rs ---------------------------------------------------------------------------------
int32_t orc_iterative_solve(orc_ctx* ctx, const orc_csr* a, const double* b, double* x, const orc_settings* s) {
    ORC_TRY({
        require(ctx && a && b && x && s, "null argument");
        Ctx& c = ctx->c;
        const int64_t n = a->m->nrows;
        HostVecIn db(c, b, n), dx(c, x, a->m->ncols);
        c.clear_flags();
        iterative_solve(c, *a->m, db.d, dx.d, solve_params(s, n), nullptr);
        to_host(c, x, dx.d, a->m->ncols);
        check_solver_flags(c);
    });
}
int32_t orc_iterative_solve3(orc_ctx* ctx, const orc_csr* a, const double* b0, const double* b1, const double* b2, double* x0, double* x1,
                             double* x2, const orc_settings* s) {
    ORC_TRY({
        require(ctx && a && b0 && b1 && b2 && x0 && x1 && x2 && s, "null argument");
        Ctx& c = ctx->c;
        const int64_t n = a->m->nrows;
        require(a->m->ncols == n, "iterative_solve: matrix must be square");
        HostVecIn db0(c, b0, n), db1(c, b1, n), db2(c, b2, n), dx0(c, x0, n), dx1(c, x1, n), dx2(c, x2, n);
        DBuf<double> b4(&c, (size_t)std::max<int64_t>(n, 1) * 4), x4(&c, (size_t)std::max<int64_t>(n, 1) * 4);
        pack3(c, n, db0.d, db1.d, db2.d, b4);
        pack3(c, n, dx0.d, dx1.d, dx2.d, x4);
        c.clear_flags();
        iterative_solve(c, *a->m, b4, x4, solve_params(s, n), nullptr, 3);
        unpack3(c, n, x4, dx0.d, dx1.d, dx2.d);
        to_host(c, x0, dx0.d, n); to_host(c, x1, dx1.d, n); to_host(c, x2, dx2.d, n);
        check_solver_flags(c);
    });
}
int32_t orc_build_restriction(orc_ctx* ctx, const orc_csr* a, int32_t method, orc_csr** r_out) {
    ORC_TRY({
        require(ctx && a && r_out, "null argument");
        Ctx& c = ctx->c;
        c.clear_flags();
        CsrPtr r = build_restriction(c, *a->m, method, nullptr);
        check_solver_flags(c);
        std::unique_ptr<orc_csr> h(new orc_csr());
        h->m = std::move(r);
        *r_out = h.release();
    });
}
int32_t orc_galerkin(orc_ctx* ctx, const orc_csr* r, const orc_csr* a, orc_csr** out) {
    ORC_TRY({
        require(ctx && r && a && out, "null argument");
        Ctx& c = ctx->c;
        // explicit transpose of an arbitrary R: build it through the generic path (host, off the hot path)
        const DCsr& R = *r->m;
        std::vector<int> rp((size_t)R.nrows + 1), cl((size_t)std::max<int64_t>(R.nnz, 1));
        std::vector<double> vl((size_t)std::max<int64_t>(R.nnz, 1));
        ORC_CUDA(cudaMemcpyAsync(rp.data(), R.rowptr, sizeof(int) * rp.size(), cudaMemcpyDeviceToHost, c.stream));
        if (R.nnz > 0) {
            ORC_CUDA(cudaMemcpyAsync(cl.data(), R.col, sizeof(int) * R.nnz, cudaMemcpyDeviceToHost, c.stream));
            ORC_CUDA(cudaMemcpyAsync(vl.data(), R.val, sizeof(double) * R.nnz, cudaMemcpyDeviceToHost, c.stream));
        }
        c.sync();
        std::vector<int> trp((size_t)R.ncols + 1, 0), tcl((size_t)std::max<int64_t>(R.nnz, 1));
        std::vector<double> tvl((size_t)std::max<int64_t>(R.nnz, 1));
        for (int64_t k = 0; k < R.nnz; ++k) trp[cl[k] + 1]++;
        for (int64_t j = 0; j < R.ncols; ++j) trp[j + 1] += trp[j];
        std::vector<int> pos(trp.begin(), trp.end() - 1);
        for (int64_t i = 0; i < R.nrows; ++i)
            for (int k = rp[i]; k < rp[i + 1]; ++k) { int q = pos[cl[k]]++; tcl[q] = (int)i; tvl[q] = vl[k]; }
        CsrPtr RT = csr_alloc(c, R.ncols, R.nrows, R.nnz);
        ORC_CUDA(cudaMemcpyAsync(RT->rowptr, trp.data(), sizeof(int) * trp.size(), cudaMemcpyHostToDevice, c.stream));
        if (R.nnz > 0) {
            ORC_CUDA(cudaMemcpyAsync(RT->col, tcl.data(), sizeof(int) * R.nnz, cudaMemcpyHostToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(RT->val, tvl.data(), sizeof(double) * R.nnz, cudaMemcpyHostToDevice, c.stream));
        }
        c.sync();
        CsrPtr ac = galerkin(c, R, *RT, *a->m);
        c.sync();
        std::unique_ptr<orc_csr> h(new orc_csr());
        h->m = std::move(ac);
        *out = h.release();
    });
}
int32_t orc_multigrid_trace(orc_ctx* ctx, const orc_csr* a, const double* b, double* x, const orc_settings* s, int32_t max_out,
                            orc_csr** r_levels, orc_csr** a_levels, int32_t* n_levels) {
    ORC_TRY({
        require(ctx && a && b && x && s && n_levels, "null argument");
        Ctx& c = ctx->c;
        HostVecIn db(c, b, a->m->nrows), dx(c, x, a->m->ncols);
        SolveParams sp = solve_params(s, a->m->nrows);
        sp.method = ORC_SOLVER_MULTIGRID;
        MgTrace tr;
        tr.keep = true;
        c.clear_flags();
        iterative_solve(c, *a->m, db.d, dx.d, sp, &tr);
        to_host(c, x, dx.d, a->m->ncols);
        check_solver_flags(c);
        *n_levels = (int32_t)tr.restriction.size();
        for (int l = 0; l < (int)tr.restriction.size() && l < max_out; ++l) {
            if (r_levels) { r_levels[l] = new orc_csr(); r_levels[l]->m = std::move(tr.restriction[l]); }
            if (a_levels) { a_levels[l] = new orc_csr(); a_levels[l]->m = std::move(tr.coarse[l]); }
        }
    });
}

// ---- discretization.rs -----------------------------------------------------------------------------------
static orc_csr* wrap(CsrPtr m) {
    orc_csr* h = new orc_csr();
    h->m = std::move(m);
    return h;
}
// a handle that shares the mesh's pattern must not outlive the mesh: detach it.
static CsrPtr detach(Ctx& c, CsrPtr s) {
    if (s->own_pattern) return s;
    CsrPtr own = csr_alloc(c, s->nrows, s->ncols, s->nnz);
    ORC_CUDA(cudaMemcpyAsync(own->rowptr, s->rowptr, sizeof(int) * (s->nrows + 1), cudaMemcpyDeviceToDevice, c.stream));
    if (s->nnz > 0) {
        ORC_CUDA(cudaMemcpyAsync(own->col, s->col, sizeof(int) * s->nnz, cudaMemcpyDeviceToDevice, c.stream));
        ORC_CUDA(cudaMemcpyAsync(own->val, s->val, sizeof(double) * s->nnz, cudaMemcpyDeviceToDevice, c.stream));
    }
    own->sym = s->sym; own->max_row = s->max_row; own->simplex = s->simplex;
    if (s->hint.on() && s->hint.shift == 0) {   // keep the positions of the unknowns: the handle owns a copy of the three planes
        const size_t n = (size_t)s->hint.n;
        own->hint = s->hint;
        own->hint_own = c.alloc_n<double>(3 * n);
        ORC_CUDA(cudaMemcpyAsync(own->hint_own, s->hint.x, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
        ORC_CUDA(cudaMemcpyAsync(own->hint_own + n, s->hint.y, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
        ORC_CUDA(cudaMemcpyAsync(own->hint_own + 2 * n, s->hint.z, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
        own->hint.x = own->hint_own; own->hint.y = own->hint_own + n; own->hint.z = own->hint_own + 2 * n;
    }
    c.sync();
    return own;
}

int32_t orc_build_momentum_diffusion(orc_ctx* ctx, orc_mesh* m, double mu, orc_csr** a_di, double* b_u, double* b_v, double* b_w) {
    ORC_TRY({
        require(ctx && m && a_di && b_u && b_v && b_w, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        CsrPtr a = mesh_matrix(c, d);
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        DBuf<double> bu(&c, N), bv(&c, N), bw(&c, N);
        c.clear_flags();
        build_momentum_diffusion(c, d, mu, *a, bu, bv, bw);
        to_host(c, b_u, bu, d.N); to_host(c, b_v, bv, d.N); to_host(c, b_w, bw, d.N);
        check_solver_flags(c);
        *a_di = wrap(detach(c, std::move(a)));
    });
}
int32_t orc_init_momentum_matrix(orc_ctx* ctx, orc_mesh* m, orc_csr** out) {
    ORC_TRY({
        require(ctx && m && out, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        CsrPtr a = mesh_matrix(c, d);
        init_momentum_matrix(c, d, *a);
        c.sync();
        *out = wrap(detach(c, std::move(a)));
    });
}
static void require_mesh_matrix(const DMesh& d, const orc_csr* a, const char* what) {
    if (!a || a->m->nrows != d.N || a->m->nnz != d.nnz) throw Error(ORC_E_INVALID, std::string(what) + ": matrix does not have the mesh pattern");
}
// the diagonals of three matrices with the mesh pattern (a_u.get(i, i) in the reference), read through the mesh's diagonal index
static void momentum_diagonals(Ctx& c, const DMesh& d, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w, double* du, double* dv,
                               double* dw) {
    const orc_csr* mats[3] = {a_u, a_v, a_w};
    double* diags[3] = {du, dv, dw};
    for (int q = 0; q < 3; ++q) {
        DCsr& A = *const_cast<orc_csr*>(mats[q])->m;
        int* keep = A.diag; bool own = A.own_diag;
        A.diag = d.diag.p; A.own_diag = false;
        extract_diagonal(c, A, diags[q]);
        A.diag = keep; A.own_diag = own;
    }
}
int32_t orc_build_momentum_advection(orc_ctx* ctx, orc_mesh* m, orc_csr* a_u, orc_csr* a_v, orc_csr* a_w, const orc_csr* a_di,
                                     const double* u, const double* v, const double* w, const double* p, const orc_settings* s,
                                     double rho, double* b_u, double* b_v, double* b_w, double* peclet3) {
    ORC_TRY({
        require(ctx && m && u && v && w && p && s && b_u && b_v && b_w, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        require_mesh_matrix(d, a_u, "a_u"); require_mesh_matrix(d, a_v, "a_v"); require_mesh_matrix(d, a_w, "a_w"); require_mesh_matrix(d, a_di, "a_di");
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn du_(c, u, d.N), dv_(c, v, d.N), dw_(c, w, d.N), dp_(c, p, d.N);
        DBuf<double> bu(&c, N), bv(&c, N), bw(&c, N), du(&c, N), dv(&c, N), dw(&c, N), pe(&c, 4);
        AsmWork work;
        c.clear_flags();
        // the diagonals of a_u/a_v/a_w are the recurrence state (Q2): a_u.get(i,i) in the reference
        for (orc_csr* a : {a_u, a_v, a_w}) { a->m->diag = d.diag.p; a->m->own_diag = false; }
        extract_diagonal(c, *a_u->m, du); extract_diagonal(c, *a_v->m, dv); extract_diagonal(c, *a_w->m, dw);
        build_momentum_advection(c, d, work, asm_settings(s), rho, *a_u->m, *a_v->m, *a_w->m, *a_di->m, du, dv, dw, du_.d, dv_.d, dw_.d, dp_.d,
                                 bu, bv, bw, pe);
        to_host(c, b_u, bu, d.N); to_host(c, b_v, bv, d.N); to_host(c, b_w, bw, d.N);
        double hpe[3] = {0, 0, 0};
        to_host(c, hpe, pe, 3);
        for (orc_csr* a : {a_u, a_v, a_w}) { a->m->diag = nullptr; a->m->own_diag = true; }
        check_solver_flags(c);
        if (peclet3) { peclet3[0] = hpe[0] / (double)d.N; peclet3[1] = hpe[1]; peclet3[2] = hpe[2]; }
    });
}
int32_t orc_build_pressure_correction(orc_ctx* ctx, orc_mesh* m, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w,
                                      const double* u, const double* v, const double* w, const double* p, const orc_settings* s,
                                      double rho, orc_csr** a_out, double* b_out) {
    ORC_TRY({
        require(ctx && m && u && v && w && p && s && a_out && b_out, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        require_mesh_matrix(d, a_u, "a_u"); require_mesh_matrix(d, a_v, "a_v"); require_mesh_matrix(d, a_w, "a_w");
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn du_(c, u, d.N), dv_(c, v, d.N), dw_(c, w, d.N), dp_(c, p, d.N);
        DBuf<double> b(&c, N), du(&c, N), dv(&c, N), dw(&c, N);
        AsmWork work;
        c.clear_flags();
        momentum_diagonals(c, d, a_u, a_v, a_w, du, dv, dw);
        CsrPtr a = mesh_matrix(c, d);
        build_pressure_correction(c, d, work, asm_settings(s), rho, du, dv, dw, du_.d, dv_.d, dw_.d, dp_.d, *a, b);
        to_host(c, b_out, b, d.N);
        check_solver_flags(c);
        *a_out = wrap(detach(c, std::move(a)));
    });
}
int32_t orc_pressure_gradient(orc_ctx* ctx, orc_mesh* m, const double* p, double* grad3n) {
    ORC_TRY({
        require(ctx && m && p && grad3n, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn dp(c, p, d.N);
        DBuf<double> gx(&c, N), gy(&c, N), gz(&c, N);
        c.clear_flags();
        pressure_gradient(c, d, dp.d, gx, gy, gz);
        std::vector<double> hx(N), hy(N), hz(N);
        to_host(c, hx.data(), gx, d.N); to_host(c, hy.data(), gy, d.N); to_host(c, hz.data(), gz, d.N);
        check_solver_flags(c);
        for (int64_t i = 0; i < d.N; ++i) { grad3n[3 * i] = hx[i]; grad3n[3 * i + 1] = hy[i]; grad3n[3 * i + 2] = hz[i]; }
    });
}
int32_t orc_apply_pressure_correction(orc_ctx* ctx, orc_mesh* m, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w,
                                      const double* p_prime, double* u, double* v, double* w, double* p, const orc_settings* s,
                                      double* norms2) {
    ORC_TRY({
        require(ctx && m && p_prime && u && v && w && p && s, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        require_mesh_matrix(d, a_u, "a_u"); require_mesh_matrix(d, a_v, "a_v"); require_mesh_matrix(d, a_w, "a_w");
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn du_(c, u, d.N), dv_(c, v, d.N), dw_(c, w, d.N), dp_(c, p, d.N), dpp(c, p_prime, d.N);
        DBuf<double> du(&c, N), dv(&c, N), dw(&c, N), out(&c, 8);
        c.clear_flags();
        momentum_diagonals(c, d, a_u, a_v, a_w, du, dv, dw);
        apply_pressure_correction(c, d, du, dv, dw, dpp.d, du_.d, dv_.d, dw_.d, dp_.d, s->pressure_relaxation, s->momentum_relaxation, out);
        to_host(c, u, du_.d, d.N); to_host(c, v, dv_.d, d.N); to_host(c, w, dw_.d, d.N); to_host(c, p, dp_.d, d.N);
        double h[8];
        to_host(c, h, out, 8);
        check_solver_flags(c);
        if (norms2) { norms2[0] = sqrt(h[0]); norms2[1] = sqrt(h[1]); }
    });
}

// ---- solver.rs ---------------------------------------------------------------------------------------------
int32_t orc_steady_create(orc_ctx* ctx, orc_mesh* m, const orc_settings* s, double rho, double mu, orc_steady** out) {
    ORC_TRY({
        require(ctx && m && s && out, "null argument");
        ctx->c.clear_flags();
        *out = steady_create(ctx, m, s, rho, mu);
    });
}
int32_t orc_steady_set_fields(orc_steady* st, const double* u, const double* v, const double* w, const double* p) {
    ORC_TRY({
        require(st && u && v && w && p, "null argument");
        Ctx& c = *st->c;
        const double* src[4] = {u, v, w, p};
        double* dst[4] = {st->u.p, st->v.p, st->w.p, st->p.p};
        const int64_t lo = st->dm->own_lo, cnt = st->dm->own_hi - lo;  // a partition exposes its OWNED cells only
        for (int q = 0; q < 4; ++q)
            if (cnt > 0) ORC_CUDA(cudaMemcpyAsync(dst[q] + lo, src[q], sizeof(double) * cnt, cudaMemcpyHostToDevice, c.stream));
        c.sync();
    });
}
int32_t orc_steady_get_fields(orc_steady* st, double* u, double* v, double* w, double* p) {
    ORC_TRY({
        require(st && u && v && w && p, "null argument");
        Ctx& c = *st->c;
        double* dst[4] = {u, v, w, p};
        const double* src[4] = {st->u.p, st->v.p, st->w.p, st->p.p};
        const int64_t lo = st->dm->own_lo, cnt = st->dm->own_hi - lo;
        for (int q = 0; q < 4; ++q)
            if (cnt > 0) ORC_CUDA(cudaMemcpyAsync(dst[q], src[q] + lo, sizeof(double) * cnt, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
    });
}
int32_t orc_steady_reset(orc_steady* st) {
    ORC_TRY({
        require(st != nullptr, "null argument");
        Ctx& c = *st->c;
        DMesh& d = device_mesh(c, st->mesh);
        init_momentum_matrix(c, d, *st->a_u); init_momentum_matrix(c, d, *st->a_v); init_momentum_matrix(c, d, *st->a_w);
        dev_fill(c, st->du, 1., d.N); dev_fill(c, st->dv, 1., d.N); dev_fill(c, st->dw, 1., d.N);
        for (DBuf<double>* b : {&st->b_u, &st->b_v, &st->b_w, &st->p_prime, &st->u, &st->v, &st->w, &st->p}) b->zero();
        st->phi.zero();   // the resident phi, if any; the coupling stays
        st->iteration = 0;
    });
}
int32_t orc_steady_iterate(orc_steady* st, uint64_t iterations, orc_report* last) {
    ORC_TRY({
        require(st != nullptr, "null argument");
        steady_iterate(*st, iterations, 0, nullptr, nullptr, last);
    });
}
int32_t orc_steady_phase_ms(orc_steady* st, double* out5) {
    ORC_TRY({ require(st && out5, "null argument"); for (int q = 0; q < 5; ++q) out5[q] = st->phase_ms[q]; });
}
int32_t orc_steady_batched(orc_steady* st, int32_t* out) {
    ORC_TRY({ require(st && out, "null argument"); *out = st->last_batched ? 1 : 0; });
}
int32_t orc_steady_level_sizes(orc_steady* st, int64_t* out, int32_t cap, int32_t* n_levels) {
    ORC_TRY({
        require(st && out && n_levels, "null argument");
        int n = (int)st->trace.rows.size();
        *n_levels = n;
        for (int l = 0; l < n && l < cap; ++l) { out[2 * l] = st->trace.rows[l]; out[2 * l + 1] = st->trace.nnz[l]; }
    });
}
void orc_steady_destroy(orc_steady* st) {
    if (!st) return;
    if (st->c) cudaStreamSynchronize(st->c->stream);
    delete st;
}

int32_t orc_solve_steady(orc_ctx* ctx, orc_mesh* m, double* u, double* v, double* w, double* p, const orc_settings* s, double rho,
                         double mu, uint64_t iteration_count, uint64_t reporting_interval, orc_report_cb cb, void* user) {
    ORC_TRY({
        require(ctx && m && u && v && w && p && s, "null argument");
        ctx->c.clear_flags();
        std::unique_ptr<orc_steady> st(steady_create(ctx, m, s, rho, mu));
        int32_t rc = orc_steady_set_fields(st.get(), u, v, w, p);
        if (rc != ORC_OK) throw Error(rc, g_err);
        // like the reference, the fields hold whatever was reached when the solve fails
        try {
            steady_iterate(*st, iteration_count, reporting_interval, cb, user, nullptr);
        } catch (...) {
            orc_steady_get_fields(st.get(), u, v, w, p);
            throw;
        }
        rc = orc_steady_get_fields(st.get(), u, v, w, p);
        if (rc != ORC_OK) throw Error(rc, g_err);
    });
}

// ---- flow initialisation: the step before the loop (src/solver.rs:246-352, 414-509, 703-770) ---------------------------------
// check_boundary_conditions (:710-770), host logic. The two angle checks compare against TOL = 5 * 180 / PI = 286.5 (radians),
// so they can never fire; the counters are u16 and count EVERY face of the mesh for a moving wall: a release build wraps.
// `mesh_faces`: the face count of the whole mesh (h.n_faces unless h is a partition).
static int check_boundary_conditions(const HostMesh& h, int64_t mesh_faces) {
    const double PI = (double)3.14159274101257324f;  // std::f32::consts::PI as Float
    const double TOL = 5. * 180. / PI;
    uint16_t pressure_bc = 0, velocity_bc = 0;
    auto angle = [&](int64_t f, const double* v) {
        const double* n = &h.face_normal[3 * f];
        const double dot = n[0] * v[0] + n[1] * v[1] + n[2] * v[2];
        return acos(dot / (sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]) * sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])));
    };
    for (const HostZone& z : h.zones) {
        switch (z.type) {
            case ORC_BC_WALL:
                if (sqrt(z.vec[0] * z.vec[0] + z.vec[1] * z.vec[1] + z.vec[2] * z.vec[2]) > 0.) {
                    velocity_bc = (uint16_t)(velocity_bc + (uint16_t)mesh_faces);   // += 1 per face, wrapping
                    for (int64_t f = 0; f < h.n_faces; ++f)
                        if (PI / 2. - fabs(angle(f, z.vec)) > TOL) throw Error(ORC_E_INVALID, "Wall velocity must be tangent to faces in zone.");
                }
                break;
            case ORC_BC_VELOCITY_INLET:
                velocity_bc = (uint16_t)(velocity_bc + 1);
                for (int64_t f = 0; f < h.n_faces; ++f)
                    if (fabs(angle(f, z.vec)) > TOL) throw Error(ORC_E_INVALID, "VelocityInlet velocity must not be tangent to faces in zone.");
                break;
            case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: pressure_bc = (uint16_t)(pressure_bc + 1); break;
            default: break;
        }
    }
    if (velocity_bc > 0) return pressure_bc > 1 ? ORC_CONSTRAINT_HYBRID : ORC_CONSTRAINT_VELOCITY_ONLY;
    if (pressure_bc > 0) return ORC_CONSTRAINT_PRESSURE_ONLY;
    throw Error(ORC_E_INVALID, "You must set boundary conditions.");
}
int32_t orc_check_boundary_conditions(const orc_mesh* m, int32_t* constraint_type) {
    ORC_TRY({ require(m && m->h && constraint_type, "null argument"); *constraint_type = check_boundary_conditions(*m->h, m->h->n_faces); });
}
int32_t orc_build_pressure_laplace(orc_ctx* ctx, orc_mesh* m, orc_csr** a_out, double* b_out) {
    ORC_TRY({
        require(ctx && m && a_out && b_out, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        CsrPtr a = mesh_matrix(c, d);
        DBuf<double> b(&c, (size_t)std::max<int64_t>(d.N, 1));
        b.zero();
        build_pressure_laplace(c, d, *a, b);
        to_host(c, b_out, b, d.N);
        c.sync();
        *a_out = wrap(detach(c, std::move(a)));
    });
}
// ---- the initialisation on a partition mesh: every rank runs the same steps on its owned cells, collectives in lockstep ----
// check_solver_flags with the status word of all ranks: some flags are local (a singular least-squares fit on one rank), and every
// rank must return the same status (and stay in the collectives together)
static void check_agreed_flags(Ctx& c, const DistEnv& env) {
    if (!env.on()) { check_solver_flags(c); return; }
    DBuf<double> d(&c, 1);
    k_flags_to_double<<<1, 1, 0, c.stream>>>(c.d_flags, d.p);
    c.after_launch("k_flags_to_double");
    env.comm->allreduce(c, d.p, 1, 0);
    double h = 0.;
    ORC_CUDA(cudaMemcpyAsync(&h, d.p, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    c.clear_flags();
    throw_for_flags(flags_from_double(h));
}
struct InitEnv {
    DistEnv env;
    bool exact_order = false;
    int constraint = ORC_CONSTRAINT_PRESSURE_ONLY;
    int64_t lo = 0, n_own = 0;   // the cells the caller receives
};
// What both initialisations do first: the boundary-condition check over the WHOLE mesh (a partition counts the faces whose c0 it
// owns, so that every face is counted once), the reduction mode, and the halo plan of a partition (its hook goes into `work`).
static InitEnv init_env(orc_ctx* ctx, orc_mesh* m, int reduction_mode, AsmWork* work) {
    Ctx& c = ctx->c;
    InitEnv ie;
    const HostMesh& h = *m->h;
    if (!m->plan) {
        ie.constraint = check_boundary_conditions(h, h.n_faces);
        DMesh& d = device_mesh(c, m);
        ie.exact_order = resolve_exact_order(reduction_mode, d.N);
        ie.n_own = d.N;
        return ie;
    }
    if (reduction_mode == ORC_REDUCE_REFERENCE_ORDER) throw Error(ORC_E_UNSUPPORTED, "reference-order reductions are single-GPU only");
    DMesh& d = device_mesh(c, m);
    ie.env = partition_env(ctx, m, work);
    int64_t own_faces = 0;
    for (int64_t f = 0; f < h.n_faces; ++f) own_faces += (h.face_c0[f] >= d.own_lo && h.face_c0[f] < d.own_hi);
    ie.constraint = check_boundary_conditions(h, (int64_t)allreduce_host(c, ctx->comm, (double)own_faces, 0));
    ie.lo = d.own_lo; ie.n_own = d.own_hi - d.own_lo;
    return ie;
}

// initialize_flow (:246-352): Laplace pressure field (Jacobi x10), one UD / LinearWeighted momentum assembly at rest, then six
// rounds of BiCGSTAB on a_u * (1 - f) + a_di * f, f = 1, 0.8, ... for u, v and w. The three blended matrices are bit-identical
// (UD), so the three solves of a round run in lockstep like the momentum solves of the loop.
int32_t orc_initialize_flow(orc_ctx* ctx, orc_mesh* m, double mu, double rho, uint64_t iteration_count, int32_t reduction_mode, double* u,
                            double* v, double* w, double* p) {
    ORC_TRY({
        require(ctx && m && u && v && w && p, "null argument");
        Ctx& c = ctx->c;
        c.clear_flags();
        AsmWork work;
        const InitEnv ie = init_env(ctx, m, reduction_mode, &work);                                          // :272
        const DistEnv& env = ie.env;
        DMesh& d = device_mesh(c, m);
        const int64_t N = d.N;
        const size_t Nz = (size_t)std::max<int64_t>(N, 1);
        DBuf<double> du(&c, Nz), dv(&c, Nz), dw(&c, Nz), dp(&c, Nz), b_u_di(&c, Nz), b_v_di(&c, Nz), b_w_di(&c, Nz), b_u(&c, Nz), b_v(&c, Nz),
            b_w(&c, Nz), diag_u(&c, Nz), diag_v(&c, Nz), diag_w(&c, Nz), pb(&c, Nz), pe3(&c, 4);
        for (DBuf<double>* q : {&du, &dv, &dw, &dp, &b_u, &b_v, &b_w, &pb}) q->zero();                      // :274-285
        CsrPtr a_di = mesh_matrix(c, d), a_u = mesh_matrix(c, d), a_v = mesh_matrix(c, d), a_w = mesh_matrix(c, d), lap = mesh_matrix(c, d),
               blend = mesh_matrix(c, d);
        build_momentum_diffusion(c, d, mu, *a_di, b_u_di, b_v_di, b_w_di);                                  // :278-279
        init_momentum_matrix(c, d, *a_u); init_momentum_matrix(c, d, *a_v); init_momentum_matrix(c, d, *a_w);  // :280-282
        dev_fill(c, diag_u, 1., N); dev_fill(c, diag_v, 1., N); dev_fill(c, diag_w, 1., N);
        SolveParams sp;
        sp.exact_order = ie.exact_order;
        // initialize_pressure_field (:414-509)
        build_pressure_laplace(c, d, *lap, pb);
        sp.iterations = 10; sp.method = ORC_SOLVER_JACOBI; sp.relaxation = 0.1; sp.threshold = 1e-6; sp.preconditioner = ORC_PC_JACOBI;
        iterative_solve(c, *lap, pb, dp, sp, nullptr, 1, &env);                                             // :498-507
        check_agreed_flags(c, env);
        // :288-306: UD, LinearWeighted velocity and pressure interpolation, Green-Gauss cell based; u = v = w = 0
        AsmSettings as;
        as.momentum = ORC_MOM_UD; as.limiter = ORC_PSI_UD; as.p_interp = ORC_P_LINEAR_WEIGHTED; as.v_interp = ORC_V_LINEAR_WEIGHTED;
        as.gradient = ORC_G_GREEN_GAUSS_CELL; as.assembly_mode = ORC_ASSEMBLY_EXACT;
        exchange(c, env, {dp.p});                                                                          // the neighbours' pressure
        build_momentum_advection(c, d, work, as, rho, *a_u, *a_v, *a_w, *a_di, diag_u, diag_v, diag_w, du, dv, dw, dp, b_u, b_v, b_w, pe3);
        dev_axpy_inplace(c, b_u, b_u_di, N); dev_axpy_inplace(c, b_v, b_v_di, N); dev_axpy_inplace(c, b_w, b_w_di, N);  // :307-309
        sp.iterations = iteration_count; sp.method = ORC_SOLVER_BICGSTAB; sp.relaxation = 0.5; sp.threshold = 1e-6;
        const bool batch3 = lockstep(c, env, lockstep_enabled(), sp, *a_u, *a_v, *a_w);
        double f = 1.;
        while (f >= 0.) {                                                                                  // :316-350
            if (batch3) {
                csr_blend(c, *a_u, 1. - f, *a_di, f, *blend);
                solve_lockstep(c, env, *blend, b_u, b_v, b_w, du, dv, dw, N, sp);
            } else {
                csr_blend(c, *a_u, 1. - f, *a_di, f, *blend); iterative_solve(c, *blend, b_u, du, sp, nullptr, 1, &env);
                csr_blend(c, *a_v, 1. - f, *a_di, f, *blend); iterative_solve(c, *blend, b_v, dv, sp, nullptr, 1, &env);
                csr_blend(c, *a_w, 1. - f, *a_di, f, *blend); iterative_solve(c, *blend, b_w, dw, sp, nullptr, 1, &env);
            }
            f -= 0.2;
        }
        to_host(c, u, du + ie.lo, ie.n_own); to_host(c, v, dv + ie.lo, ie.n_own); to_host(c, w, dw + ie.lo, ie.n_own); to_host(c, p, dp + ie.lo, ie.n_own);
        check_agreed_flags(c, env);
    });
}

// initialize_flow_new (src/solver.rs:354-410), what the reference's current main() calls before solve_steady (src/tests.rs:195-197).
// The match arms overlap — `PressureOnly | Hybrid` comes first — so a Hybrid system gets its pressure field only. VelocityOnly:
// initialize_velocity_field (:511-696): potential system, BiCGSTAB x10 (Jacobi preconditioner), velocity = least-squares grad psi.
// The two debug files the reference writes on the way (psi.csv, psi_gradients.csv) are not written here (orc_b200.io has both writers).
int32_t orc_build_velocity_potential(orc_ctx* ctx, orc_mesh* m, orc_csr** a_out, double* b_out) {
    ORC_TRY({
        require(ctx && m && a_out && b_out, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        CsrPtr a = mesh_matrix(c, d);
        DBuf<double> b(&c, (size_t)std::max<int64_t>(d.N, 1));
        b.zero();
        build_velocity_potential(c, d, *a, b);
        to_host(c, b_out, b, d.N);
        c.sync();
        *a_out = wrap(detach(c, std::move(a)));
    });
}
int32_t orc_potential_gradient(orc_ctx* ctx, orc_mesh* m, const double* psi, double* u, double* v, double* w) {
    ORC_TRY({
        require(ctx && m && psi && u && v && w, "null argument");
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        const size_t Nz = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn dpsi(c, psi, d.N);
        DBuf<double> du(&c, Nz), dv(&c, Nz), dw(&c, Nz);
        potential_gradient(c, d, dpsi.d, du, dv, dw);
        to_host(c, u, du, d.N); to_host(c, v, dv, d.N); to_host(c, w, dw, d.N);
        c.sync();
    });
}
int32_t orc_initialize_flow_new(orc_ctx* ctx, orc_mesh* m, double mu, double rho, uint64_t iteration_count, int32_t reduction_mode, double* u,
                                double* v, double* w, double* p) {
    ORC_TRY({
        require(ctx && m && u && v && w && p, "null argument");
        (void)mu; (void)rho; (void)iteration_count;   // unused by the reference as well (:354-358, `_iteration_count` :414)
        Ctx& c = ctx->c;
        c.clear_flags();
        const InitEnv ie = init_env(ctx, m, reduction_mode, nullptr);                                      // :395
        const DistEnv& env = ie.env;
        DMesh& d = device_mesh(c, m);
        const int64_t N = d.N;
        const size_t Nz = (size_t)std::max<int64_t>(N, 1);
        DBuf<double> du(&c, Nz), dv(&c, Nz), dw(&c, Nz), dp(&c, Nz), rhs(&c, Nz), psi(&c, Nz);
        for (DBuf<double>* q : {&du, &dv, &dw, &dp, &rhs, &psi}) q->zero();
        CsrPtr a = mesh_matrix(c, d);
        SolveParams sp;
        sp.exact_order = ie.exact_order;
        sp.preconditioner = ORC_PC_JACOBI; sp.iterations = 10; sp.relaxation = 0.1; sp.threshold = 1e-6;
        if (ie.constraint == ORC_CONSTRAINT_PRESSURE_ONLY || ie.constraint == ORC_CONSTRAINT_HYBRID) {      // :399-402
            build_pressure_laplace(c, d, *a, rhs);
            sp.method = ORC_SOLVER_JACOBI;
            iterative_solve(c, *a, rhs, dp, sp, nullptr, 1, &env);                                         // :498-507
        } else {                                                                                           // :403-405
            build_velocity_potential(c, d, *a, rhs);
            sp.method = ORC_SOLVER_BICGSTAB;
            iterative_solve(c, *a, rhs, psi, sp, nullptr, 1, &env);                                        // :592-601
            exchange(c, env, {psi.p});                                                                     // the neighbours' psi
            potential_gradient(c, d, psi, du, dv, dw);                                                     // :624-693
        }
        to_host(c, u, du + ie.lo, ie.n_own); to_host(c, v, dv + ie.lo, ie.n_own); to_host(c, w, dw + ie.lo, ie.n_own); to_host(c, p, dp + ie.lo, ie.n_own);
        check_agreed_flags(c, env);
    });
}
// calculate_pressure_gradient / calculate_velocity_gradient of every cell (src/solver.rs:774-949): what write_gradients prints
// (src/io.rs:623-662). grad_p3n: N x 3, grad_u9n: N x 9 row-major tensors; either may be null.
static void require_gradient_scheme(int32_t gradient, bool pressure) {
    if (gradient == ORC_G_GREEN_GAUSS_NODE && pressure) throw Error(ORC_E_UNSUPPORTED, "unsupported Green-Gauss scheme");   // solver.rs:901
    if (gradient != ORC_G_GREEN_GAUSS_CELL && gradient != ORC_G_GREEN_GAUSS_NODE && gradient != ORC_G_LEAST_SQUARES)
        throw Error(ORC_E_UNSUPPORTED, "unsupported gradient scheme");                                                      // :870, 948
}
// the gradients of device fields u, v, w, p; rows [lo, lo + cnt) of the mesh go to the host in orc_gradients' layout
static void gradients_to_host(Ctx& c, const DMesh& d, const double* u, const double* v, const double* w, const double* p, int32_t gradient,
                              int64_t lo, int64_t cnt, double* grad_p3n, double* grad_u9n) {
    const size_t N = (size_t)std::max<int64_t>(d.N, 1);
    const int g = (gradient == ORC_G_LEAST_SQUARES) ? ORC_G_LEAST_SQUARES : ORC_G_GREEN_GAUSS_CELL;
    if (grad_p3n) {
        DBuf<double> gx(&c, N), gy(&c, N), gz(&c, N);
        pressure_gradient(c, d, p, gx, gy, gz, g);
        std::vector<double> hx(N), hy(N), hz(N);
        to_host(c, hx.data(), gx, d.N); to_host(c, hy.data(), gy, d.N); to_host(c, hz.data(), gz, d.N);
        c.sync();
        for (int64_t i = 0; i < cnt; ++i) { grad_p3n[3 * i] = hx[lo + i]; grad_p3n[3 * i + 1] = hy[lo + i]; grad_p3n[3 * i + 2] = hz[lo + i]; }
    }
    if (grad_u9n) {
        DBuf<double> gu(&c, 9 * N);
        velocity_gradient(c, d, u, v, w, gu, g);
        std::vector<double> h(9 * N);
        to_host(c, h.data(), gu, 9 * d.N);
        c.sync();
        for (int64_t i = 0; i < cnt; ++i) for (int k = 0; k < 9; ++k) grad_u9n[9 * i + k] = h[(size_t)k * d.N + lo + i];
    }
}
int32_t orc_gradients(orc_ctx* ctx, orc_mesh* m, const double* u, const double* v, const double* w, const double* p, int32_t gradient,
                      double* grad_p3n, double* grad_u9n) {
    ORC_TRY({
        require(ctx && m && u && v && w && p, "null argument");
        require_gradient_scheme(gradient, grad_p3n != nullptr);
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        HostVecIn du(c, u, d.N), dv(c, v, d.N), dw(c, w, d.N), dp(c, p, d.N);
        c.clear_flags();
        gradients_to_host(c, d, du.d, dv.d, dw.d, dp.d, gradient, 0, d.N, grad_p3n, grad_u9n);
        check_solver_flags(c);
    });
}
int32_t orc_steady_gradients(orc_steady* st, int32_t gradient, double* grad_p3n, double* grad_u9n) {
    ORC_TRY({
        require(st != nullptr, "null argument");
        require_gradient_scheme(gradient, grad_p3n != nullptr);
        Ctx& c = *st->c;
        DMesh& d = device_mesh(c, st->mesh);
        c.clear_flags();
        exchange(c, st->env, {st->u.p, st->v.p, st->w.p, st->p.p});   // the halo cells hold whatever the last exchange left
        gradients_to_host(c, d, st->u, st->v, st->w, st->p, gradient, d.own_lo, d.own_hi - d.own_lo, grad_p3n, grad_u9n);
        check_agreed_flags(c, st->env);
    });
}

// ---- passive scalar transport (an extension beyond the reference, DESIGN.md §1) ---------------------------------------------------
int32_t orc_mesh_set_zone_scalar(orc_mesh* m, const char* name, int32_t kind, double value) {
    ORC_TRY({
        require(m && name, "null argument");
        int k = m->h->find_zone(name);
        if (k < 0) throw Error(ORC_E_INVALID, std::string("face zone '") + name + "' should exist in mesh");
        require(kind == ORC_SBC_ZERO_GRADIENT || kind == ORC_SBC_FIXED, "unknown scalar boundary condition kind");
        require(std::isfinite(value), "scalar boundary value must be finite");
        HostZone& z = m->h->zones[k];
        z.scalar_bc_kind = kind; z.scalar_bc_value = value;
        m->h->zone_epoch++;
    });
}
int32_t orc_build_scalar_transport(orc_ctx* ctx, orc_mesh* m, const orc_csr* a_u, const orc_csr* a_v, const orc_csr* a_w,
                                   const double* u, const double* v, const double* w, const double* p, const double* phi,
                                   double gamma, double rho, const orc_settings* s, orc_csr** a_out, double* b_out) {
    ORC_TRY({
        require(ctx && m && m->h && u && v && w && p && phi && s && a_out && b_out, "null argument");
        const AsmSettings as = asm_settings(s);
        require_scalar_problem(*m->h, gamma, as);
        Ctx& c = ctx->c;
        DMesh& d = device_mesh(c, m);
        require_mesh_matrix(d, a_u, "a_u"); require_mesh_matrix(d, a_v, "a_v"); require_mesh_matrix(d, a_w, "a_w");
        ScalarWork work;
        const DistEnv env = m->plan ? partition_env(ctx, m, nullptr) : DistEnv();
        if (env.on()) { Comm* cm = env.comm; Halo* hl = env.halo; Ctx* cp = &c; work.halo_exchange = [cm, hl, cp](double* const* f, int n) { hl->exchange(*cp, *cm, f, n); }; }
        const size_t N = (size_t)std::max<int64_t>(d.N, 1);
        HostVecIn du_(c, u, d.N), dv_(c, v, d.N), dw_(c, w, d.N), dp_(c, p, d.N), dphi(c, phi, d.N);
        DBuf<double> b(&c, N), du(&c, N), dv(&c, N), dw(&c, N);
        c.clear_flags();
        momentum_diagonals(c, d, a_u, a_v, a_w, du, dv, dw);
        exchange(c, env, {du_.d.p, dv_.d.p, dw_.d.p, dp_.d.p});
        exchange(c, env, {du.p, dv.p, dw.p, dphi.d.p});
        CsrPtr a = mesh_matrix(c, d);
        scalar_face_flux(c, d, work, as, du, dv, dw, du_.d, dv_.d, dw_.d, dp_.d);
        build_scalar_transport(c, d, work, as, gamma, rho, dphi.d, *a, b);
        to_host(c, b_out, b, d.N);
        check_agreed_flags(c, env);
        *a_out = wrap(detach(c, std::move(a)));
    });
}
// The handle's u, v, w, p, du, dv, dw with their halo cells filled, read, never written: on a partition they are copied to `flow`
// before their halo exchange (the copies' halo cells get the owners' values), so the next iterate() sees exactly what it would have
// seen.
static void resident_flow(orc_steady& st, DBuf<double>& flow, const double* out[7]) {
    const double* src[7] = {st.u, st.v, st.w, st.p, st.du, st.dv, st.dw};
    for (int k = 0; k < 7; ++k) out[k] = src[k];
    if (!st.env.on()) return;
    Ctx& c = *st.c;
    const size_t Nz = (size_t)std::max<int64_t>(st.N, 1);
    flow.alloc(&c, 7 * Nz);
    for (int k = 0; k < 7; ++k) {
        ORC_CUDA(cudaMemcpyAsync(flow.p + k * Nz, src[k], sizeof(double) * st.N, cudaMemcpyDeviceToDevice, c.stream));
        out[k] = flow.p + k * Nz;
    }
    exchange(c, st.env, {flow.p, flow.p + Nz, flow.p + 2 * Nz, flow.p + 3 * Nz});
    exchange(c, st.env, {flow.p + 4 * Nz, flow.p + 5 * Nz, flow.p + 6 * Nz});
}
// The flow state of the handle is left as it was (resident_flow).
int32_t orc_steady_solve_scalar(orc_steady* st, double gamma, uint64_t sweeps, double* phi) {
    ORC_TRY({
        require(st && phi, "null argument");
        const AsmSettings as = asm_settings(&st->s);
        require_scalar_problem(*st->mesh->h, gamma, as);
        Ctx& c = *st->c;
        DMesh& d = device_mesh(c, st->mesh);
        const DistEnv& env = st->env;
        const SolveParams sp = solve_params(&st->s, env.on() ? INT64_MAX : st->N_global);
        const int64_t lo = d.own_lo, cnt = d.own_hi - d.own_lo;
        const size_t Nz = (size_t)std::max<int64_t>(d.N, 1);
        c.clear_flags();
        ScalarWork work;
        work.halo_exchange = st->work.halo_exchange;
        DBuf<double> flow;
        const double* f[7];
        resident_flow(*st, flow, f);
        DBuf<double> x(&c, Nz), b(&c, Nz);
        x.zero();
        if (cnt > 0) ORC_CUDA(cudaMemcpyAsync(x.p + lo, phi, sizeof(double) * cnt, cudaMemcpyHostToDevice, c.stream));
        CsrPtr a = mesh_matrix(c, d);
        scalar_sweeps(c, d, env, work, as, sp, gamma, st->rho, sweeps, f[4], f[5], f[6], f[0], f[1], f[2], f[3], *a, b, x);
        to_host(c, phi, x.p + lo, cnt);
        check_agreed_flags(c, env);
        c.prof_resolve();
    });
}

// ---- Boussinesq coupling of the scalar into the loop (an extension beyond the reference, DESIGN.md §1) -----------------------------
int32_t orc_steady_couple_scalar(orc_steady* st, double gamma, double beta, double phi_ref, double gx, double gy, double gz, uint64_t sweeps) {
    ORC_TRY({
        require(st != nullptr, "null argument");
        if (sweeps == 0) {
            st->cpl = orc_steady::Coupling();
        } else {
            require_scalar_problem(*st->mesh->h, gamma, asm_settings(&st->s));
            require(std::isfinite(beta) && std::isfinite(phi_ref) && std::isfinite(gx) && std::isfinite(gy) && std::isfinite(gz),
                    "beta, phi_ref and g must be finite");
            ensure_scalar(*st);
            orc_steady::Coupling k;
            k.gamma = gamma; k.beta = beta; k.phi_ref = phi_ref; k.g[0] = gx; k.g[1] = gy; k.g[2] = gz; k.sweeps = sweeps;
            st->cpl = k;
        }
    });
}
int32_t orc_steady_set_scalar(orc_steady* st, const double* phi) {
    ORC_TRY({
        require(st && phi, "null argument");
        ensure_scalar(*st);
        Ctx& c = *st->c;
        const int64_t lo = st->dm->own_lo, cnt = st->dm->own_hi - lo;
        if (cnt > 0) ORC_CUDA(cudaMemcpyAsync(st->phi.p + lo, phi, sizeof(double) * cnt, cudaMemcpyHostToDevice, c.stream));
        c.sync();
    });
}
int32_t orc_steady_get_scalar(orc_steady* st, double* phi) {
    ORC_TRY({
        require(st && phi, "null argument");
        ensure_scalar(*st);
        to_host(*st->c, phi, st->phi.p + st->dm->own_lo, st->dm->own_hi - st->dm->own_lo);
        st->c->sync();
    });
}
int32_t orc_steady_scalar_zone_flux(orc_steady* st, const char* name, double* out2) {
    ORC_TRY({
        require(st && name && out2, "null argument");
        const HostMesh& h = *st->mesh->h;
        const int zone = h.find_zone(name);
        if (zone < 0) throw Error(ORC_E_INVALID, std::string("face zone '") + name + "' should exist in mesh");
        require(st->cpl.sweeps > 0, "the handle is not coupled (orc_steady_couple_scalar): the zone flux uses the coupling's gamma");
        const AsmSettings as = asm_settings(&st->s);
        require_scalar_problem(h, st->cpl.gamma, as);
        Ctx& c = *st->c;
        DMesh& d = device_mesh(c, st->mesh);
        c.clear_flags();
        DBuf<double> flow;
        const double* f[7];
        resident_flow(*st, flow, f);
        scalar_face_flux(c, d, st->swork, as, f[4], f[5], f[6], f[0], f[1], f[2], f[3]);
        const size_t F = (size_t)std::max<int64_t>(d.F, 1);
        DBuf<double> terms(&c, 2 * F);
        terms.zero();
        scalar_zone_flux(c, d, st->swork, st->cpl.gamma, st->rho, st->phi, zone, terms);
        std::vector<double> t(2 * F);
        to_host(c, t.data(), terms, 2 * (int64_t)F);
        c.sync();
        double mine[2] = {0., 0.};   // ascending face order; faces of other zones hold +0
        for (int64_t q = 0; q < d.F; ++q) { mine[0] += t[q]; mine[1] += t[F + q]; }
        out2[0] = mine[0]; out2[1] = mine[1];
        if (st->env.on()) {   // every boundary face belongs to one rank: the ranks' totals, added in rank order
            Comm& cm = *st->env.comm;
            DBuf<double> one(&c, 2);
            out2[0] = out2[1] = 0.;
            for (int r = 0; r < cm.nranks; ++r) {
                double v[2] = {r == cm.rank ? mine[0] : 0., r == cm.rank ? mine[1] : 0.};
                ORC_CUDA(cudaMemcpyAsync(one.p, v, sizeof(v), cudaMemcpyHostToDevice, c.stream));
                cm.allreduce(c, one.p, 2, 0);
                ORC_CUDA(cudaMemcpyAsync(v, one.p, sizeof(v), cudaMemcpyDeviceToHost, c.stream));
                c.sync();
                out2[0] += v[0]; out2[1] += v[1];
            }
        }
        check_agreed_flags(c, st->env);
    });
}

// ---- multi-GPU ------------------------------------------------------------------------------------------------------
int32_t orc_comm_unique_id(char* out128) { ORC_TRY({ require(out128 != nullptr, "null argument"); Comm::unique_id(out128); }); }
int32_t orc_ctx_comm_init(orc_ctx* ctx, int32_t rank, int32_t nranks, const char* id128) {
    ORC_TRY({ require(ctx && (nranks == 1 || id128), "null argument"); ctx->comm.init(ctx->c, rank, nranks, id128); });
}
// Peer windows (symmetric memory over CUDA IPC, dist.cuh): step 1 allocates this rank's window and returns its 64-byte IPC handle;
// the caller gathers the handles of all ranks (any transport: torch.distributed in the Python mirror) and step 2 maps them. Every rank
// must end in the same state: if any rank fails to open, all call orc_ctx_peer_disable (the NCCL path is used then).
int32_t orc_ctx_peer_window(orc_ctx* ctx, char* handle_out64) {
    ORC_TRY({
        require(ctx && handle_out64, "null argument");
        require(ctx->comm.active(), "create the communicator first (orc_ctx_comm_init)");
        ctx->comm.peer.alloc_window(ctx->c, ctx->comm.rank, ctx->comm.nranks, handle_out64);
    });
}
int32_t orc_ctx_peer_open(orc_ctx* ctx, const char* all_handles) {
    ORC_TRY({ require(ctx && all_handles, "null argument"); ctx->comm.peer.open(ctx->c, all_handles); });
}
int32_t orc_ctx_peer_disable(orc_ctx* ctx) {
    ORC_TRY({ require(ctx != nullptr, "null argument"); ctx->c.sync(); ctx->comm.peer.destroy(); });
}
int32_t orc_ctx_peer_enabled(orc_ctx* ctx, int32_t* out) {
    ORC_TRY({ require(ctx && out, "null argument"); *out = ctx->comm.peer.on ? 1 : 0; });
}
int32_t orc_mesh_partition(const orc_mesh* global, int32_t rank, int32_t nranks, orc_mesh** out) {
    ORC_TRY({
        require(global && global->h && out, "null argument");
        require(!global->plan, "mesh is already a partition");
        std::unique_ptr<orc_mesh> m(new orc_mesh());
        m->plan.reset(new PartPlan());
        m->h.reset(extract_partition(*global->h, rank, nranks, even_cuts(global->h->n_cells, nranks), 0, global->h->n_cells, *m->plan));
        *out = m.release();
    });
}
int32_t orc_mesh_partition_window(const orc_mesh* window, int32_t rank, int32_t nranks, const int64_t* cuts, int64_t id_offset,
                                  int64_t n_global, orc_mesh** out) {
    ORC_TRY({
        require(window && window->h && cuts && out, "null argument");
        require(!window->plan, "mesh is already a partition");
        std::unique_ptr<orc_mesh> m(new orc_mesh());
        m->plan.reset(new PartPlan());
        m->h.reset(extract_partition(*window->h, rank, nranks, std::vector<int64_t>(cuts, cuts + nranks + 1), id_offset, n_global, *m->plan));
        *out = m.release();
    });
}
int32_t orc_mesh_partition_info(const orc_mesh* m, int64_t* out8) {
    ORC_TRY({
        require(m && out8, "null argument");
        require(m->plan != nullptr, "not a partition mesh");
        const PartPlan& p = *m->plan;
        out8[0] = p.g0; out8[1] = p.g1; out8[2] = p.n_lo; out8[3] = p.n_own; out8[4] = p.n_hi; out8[5] = (int64_t)p.nbr_rank.size();
        out8[6] = (int64_t)p.send_idx.size(); out8[7] = p.n_global;
    });
}
int32_t orc_mesh_partition_maps(const orc_mesh* m, int64_t* local_to_global, int32_t* nbr_rank, int32_t* send_ptr, int32_t* send_idx,
                                int32_t* recv_begin, int32_t* recv_count) {
    ORC_TRY({
        require(m && m->plan, "not a partition mesh");
        const PartPlan& p = *m->plan;
        if (local_to_global) std::copy(p.local_to_global.begin(), p.local_to_global.end(), local_to_global);
        if (nbr_rank) std::copy(p.nbr_rank.begin(), p.nbr_rank.end(), nbr_rank);
        if (send_ptr) std::copy(p.send_ptr.begin(), p.send_ptr.end(), send_ptr);
        if (send_idx) std::copy(p.send_idx.begin(), p.send_idx.end(), send_idx);
        if (recv_begin) std::copy(p.recv_begin.begin(), p.recv_begin.end(), recv_begin);
        if (recv_count) std::copy(p.recv_count.begin(), p.recv_count.end(), recv_count);
    });
}

// ---- measurement hooks -----------------------------------------------------------------------------------------
int32_t orc_prof_enable(orc_ctx* ctx, int32_t on) {
    ORC_TRY({ require(ctx != nullptr, "null ctx"); ctx->c.prof_reset(); ctx->c.prof.enabled = on != 0; });
}
int32_t orc_prof_get_ref_bytes(orc_ctx* ctx, double* bytes, int32_t n_classes) {
    ORC_TRY({
        require(ctx && bytes, "null argument");
        ctx->c.prof_resolve();
        for (int k = 0; k < n_classes && k < PC_COUNT; ++k) bytes[k] = ctx->c.prof.ref_bytes[k];
    });
}
int32_t orc_prof_get_spmv_detail(orc_ctx* ctx, int32_t cap, int64_t* rows, int64_t* nnz, int32_t* systems, double* ms, double* bytes,
                                 uint64_t* count, int32_t* n_out) {
    ORC_TRY({
        require(ctx && rows && nnz && systems && ms && bytes && count && n_out, "null argument");
        ctx->c.prof_resolve();
        int n = 0;
        for (auto& kv : ctx->c.prof.detail) {
            if (n >= cap) break;
            nnz[n] = kv.first / 8; rows[n] = ctx->c.prof.rows_of[kv.first / 8]; systems[n] = (int32_t)(kv.first % 8); ms[n] = kv.second.ms; bytes[n] = kv.second.bytes; count[n] = kv.second.count;
            ++n;
        }
        *n_out = n;
    });
}
int32_t orc_prof_config(orc_ctx* ctx, uint32_t class_mask, uint32_t sample_every) {
    ORC_TRY({
        require(ctx != nullptr && sample_every >= 1, "bad argument");
        ctx->c.prof.class_mask = class_mask; ctx->c.prof.sample_every = sample_every;
        for (auto& v : ctx->c.prof.seen) v = 0;
    });
}
int32_t orc_prof_get(orc_ctx* ctx, double* ms, double* bytes, uint64_t* count, int32_t n_classes) {
    ORC_TRY({
        require(ctx && ms && bytes && count, "null argument");
        ctx->c.prof_resolve();
        for (int k = 0; k < n_classes && k < PC_COUNT; ++k) { ms[k] = ctx->c.prof.ms[k]; bytes[k] = ctx->c.prof.bytes[k]; count[k] = ctx->c.prof.count[k]; }
    });
}
static double bench_spmv(Ctx& c, const DCsr& A, int K, int reps) {
    c.exact_order = false;   // times the fast kernels, whatever reduction mode the last solve on this context used
    const int S = K == 1 ? 1 : 4;
    DBuf<double> x(&c, (size_t)std::max<int64_t>(A.ncols, 1) * S), y(&c, (size_t)std::max<int64_t>(A.nrows, 1) * S);
    dev_fill(c, x, 1., A.ncols * S);
    for (int q = 0; q < 3; ++q) spmv(c, A, x, y, K);
    cudaEvent_t e0, e1;
    ORC_CUDA(cudaEventCreate(&e0)); ORC_CUDA(cudaEventCreate(&e1));
    ORC_CUDA(cudaEventRecord(e0, c.stream));
    for (int q = 0; q < reps; ++q) spmv(c, A, x, y, K);
    ORC_CUDA(cudaEventRecord(e1, c.stream));
    c.sync();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return ms / reps;
}
static double bench_bicgstab(Ctx& c, const DCsr& A, int K, int reps) {
    c.exact_order = false;
    const int S = K == 1 ? 1 : 4;
    const size_t n = (size_t)std::max<int64_t>(A.nrows, 1) * S;
    DBuf<double> x(&c, n), b(&c, n);
    dev_fill(c, x, 0., A.nrows * S);
    dev_fill(c, b, 1., A.nrows * S);
    bicgstab(c, A, b, x, 3, K);
    dev_fill(c, x, 0., A.nrows * S);
    cudaEvent_t e0, e1;
    ORC_CUDA(cudaEventCreate(&e0)); ORC_CUDA(cudaEventCreate(&e1));
    ORC_CUDA(cudaEventRecord(e0, c.stream));
    bicgstab(c, A, b, x, (uint64_t)reps, K);
    ORC_CUDA(cudaEventRecord(e1, c.stream));
    c.sync();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    c.clear_flags();
    return ms / reps;
}
int32_t orc_bench_amg_setup(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_restriction, double* ms_galerkin, orc_csr** coarse_out) {
    ORC_TRY({
        require(ctx && a && ms_restriction && ms_galerkin && reps > 0, "bad argument");
        Ctx& c = ctx->c;
        DCsr& A = *a->m;
        cudaEvent_t e[3];
        for (auto& q : e) ORC_CUDA(cudaEventCreate(&q));
        double tr = 1e30, tg = 1e30;
        CsrPtr Ac;
        for (int r = 0; r < reps; ++r) {
            CsrPtr RT, R;
            c.sync();
            ORC_CUDA(cudaEventRecord(e[0], c.stream));
            R = build_restriction(c, A, ORC_RESTRICT_STRONGEST, &RT);
            ORC_CUDA(cudaEventRecord(e[1], c.stream));
            Ac = galerkin(c, *R, *RT, A);
            ORC_CUDA(cudaEventRecord(e[2], c.stream));
            c.sync();
            float m0 = 0.f, m1 = 0.f;
            cudaEventElapsedTime(&m0, e[0], e[1]);
            cudaEventElapsedTime(&m1, e[1], e[2]);
            tr = std::min(tr, (double)m0); tg = std::min(tg, (double)m1);
        }
        for (auto& q : e) cudaEventDestroy(q);
        check_solver_flags(c);
        *ms_restriction = tr; *ms_galerkin = tg;
        if (coarse_out) {
            std::unique_ptr<orc_csr> h(new orc_csr());
            h->m = std::move(Ac);
            *coarse_out = h.release();
        }
    });
}
int32_t orc_bench_spmv(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_per_launch) {
    ORC_TRY({ require(ctx && a && ms_per_launch && reps > 0, "bad argument"); *ms_per_launch = bench_spmv(ctx->c, *a->m, 1, reps); });
}
int32_t orc_bench_bicgstab(orc_ctx* ctx, const orc_csr* a, int32_t reps, double* ms_per_iteration) {
    ORC_TRY({ require(ctx && a && ms_per_iteration && reps > 0, "bad argument"); *ms_per_iteration = bench_bicgstab(ctx->c, *a->m, 1, reps); });
}
int32_t orc_bench_spmv_batch(orc_ctx* ctx, const orc_csr* a, int32_t systems, int32_t reps, double* ms_per_launch) {
    ORC_TRY({
        require(ctx && a && ms_per_launch && reps > 0 && (systems == 1 || systems == 3), "bad argument");
        *ms_per_launch = bench_spmv(ctx->c, *a->m, systems, reps);
    });
}
int32_t orc_bench_bicgstab_batch(orc_ctx* ctx, const orc_csr* a, int32_t systems, int32_t reps, double* ms_per_iteration) {
    ORC_TRY({
        require(ctx && a && ms_per_iteration && reps > 0 && (systems == 1 || systems == 3), "bad argument");
        *ms_per_iteration = bench_bicgstab(ctx->c, *a->m, systems, reps);
    });
}

}  // extern "C"
