// assembly.cu — sm_100a kernels for the assembly half of ORC's SIMPLE loop: Green-Gauss gradients,
// face pressure, Rhie-Chow face flux, momentum (UD/CD1/TVD with LUD/QUICK/UMIST limiters) and
// pressure-correction coefficients, and the pressure/velocity correction.
//
// Layout and parallelisation (DESIGN.md §3-4): SoA mesh in HBM; one thread per cell gathers its faces
// in ascending face order (the reference's accumulation order, so sums are bit-identical) and writes
// coefficients straight into the shared CSR pattern through the precomputed (cell, face) -> nnz map:
// no atomics, no COO, no sort. Side-independent face quantities (face pressure) are computed once per
// face by a face-parallel kernel; grad p once per cell instead of up to ~24x in the reference.
// The reference's in-place diagonal recurrence (SURVEY.md Q2) is kept exact by a level-scheduled
// cooperative kernel. All arithmetic keeps the reference's operator order; compiled with -fmad=false.
#include "assembly.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "vecmath.cuh"

namespace cg = cooperative_groups;

namespace orc {

// -------------------------------------------------------------------------------------------------
// device view of the mesh
// -------------------------------------------------------------------------------------------------
struct MV {
    int N, F;
    int lo, hi;  // owned cell range (whole mesh unless this is a partition: halo cells have no faces and no matrix row)
    const int *c0, *c1, *fz;
    const double *area, *fnx, *fny, *fnz, *fcx, *fcy, *fcz;
    const double *vol, *ccx, *ccy, *ccz;
    const int *cf_ptr, *cf_face, *cf_nb, *cf_slot, *diag;
    const int* zt;
    const double *zs, *zv;
};
static MV view(const DMesh& d) {
    MV m;
    m.N = (int)d.N; m.F = (int)d.F; m.lo = (int)d.own_lo; m.hi = (int)d.own_hi;
    m.c0 = d.face_c0; m.c1 = d.face_c1; m.fz = d.face_zone;
    m.area = d.face_area; m.fnx = d.fnx; m.fny = d.fny; m.fnz = d.fnz; m.fcx = d.fcx; m.fcy = d.fcy; m.fcz = d.fcz;
    m.vol = d.cvol; m.ccx = d.ccx; m.ccy = d.ccy; m.ccz = d.ccz;
    m.cf_ptr = d.cf_ptr; m.cf_face = d.cf_face; m.cf_nb = d.cf_nb; m.cf_slot = d.cf_slot; m.diag = d.diag;
    m.zt = d.zone_type; m.zs = d.zone_scalar; m.zv = d.zone_vec;
    return m;
}

template <class T>
static void up(Ctx& c, DBuf<T>& b, const std::vector<T>& h) {
    b.alloc(&c, std::max<size_t>(h.size(), 1));
    if (!h.empty()) ORC_CUDA(cudaMemcpyAsync(b.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, c.stream));
}

std::unique_ptr<DMesh> mesh_upload(Ctx& c, const HostMesh& m) {
    std::unique_ptr<DMesh> d(new DMesh());
    d->ctx = &c;
    d->N = m.n_cells; d->F = m.n_faces; d->S = (int64_t)m.cf_face.size(); d->nnz = m.nnz();
    d->nlevels = (int)m.level_ptr.size() - 1;
    d->own_lo = m.own_hi < 0 ? 0 : m.own_lo; d->own_hi = m.own_hi < 0 ? m.n_cells : m.own_hi;
    up(c, d->face_c0, m.face_c0); up(c, d->face_c1, m.face_c1); up(c, d->face_zone, m.face_zone);
    up(c, d->face_area, m.face_area);
    std::vector<double> t0(m.n_faces), t1(m.n_faces), t2(m.n_faces);
    for (int64_t f = 0; f < m.n_faces; ++f) { t0[f] = m.face_normal[3 * f]; t1[f] = m.face_normal[3 * f + 1]; t2[f] = m.face_normal[3 * f + 2]; }
    up(c, d->fnx, t0); up(c, d->fny, t1); up(c, d->fnz, t2);
    c.sync();
    for (int64_t f = 0; f < m.n_faces; ++f) { t0[f] = m.face_centroid[3 * f]; t1[f] = m.face_centroid[3 * f + 1]; t2[f] = m.face_centroid[3 * f + 2]; }
    up(c, d->fcx, t0); up(c, d->fcy, t1); up(c, d->fcz, t2);
    c.sync();
    t0.resize(m.n_cells); t1.resize(m.n_cells); t2.resize(m.n_cells);
    for (int64_t i = 0; i < m.n_cells; ++i) { t0[i] = m.cell_centroid[3 * i]; t1[i] = m.cell_centroid[3 * i + 1]; t2[i] = m.cell_centroid[3 * i + 2]; }
    up(c, d->ccx, t0); up(c, d->ccy, t1); up(c, d->ccz, t2);
    if (m.n_cells > 0) {
        const std::vector<double>* pl[3] = {&t0, &t1, &t2};
        for (int a = 0; a < 3; ++a) {
            const auto mm = std::minmax_element(pl[a]->begin(), pl[a]->end());
            d->cc_lo[a] = *mm.first; d->cc_hi[a] = *mm.second;
        }
    }
    up(c, d->cvol, m.cell_volume);
    up(c, d->cf_ptr, m.cf_ptr); up(c, d->cf_face, m.cf_face); up(c, d->cf_nb, m.cf_nb); up(c, d->cf_slot, m.cf_slot);
    up(c, d->rowptr, m.rowptr); up(c, d->col, m.col); up(c, d->diag, m.diag_idx);
    for (size_t r = 0; r + 1 < m.rowptr.size(); ++r) d->max_row = std::max(d->max_row, (int)(m.rowptr[r + 1] - m.rowptr[r]));
    up(c, d->level_ptr, m.level_ptr); up(c, d->level_order, m.level_order);
    for (int l = 0; l < d->nlevels; ++l) d->max_level_width = std::max(d->max_level_width, m.level_ptr[l + 1] - m.level_ptr[l]);
    c.sync();
    mesh_refresh_zones(c, *d, m);
    return d;
}

void mesh_refresh_zones(Ctx& c, DMesh& d, const HostMesh& m) {
    if (d.zone_epoch == m.zone_epoch) return;
    const size_t Z = m.zones.size();
    std::vector<int> zt(Z), sk(Z);
    std::vector<double> zs(Z), zv(3 * Z), sv(Z);
    for (size_t k = 0; k < Z; ++k) {
        zt[k] = m.zones[k].type; zs[k] = m.zones[k].scalar;
        zv[3 * k] = m.zones[k].vec[0]; zv[3 * k + 1] = m.zones[k].vec[1]; zv[3 * k + 2] = m.zones[k].vec[2];
        sk[k] = m.zones[k].scalar_bc_kind; sv[k] = m.zones[k].scalar_bc_value;
    }
    up(c, d.zone_type, zt); up(c, d.zone_scalar, zs); up(c, d.zone_vec, zv);
    up(c, d.zone_sbc_kind, sk); up(c, d.zone_sbc_value, sv);
    c.sync();
    d.nzones = (int)Z;
    d.zone_epoch = m.zone_epoch;
}

// -------------------------------------------------------------------------------------------------
// Mesh geometry on the device (src/io.rs:289-438, the same operator order as build_geometry in mesh_host.cpp through the shared
// vecmath.cuh, compiled without FMA contraction: bit-identical to the host pass). For multi-million-cell meshes: one thread per
// face (normal, centroid, triangle-fan area about the centroid), then one thread per cell (centroid = mean of its face centroids
// in ascending face order, volume = sum A |(f_c - c_c) . n| / dims).
// -------------------------------------------------------------------------------------------------
__global__ void k_face_geometry(int64_t F, int dims, const double* __restrict__ xyz, const long long* __restrict__ fptr, const int* __restrict__ fnodes,
                                const unsigned char* __restrict__ flipped, double* area, double* normal3, double* centroid3) {
    for (int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; f < F; f += (int64_t)gridDim.x * blockDim.x) {
        const long long p0 = fptr[f];
        const int cnt = (int)(fptr[f + 1] - p0);
        auto P = [&](int k) { const int n = fnodes[p0 + k]; return v3(xyz[3 * (size_t)n], xyz[3 * (size_t)n + 1], xyz[3 * (size_t)n + 2]); };
        V3 nrm;
        if (dims == 2) {
            const V3 t = vsub(P(1), P(0));
            nrm = (t.x == 0.) ? v3(1., -t.x / t.y, 0.) : v3(-t.y / t.x, 1., 0.);
            nrm = vunit(nrm);
        } else {
            nrm = vunit(vcross(vsub(P(2), P(1)), vsub(P(1), P(0))));
        }
        if (flipped[f]) nrm = vneg(nrm);
        V3 acc = vzero();
        for (int k = 0; k < cnt; ++k) acc = vadd(acc, P(k));
        const V3 cen = vdivs(acc, (double)cnt);
        double a;
        if (cnt == 2) {
            a = vnorm(vsub(P(1), P(0)));
        } else {
            auto tri = [](V3 p, V3 q, V3 r) { return fabs(vnorm(vcross(vsub(q, p), vsub(r, p)))) / 2.; };
            a = 0.;
            for (int k = 0; k + 1 < cnt; ++k) a = a + tri(cen, P(k), P(k + 1));
            a = a + tri(cen, P(0), P(cnt - 1));
        }
        area[f] = a;
        normal3[3 * f] = nrm.x; normal3[3 * f + 1] = nrm.y; normal3[3 * f + 2] = nrm.z;
        centroid3[3 * f] = cen.x; centroid3[3 * f + 1] = cen.y; centroid3[3 * f + 2] = cen.z;
    }
}
__global__ void k_cell_geometry(int64_t N, int dims, const int* __restrict__ cf_ptr, const int* __restrict__ cf_face, const double* __restrict__ area,
                                const double* __restrict__ normal3, const double* __restrict__ centroid3, double* volume, double* ccentroid3) {
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < N; c += (int64_t)gridDim.x * blockDim.x) {
        const int q0 = cf_ptr[c], q1 = cf_ptr[c + 1];
        V3 sum = vzero();
        for (int q = q0; q < q1; ++q) { const size_t f = (size_t)cf_face[q]; sum = vadd(sum, v3(centroid3[3 * f], centroid3[3 * f + 1], centroid3[3 * f + 2])); }
        const V3 cc = vdivs(sum, (double)(q1 - q0));
        double vol = 0.;
        for (int q = q0; q < q1; ++q) {
            const size_t f = (size_t)cf_face[q];
            const V3 fc = v3(centroid3[3 * f], centroid3[3 * f + 1], centroid3[3 * f + 2]);
            const V3 fn = v3(normal3[3 * f], normal3[3 * f + 1], normal3[3 * f + 2]);
            vol = vol + area[f] * fabs(vdot(vsub(fc, cc), fn)) / (double)dims;
        }
        volume[c] = vol;
        ccentroid3[3 * c] = cc.x; ccentroid3[3 * c + 1] = cc.y; ccentroid3[3 * c + 2] = cc.z;
    }
}
void mesh_geometry_device(Ctx& c, const HostMesh& m, double* face_area, double* face_normal3, double* face_centroid3, double* cell_volume,
                          double* cell_centroid3, double* device_ms) {
    ORC_REQUIRE(!m.xyz.empty() && !m.face_nodes.empty() && (int64_t)m.face_flipped.size() == m.n_faces, ORC_E_INVALID,
                "the mesh has no node coordinates (built from geometry or a partition): nothing to compute");
    const int64_t F = m.n_faces, N = m.n_cells;
    DBuf<double> xyz, area(&c, (size_t)F), nrm(&c, 3 * (size_t)F), cen(&c, 3 * (size_t)F), vol(&c, (size_t)N), cc(&c, 3 * (size_t)N);
    DBuf<long long> fptr(&c, (size_t)F + 1);
    DBuf<int> fnodes, cfp, cff;
    DBuf<unsigned char> flip;
    up(c, xyz, m.xyz); up(c, fnodes, m.face_nodes); up(c, cfp, m.cf_ptr); up(c, cff, m.cf_face); up(c, flip, m.face_flipped);
    static_assert(sizeof(long long) == sizeof(int64_t), "int64 layout");
    ORC_CUDA(cudaMemcpyAsync(fptr.p, m.face_node_ptr.data(), sizeof(int64_t) * ((size_t)F + 1), cudaMemcpyHostToDevice, c.stream));
    cudaEvent_t e0, e1;
    ORC_CUDA(cudaEventCreate(&e0)); ORC_CUDA(cudaEventCreate(&e1));
    ORC_CUDA(cudaEventRecord(e0, c.stream));
    k_face_geometry<<<grid_for(F, 128, c.sm_count * 16), 128, 0, c.stream>>>(F, m.dims, xyz, fptr, fnodes, flip, area, nrm, cen);
    c.after_launch("k_face_geometry");
    k_cell_geometry<<<grid_for(N, 128, c.sm_count * 16), 128, 0, c.stream>>>(N, m.dims, cfp, cff, area, nrm, cen, vol, cc);
    c.after_launch("k_cell_geometry");
    ORC_CUDA(cudaEventRecord(e1, c.stream));
    ORC_CUDA(cudaMemcpyAsync(face_area, area.p, sizeof(double) * F, cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(face_normal3, nrm.p, sizeof(double) * 3 * F, cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(face_centroid3, cen.p, sizeof(double) * 3 * F, cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(cell_volume, vol.p, sizeof(double) * N, cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(cell_centroid3, cc.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (device_ms) *device_ms = ms;
}

CsrPtr mesh_matrix(Ctx& c, const DMesh& d) {
    CsrPtr a(new DCsr());
    a->ctx = &c; a->nrows = a->ncols = d.N; a->nnz = d.nnz;
    a->rowptr = d.rowptr.p; a->col = d.col.p; a->diag = d.diag.p;
    a->own_pattern = false; a->own_diag = false; a->sym = 1; a->full_diag = 1; a->max_row = d.max_row; a->simplex = (d.max_row <= 5) ? 1 : 0;
    a->val = c.alloc_n<double>((size_t)std::max<int64_t>(d.nnz, 1));
    // where the unknowns sit: lets a Multigrid solve store its coarse levels along a space-filling curve (linalg.cu)
    a->hint.x = d.ccx.p; a->hint.y = d.ccy.p; a->hint.z = d.ccz.p; a->hint.n = d.N; a->hint.shift = 0;
    for (int k = 0; k < 3; ++k) {
        const double ext = d.cc_hi[k] - d.cc_lo[k];
        a->hint.lo[k] = d.cc_lo[k];
        a->hint.inv[k] = (ext > 0. && std::isfinite(ext)) ? 1024. / ext : 0.;
    }
    return a;
}

void validate_settings(const AsmSettings& s) {
    if (s.momentum != ORC_MOM_UD && s.momentum != ORC_MOM_CD1 && s.momentum != ORC_MOM_TVD)
        throw Error(ORC_E_UNSUPPORTED, "unsupported momentum scheme");                                   // discretization.rs:287
    if (s.momentum == ORC_MOM_TVD && (s.limiter < ORC_PSI_UD || s.limiter > ORC_PSI_UMIST)) throw Error(ORC_E_INVALID, "unknown TVD limiter");
    if (s.p_interp == ORC_P_STANDARD) throw Error(ORC_E_UNSUPPORTED, "`standard` pressure interpolation unsupported");  // solver.rs:1134-1137
    if (s.p_interp != ORC_P_LINEAR && s.p_interp != ORC_P_LINEAR_WEIGHTED && s.p_interp != ORC_P_SECOND_ORDER)
        throw Error(ORC_E_UNSUPPORTED, "unsupported pressure interpolation");                           // solver.rs:1145
    if (s.v_interp != ORC_V_LINEAR && s.v_interp != ORC_V_LINEAR_WEIGHTED && s.v_interp != ORC_V_RHIE_CHOW)
        throw Error(ORC_E_UNSUPPORTED, "`None` VelocityInterpolation cannot be used for interior faces");  // solver.rs:1097-1099
    if (s.gradient == ORC_G_GREEN_GAUSS_NODE) throw Error(ORC_E_UNSUPPORTED, "unsupported Green-Gauss scheme");  // solver.rs:901
    if (s.gradient != ORC_G_GREEN_GAUSS_CELL && s.gradient != ORC_G_LEAST_SQUARES) throw Error(ORC_E_UNSUPPORTED, "unsupported gradient scheme");  // solver.rs:870, 948
}

void AsmWork::ensure(Ctx& c, const DMesh& d, const AsmSettings& s) {
    const size_t N = (size_t)std::max<int64_t>(d.N, 1), F = (size_t)std::max<int64_t>(d.F, 1);
    if (gpx.n != N) { gpx.alloc(&c, N); gpy.alloc(&c, N); gpz.alloc(&c, N); pe.alloc(&c, 3 * N); gpx.zero(); gpy.zero(); gpz.zero(); pe.zero(); }
    if (pface.n != F) pface.alloc(&c, F);
    if (s.momentum == ORC_MOM_TVD && gu.n != 9 * N) gu.alloc(&c, 9 * N);
    if (s.assembly_mode == ORC_ASSEMBLY_FROZEN && du_old.n != N) { du_old.alloc(&c, N); dv_old.alloc(&c, N); dw_old.alloc(&c, N); }
}

// -------------------------------------------------------------------------------------------------
// face helpers (solver.rs)
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ V3 fnormal(const MV& m, int f) { return v3(m.fnx[f], m.fny[f], m.fnz[f]); }
__device__ __forceinline__ V3 fcentroid(const MV& m, int f) { return v3(m.fcx[f], m.fcy[f], m.fcz[f]); }
__device__ __forceinline__ V3 ccentroid(const MV& m, int c) { return v3(m.ccx[c], m.ccy[c], m.ccz[c]); }
__device__ __forceinline__ V3 outward(const MV& m, int f, int cell) {  // mesh.rs:216-222
    V3 n = fnormal(m, f);
    return (cell == m.c0[f]) ? n : vneg(n);
}
__device__ __forceinline__ V3 zvec(const MV& m, int z) { return v3(m.zv[3 * z], m.zv[3 * z + 1], m.zv[3 * z + 2]); }
__device__ __forceinline__ V3 vel(const double* u, const double* v, const double* w, int c) { return v3(u[c], v[c], w[c]); }

// get_face_pressure with PressureInterpolation::Linear (the Green-Gauss face value, solver.rs:887-894)
__device__ __forceinline__ double face_pressure_linear(const MV& m, const double* p, int f, int* flags) {
    const int z = m.fz[f], zt = m.zt[z];
    switch (zt) {
        case ORC_BC_SYMMETRY: case ORC_BC_WALL: case ORC_BC_VELOCITY_INLET: return p[m.c0[f]];
        case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: return m.zs[z];
        case ORC_BC_INTERIOR: return (p[m.c0[f]] + p[m.c1[f]]) * 0.5;
        default: atomicOr(flags, DF_UNSUPPORTED_BC); return 0.;
    }
}
// get_face_velocity with VelocityInterpolation::Linear / LinearWeighted / None (solver.rs:952-1003)
__device__ __forceinline__ V3 face_velocity(const MV& m, const double* u, const double* v, const double* w, int f, int interp, int* flags) {
    const int z = m.fz[f], zt = m.zt[z];
    const int c = m.c0[f];
    switch (zt) {
        case ORC_BC_WALL: case ORC_BC_VELOCITY_INLET: return zvec(m, z);
        case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: case ORC_BC_SYMMETRY: return vel(u, v, w, c);
        case ORC_BC_INTERIOR: {
            const int nb = m.c1[f];
            V3 vel0 = vel(u, v, w, c), vel1 = vel(u, v, w, nb);
            if (interp == ORC_V_LINEAR) return vdivs(vadd(vel0, vel1), 2.);
            double dx0 = vnorm(vsub(ccentroid(m, c), fcentroid(m, f)));
            double dx1 = vnorm(vsub(ccentroid(m, nb), fcentroid(m, f)));
            return vadd(vel0, vdivs(vmuls(vsub(vel1, vel0), dx0), dx0 + dx1));
        }
        default: atomicOr(flags, DF_UNSUPPORTED_BC); return vzero();
    }
}

// -------------------------------------------------------------------------------------------------
// K1: Green-Gauss cell-based grad p (solver.rs:874-902). `Float * Float * Vector`: the last product is the
// reference's Float*Vector operator, so .z receives the .y sum (Q1).
// -------------------------------------------------------------------------------------------------
__global__ void k_grad_p(MV m, const double* __restrict__ p, double* gx, double* gy, double* gz, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        V3 acc = vzero();
        const double vol = m.vol[i];
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            double fv = face_pressure_linear(m, p, f, flags);
            V3 term = smulv_q1(fv * (m.area[f] / vol), outward(m, f, i));
            acc = vadd(acc, term);
        }
        gx[i] = acc.x; gy[i] = acc.y; gz[i] = acc.z;
    }
}
// K2: Green-Gauss grad u (solver.rs:774-802), row-major 9 per cell in SoA planes: gu[k*N + i]
__global__ void k_grad_u(MV m, const double* __restrict__ u, const double* __restrict__ v, const double* __restrict__ w, double* gu, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        T3 acc; acc.x = vzero(); acc.y = vzero(); acc.z = vzero();
        const double vol = m.vol[i];
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            V3 fv = face_velocity(m, u, v, w, f, ORC_V_LINEAR, flags);
            acc = tadd(acc, vouter(fv, vmuls(outward(m, f, i), m.area[f] / vol)));
        }
        const size_t N = (size_t)m.N;
        gu[0 * N + i] = acc.x.x; gu[1 * N + i] = acc.x.y; gu[2 * N + i] = acc.x.z;
        gu[3 * N + i] = acc.y.x; gu[4 * N + i] = acc.y.y; gu[5 * N + i] = acc.y.z;
        gu[6 * N + i] = acc.z.x; gu[7 * N + i] = acc.z.y; gu[8 * N + i] = acc.z.z;
    }
}
// Least-squares gradients (solver.rs:903-947 and :803-869): one fit per cell over its faces in ascending face order. An interior
// face contributes (neighbour centroid - cell centroid, neighbour value - cell value); a boundary face contributes (face centroid -
// cell centroid, the boundary face VALUE) — not a difference: the reference's formula, kept. Normal equations and inverse follow
// nalgebra (vecmath.cuh Lsq3); a singular system is the reference's `.unwrap()` panic (DF_SINGULAR).
__global__ void k_grad_p_lsq(MV m, const double* __restrict__ p, double* gx, double* gy, double* gz, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        Lsq3<1> ls;
        ls.clear();
        const V3 cc = ccentroid(m, i);
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            V3 x; double b[1];
            if (m.zt[m.fz[f]] == ORC_BC_INTERIOR) {
                int nb = m.c0[f];
                if (nb == i) nb = m.c1[f];
                x = vsub(ccentroid(m, nb), cc);
                b[0] = p[nb] - p[i];
            } else {
                x = vsub(fcentroid(m, f), cc);
                b[0] = face_pressure_linear(m, p, f, flags);   // boundary faces: the interpolation scheme is never consulted
            }
            ls.add(x, b);
        }
        V3 g[1];
        if (!ls.solve(g)) { atomicOr(flags, DF_SINGULAR); g[0] = vzero(); }
        gx[i] = g[0].x; gy[i] = g[0].y; gz[i] = g[0].z;
    }
}
__global__ void k_grad_u_lsq(MV m, const double* __restrict__ u, const double* __restrict__ v, const double* __restrict__ w, double* gu, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        Lsq3<3> ls;
        ls.clear();
        const V3 cc = ccentroid(m, i);
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            V3 x; double b[3];
            if (m.zt[m.fz[f]] == ORC_BC_INTERIOR) {
                int nb = m.c0[f];
                if (nb == i) nb = m.c1[f];
                x = vsub(ccentroid(m, nb), cc);
                b[0] = u[nb] - u[i]; b[1] = v[nb] - v[i]; b[2] = w[nb] - w[i];
            } else {
                const V3 fv = face_velocity(m, u, v, w, f, ORC_V_NONE, flags);
                x = vsub(fcentroid(m, f), cc);
                b[0] = fv.x; b[1] = fv.y; b[2] = fv.z;
            }
            ls.add(x, b);
        }
        V3 g[3];
        if (!ls.solve(g)) { atomicOr(flags, DF_SINGULAR); g[0] = g[1] = g[2] = vzero(); }
        const size_t N = (size_t)m.N;
        gu[0 * N + i] = g[0].x; gu[1 * N + i] = g[0].y; gu[2 * N + i] = g[0].z;
        gu[3 * N + i] = g[1].x; gu[4 * N + i] = g[1].y; gu[5 * N + i] = g[1].z;
        gu[6 * N + i] = g[2].x; gu[7 * N + i] = g[2].y; gu[8 * N + i] = g[2].z;
    }
}
// face-parallel get_face_pressure (solver.rs:1104-1150): side independent, so evaluated once per face
__global__ void k_face_pressure(MV m, const double* __restrict__ p, const double* __restrict__ gx, const double* __restrict__ gy,
                                const double* __restrict__ gz, int interp, double* pf, int* flags) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < m.F; f += gridDim.x * blockDim.x) {
        const int z = m.fz[f], zt = m.zt[z];
        double r;
        switch (zt) {
            case ORC_BC_SYMMETRY: case ORC_BC_WALL: case ORC_BC_VELOCITY_INLET: r = p[m.c0[f]]; break;
            case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: r = m.zs[z]; break;
            case ORC_BC_INTERIOR: {
                const int c0 = m.c0[f], c1 = m.c1[f];
                if (interp == ORC_P_LINEAR) {
                    r = (p[c0] + p[c1]) * 0.5;
                } else if (interp == ORC_P_LINEAR_WEIGHTED) {
                    double x0 = vnorm(vsub(ccentroid(m, c0), fcentroid(m, f)));
                    double x1 = vnorm(vsub(ccentroid(m, c1), fcentroid(m, f)));
                    r = p[c0] + (p[c1] - p[c0]) * x0 / (x0 + x1);
                } else {  // SecondOrder
                    V3 g0 = v3(gx[c0], gy[c0], gz[c0]), g1 = v3(gx[c1], gy[c1], gz[c1]);
                    V3 r0 = vsub(fcentroid(m, f), ccentroid(m, c0));
                    V3 r1 = vsub(fcentroid(m, f), ccentroid(m, c1));
                    r = 0.5 * ((p[c0] + p[c1]) + (vdot(g0, r0) + vdot(g1, r1)));
                }
                break;
            }
            default: atomicOr(flags, DF_UNSUPPORTED_BC); r = 0.;
        }
        pf[f] = r;
    }
}

// get_face_flux (solver.rs:1007-1102) as seen from `cell`. di_* / dj_* are the momentum diagonals the
// reference would read through a_u.get(i,i): which state they are in (old/new) is the caller's business.
struct FluxIn {
    const double *u, *v, *w, *p, *gx, *gy, *gz;
    int v_interp;
};
template <bool COHERENT>
__device__ __forceinline__ double ld_diag(const double* d, int i) { return COHERENT ? __ldcg(d + i) : d[i]; }

template <bool COHERENT>
__device__ __forceinline__ double face_flux(const MV& m, const FluxIn& in, int f, int cell, V3 n, V3 diag_i, const double* du,
                                            const double* dv, const double* dw, int* flags) {
    const int z = m.fz[f], zt = m.zt[z];
    switch (zt) {
        case ORC_BC_WALL: case ORC_BC_SYMMETRY: return 0.;
        case ORC_BC_VELOCITY_INLET: case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET:
            return vdot(n, face_velocity(m, in.u, in.v, in.w, f, ORC_V_NONE, flags));
        case ORC_BC_INTERIOR: {
            if (in.v_interp != ORC_V_RHIE_CHOW) return vdot(n, face_velocity(m, in.u, in.v, in.w, f, in.v_interp, flags));
            int nb = m.c0[f];
            if (nb == cell) nb = m.c1[f];
            V3 vel_i = vel(in.u, in.v, in.w, cell), vel_j = vel(in.u, in.v, in.w, nb);
            V3 d = vsub(ccentroid(m, nb), ccentroid(m, cell));
            double a_i = vnorm(v3(diag_i.x * n.x, diag_i.y * n.y, diag_i.z * n.z));                     // discretization.rs:14-23
            V3 g_i = v3(in.gx[cell], in.gy[cell], in.gz[cell]), g_j = v3(in.gx[nb], in.gy[nb], in.gz[nb]);
            double vol_i = m.vol[cell], vol_j = m.vol[nb];
            const double p_i = in.p[cell], p_j = in.p[nb];
            double a_j = vnorm(v3(ld_diag<COHERENT>(du, nb) * n.x, ld_diag<COHERENT>(dv, nb) * n.y, ld_diag<COHERENT>(dw, nb) * n.z));
            double term_1 = vdot(vadd(vel_i, vel_j), n);
            double term_2 = (vol_i / a_i + vol_j / a_j) * (p_i - p_j) / vnorm(d);
            double term_3 = vdot(vadd(smulv_q1(vol_i / a_i, g_i), smulv_q1(vol_j / a_j, g_j)), vunit(d));  // Float * Vector: Q1
            return 0.5 * (term_1 + term_2 - term_3);
        }
        default: atomicOr(flags, DF_UNSUPPORTED_BC); return 0.;
    }
}

// TVD limiter functions psi(r) (lib.rs:107-118). Rust f64::min/max return the non-NaN operand == fmin/fmax.
__device__ __forceinline__ double psi(int limiter, double r) {
    switch (limiter) {
        case ORC_PSI_UD: return 0.;
        case ORC_PSI_CD1: return 1.;
        case ORC_PSI_LUD: return r;
        case ORC_PSI_QUICK: return (3. + r) / 4.;
        default: {  // UMIST
            double acc = INFINITY;
            acc = fmin(acc, 2. * r);
            acc = fmin(acc, (1. + 3. * r) / 4.);
            acc = fmin(acc, (3. + r) / 4.);
            acc = fmin(acc, 2.);
            return fmax(0., acc);
        }
    }
}

// -------------------------------------------------------------------------------------------------
// A1: build_momentum_diffusion_matrix (discretization.rs:39-131)
// -------------------------------------------------------------------------------------------------
__global__ void k_diffusion(MV m, double mu, double* val, double* bu, double* bv, double* bw, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        double a_p = 0., su = 0., sv = 0., sw = 0.;
        V3 cc = ccentroid(m, i);
        // duplicate (i, nb) pairs are summed by CsrMatrix::from(&Coo): clear the off-diagonals first
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = 0.;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int z = m.fz[f], zt = m.zt[z];
            double d_i;
            int slot = -1;
            switch (zt) {
                case ORC_BC_WALL: case ORC_BC_VELOCITY_INLET: {
                    d_i = mu * m.area[f] / vnorm(vsub(fcentroid(m, f), cc));
                    V3 src = vmuls(zvec(m, z), d_i);
                    su += src.x; sv += src.y; sw += src.z;
                    break;
                }
                case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: case ORC_BC_SYMMETRY: d_i = 0.; break;
                case ORC_BC_INTERIOR: {
                    int nb = m.c0[f];
                    if (nb == i) nb = m.c1[f];
                    V3 e_xi = vsub(ccentroid(m, nb), cc);
                    d_i = mu * m.area[f] / vnorm(e_xi);
                    slot = m.cf_slot[q];
                    break;
                }
                default: atomicOr(flags, DF_UNSUPPORTED_BC); d_i = 0.;
            }
            a_p += d_i;
            if (slot >= 0) val[slot] = val[slot] + (-d_i);
        }
        val[m.diag[i]] = a_p;
        bu[i] = su; bv[i] = sv; bw[i] = sw;
    }
}
void build_momentum_diffusion(Ctx& c, const DMesh& d, double mu, DCsr& a_di, double* b_u, double* b_v, double* b_w) {
    if (d.N == 0) return;
    k_diffusion<<<grid_for(d.N, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), mu, a_di.val, b_u, b_v, b_w, c.d_flags);
    c.after_launch("k_diffusion");
}

// A12: the Laplace system of initialize_pressure_field (solver.rs:437-494). a_nb = reciprocal(c_i - c_nb) . n_out * (A / V):
// the component-wise reciprocal (zero stays zero, lib.rs:244-252) is the reference's formula and is kept as it is.
__device__ __forceinline__ V3 vreciprocal(V3 a) { return v3(a.x != 0. ? 1. / a.x : 0., a.y != 0. ? 1. / a.y : 0., a.z != 0. ? 1. / a.z : 0.); }
__global__ void k_pressure_laplace(MV m, double* val, double* b) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        double a_p = 0., bi = 0.;
        const V3 cc = ccentroid(m, i);
        const double vol = m.vol[i];
        // duplicate (i, nb) pairs are summed by CsrMatrix::from(&Coo): clear the off-diagonals first
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = 0.;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int z = m.fz[f], zt = m.zt[z];
            const V3 n_out = outward(m, f, i);
            double a_nb, source;
            int slot = -1;
            switch (zt) {
                case ORC_BC_INTERIOR: {
                    int nb = m.c0[f];
                    if (nb == i) nb = m.c1[f];
                    a_nb = vdot(vreciprocal(vsub(cc, ccentroid(m, nb))), n_out) * (m.area[f] / vol);
                    source = 0.;
                    slot = m.cf_slot[q];
                    break;
                }
                case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET:
                    a_nb = vdot(vreciprocal(vsub(cc, fcentroid(m, f))), n_out) * (m.area[f] / vol);
                    source = a_nb * m.zs[z];
                    break;
                default: a_nb = 0.; source = 0.;  // Symmetry | Wall | any other zone type (solver.rs:476-485)
            }
            if (slot >= 0) val[slot] = val[slot] + (-a_nb);
            bi += source;
            a_p += a_nb;
        }
        val[m.diag[i]] = a_p;
        b[i] = bi;
    }
}
void build_pressure_laplace(Ctx& c, const DMesh& d, DCsr& a, double* b) {
    if (d.N == 0) return;
    k_pressure_laplace<<<grid_for(d.N, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), a.val, b);
    c.after_launch("k_pressure_laplace");
}

// A13: the potential system of initialize_velocity_field (solver.rs:524-590): grad psi = velocity. Interior faces as in the
// Laplace system above; VelocityInlet faces give the source -(zone velocity . n_out); a PressureOutlet face fixes psi = 0 on the
// face with the coefficient reciprocal(c_i - c_f) . n_out — WITHOUT the area / volume factor of the interior faces (:561-568, as
// written); walls, symmetry planes and every other zone type are natural boundaries.
__global__ void k_velocity_potential(MV m, double* val, double* b) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        double a_p = 0., bi = 0.;
        const V3 cc = ccentroid(m, i);
        const double vol = m.vol[i];
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = 0.;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int z = m.fz[f], zt = m.zt[z];
            const V3 n_out = outward(m, f, i);
            double a_nb, source;
            int slot = -1;
            switch (zt) {
                case ORC_BC_INTERIOR: {
                    int nb = m.c0[f];
                    if (nb == i) nb = m.c1[f];
                    a_nb = vdot(vreciprocal(vsub(cc, ccentroid(m, nb))), n_out) * (m.area[f] / vol);
                    source = 0.;
                    slot = m.cf_slot[q];
                    break;
                }
                case ORC_BC_VELOCITY_INLET: a_nb = 0.; source = -vdot(zvec(m, z), n_out); break;
                case ORC_BC_PRESSURE_OUTLET: a_nb = vdot(vreciprocal(vsub(cc, fcentroid(m, f))), n_out); source = 0.; break;
                default: a_nb = 0.; source = 0.;
            }
            if (slot >= 0) val[slot] = val[slot] + (-a_nb);
            bi += source;
            a_p += a_nb;
        }
        val[m.diag[i]] = a_p;
        b[i] = bi;
    }
}
void build_velocity_potential(Ctx& c, const DMesh& d, DCsr& a, double* b) {
    if (d.N == 0) return;
    k_velocity_potential<<<grid_for(d.N, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), a.val, b);
    c.after_launch("k_velocity_potential");
}
// The cell velocity as the least-squares gradient of psi over the cell NEIGHBOURS only (solver.rs:624-693): columns of the
// neighbour-offset matrix that are entirely zero are dropped before the normal equations (a one-cell-thick mesh has no z
// differences), so the system is 3 x 3, 2 x 2 or 1 x 1; a singular one leaves the cell at zero, NaN components become zero.
__global__ void k_potential_gradient(MV m, const double* __restrict__ psi, double* u, double* v, double* w) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        const V3 cc = ccentroid(m, i);
        bool nz[3] = {false, false, false};
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            if (m.c1[f] < 0) continue;   // faces with two cells only (:631)
            const int nb = (m.c0[f] != i) ? m.c0[f] : m.c1[f];
            const V3 dx = vsub(ccentroid(m, nb), cc);
            if (dx.x != 0.) nz[0] = true;
            if (dx.y != 0.) nz[1] = true;
            if (dx.z != 0.) nz[2] = true;
        }
        int idx[3], nsel = 0;
        for (int a = 0; a < 3; ++a) if (nz[a]) idx[nsel++] = a;
        double cmat[3][3], rhs[3];
        for (int a = 0; a < 3; ++a) { rhs[a] = 0.; for (int b2 = 0; b2 < 3; ++b2) cmat[a][b2] = 0.; }
        int rows = 0;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            if (m.c1[f] < 0) continue;
            const int nb = (m.c0[f] != i) ? m.c0[f] : m.c1[f];
            const V3 dx = vsub(ccentroid(m, nb), cc);
            const double d3[3] = {dx.x, dx.y, dx.z};
            const double dpsi = psi[nb] - psi[i];
            for (int a = 0; a < nsel; ++a) {
                for (int b2 = 0; b2 < nsel; ++b2) { const double t = d3[idx[a]] * d3[idx[b2]]; cmat[a][b2] = rows == 0 ? t : t + cmat[a][b2]; }
                const double t = d3[idx[a]] * dpsi;
                rhs[a] = rows == 0 ? t : t + rhs[a];
            }
            ++rows;
        }
        double vel[3] = {0., 0., 0.};
        double inv[3][3];
        if (nsel > 0 && inv_n(nsel, cmat, inv)) {
            for (int a = 0; a < nsel; ++a) {
                double acc = inv[a][0] * rhs[0];
                for (int b2 = 1; b2 < nsel; ++b2) acc = inv[a][b2] * rhs[b2] + acc;
                vel[a] = acc;
            }
        }
        double out[3] = {0., 0., 0.};
        for (int a = 0; a < nsel; ++a) out[idx[a]] = vel[a];
        u[i] = (out[0] != out[0]) ? 0. : out[0];
        v[i] = (out[1] != out[1]) ? 0. : out[1];
        w[i] = (out[2] != out[2]) ? 0. : out[2];
    }
}
void potential_gradient(Ctx& c, const DMesh& d, const double* psi, double* u, double* v, double* w) {
    if (d.N == 0) return;
    k_potential_gradient<<<grid_for(d.N, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), psi, u, v, w);
    c.after_launch("k_potential_gradient");
}

// A2: initialize_momentum_matrix (discretization.rs:450-472): diag 1, off-diagonals -1/(#faces of the cell)
__global__ void k_init_momentum(MV m, double* val) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        const int q0 = m.cf_ptr[i], q1 = m.cf_ptr[i + 1];
        const double nf = (double)(q1 - q0);
        for (int q = q0; q < q1; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = 0.;
        for (int q = q0; q < q1; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = val[m.cf_slot[q]] + (-1. / nf);
        val[m.diag[i]] = 1.;
    }
}
void init_momentum_matrix(Ctx& c, const DMesh& d, DCsr& a) {
    if (d.N == 0) return;
    k_init_momentum<<<grid_for(d.N, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), a.val);
    c.after_launch("k_init_momentum");
}

// calculate_pressure_gradient / calculate_velocity_gradient for every cell with the selected reconstruction (solver.rs:774-949)
static void launch_grad_p(Ctx& c, const MV& m, int gradient, const double* p, double* gx, double* gy, double* gz) {
    const int g = grid_for(m.N, 128, c.sm_count * 16);
    if (gradient == ORC_G_LEAST_SQUARES) k_grad_p_lsq<<<g, 128, 0, c.stream>>>(m, p, gx, gy, gz, c.d_flags);
    else k_grad_p<<<g, 128, 0, c.stream>>>(m, p, gx, gy, gz, c.d_flags);
    c.after_launch("k_grad_p");
}
static void launch_grad_u(Ctx& c, const MV& m, int gradient, const double* u, const double* v, const double* w, double* gu) {
    const int g = grid_for(m.N, 128, c.sm_count * 16);
    if (gradient == ORC_G_LEAST_SQUARES) k_grad_u_lsq<<<g, 128, 0, c.stream>>>(m, u, v, w, gu, c.d_flags);
    else k_grad_u<<<g, 128, 0, c.stream>>>(m, u, v, w, gu, c.d_flags);
    c.after_launch("k_grad_u");
}
void pressure_gradient(Ctx& c, const DMesh& d, const double* p, double* gx, double* gy, double* gz, int gradient) {
    if (d.N == 0) return;
    launch_grad_p(c, view(d), gradient, p, gx, gy, gz);
}
void velocity_gradient(Ctx& c, const DMesh& d, const double* u, const double* v, const double* w, double* gu9, int gradient) {
    if (d.N == 0) return;
    launch_grad_u(c, view(d), gradient, u, v, w, gu9);
}

// -------------------------------------------------------------------------------------------------
// A3: build_momentum_advection_matrices (discretization.rs:134-356), one cell.
// -------------------------------------------------------------------------------------------------
struct MomArgs {
    MV m;
    FluxIn in;
    const double* pface;
    const double* gu;
    const double* adi;          // a_di values
    double *au, *av, *aw;       // coefficient values of a_u / a_v / a_w
    const double *du_in, *dv_in, *dw_in;  // diagonals read for neighbours (== du_out in exact mode)
    double *du_out, *dv_out, *dw_out;
    double *bu, *bv, *bw;
    double* pe;                 // 3 N Peclet components
    int momentum, limiter;
    double rho;
    int* flags;
};

// The advective neighbour coefficient a_nb of one face (discretization.rs:217-286), shared by the one-thread and the eight-lane
// cell below: UD, CD1, or TVD(psi) with the reference's `Float * Vector` products (Q1). `nb` < 0: boundary face.
__device__ __forceinline__ V3 neighbour_coefficient(const MomArgs& a, int i, int nb, double f_i, V3 cvel) {
    const MV& m = a.m;
    V3 a_nb;
    if (a.momentum == ORC_MOM_UD) {
        a_nb = smulv_q1(fmin(f_i, 0.), v3(1., 1., 1.));
    } else if (a.momentum == ORC_MOM_CD1) {
        a_nb = vdivs(smulv_q1(f_i, v3(1., 1., 1.)), 2.);
    } else {  // TVD(psi), discretization.rs:233-286
        if (nb < 0) {
            a_nb = smulv_q1(fmin(f_i, 0.), v3(1., 1., 1.));
        } else {
            const int downstream = f_i > 0. ? nb : i;
            const V3 dvel = vel(a.in.u, a.in.v, a.in.w, downstream);
            const V3 dv_ = vsub(dvel, cvel);
            if (vnorm(dv_) == 0.) {
                a_nb = vdivs(smulv_q1(f_i, v3(1., 1., 1.)), 2.);
            } else {
                const size_t N = (size_t)m.N;
                T3 g;
                g.x = v3(a.gu[0 * N + i], a.gu[1 * N + i], a.gu[2 * N + i]);
                g.y = v3(a.gu[3 * N + i], a.gu[4 * N + i], a.gu[5 * N + i]);
                g.z = v3(a.gu[6 * N + i], a.gu[7 * N + i], a.gu[8 * N + i]);
                const V3 r_pa = vsub(ccentroid(m, nb), ccentroid(m, i));
                const V3 r = vsubs(vdivv(smulv_q1(2., tinner(g, r_pa)), dv_), 1.);            // `2. * Vector`: Q1
                a_nb = vdivs(smulv_q1(f_i, v3(psi(a.limiter, r.x), psi(a.limiter, r.y), psi(a.limiter, r.z))), 2.);  // Q1 again
            }
        }
    }
    return a_nb;
}

template <bool COHERENT>
__device__ __forceinline__ void momentum_cell(const MomArgs& a, int i) {
    const MV& m = a.m;
    V3 s_u = vzero();                      // get_momentum_source_term == 0 (solver.rs:698-701)
    const V3 s_u_dc = vzero(), s_d_cross = vzero();
    const int di = m.diag[i];
    const double a_ii_di = a.adi[di];
    V3 a_p = vzero();
    // own diagonal: still the OLD value while this cell's faces are processed (written at :340-351)
    const V3 diag_i = v3(ld_diag<COHERENT>(a.du_in, i), ld_diag<COHERENT>(a.dv_in, i), ld_diag<COHERENT>(a.dw_in, i));
    const V3 cvel = vel(a.in.u, a.in.v, a.in.w, i);
    for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
        const int f = m.cf_face[q];
        const int nb = m.cf_nb[q];
        const V3 n_out = outward(m, f, i);
        const double area = m.area[f];
        const double face_flux_v = face_flux<COHERENT>(m, a.in, f, i, n_out, diag_i, a.du_in, a.dv_in, a.dw_in, a.flags);
        const double f_i = face_flux_v * area * a.rho;
        const double face_pressure = a.pface[f];
        const V3 a_nb = neighbour_coefficient(a, i, nb, f_i, cvel);
        a_p = vadd(a_p, vadds(vneg(a_nb), f_i));
        s_u = vadd(s_u, vmuls(vmuls(vneg(n_out), face_pressure), area));
        if (nb < 0) {
            const int z = m.fz[f], zt = m.zt[z];
            if (zt == ORC_BC_WALL || zt == ORC_BC_VELOCITY_INLET) {
                const V3 bc = zvec(m, z);
                s_u = vadd(s_u, v3((a_nb.x - f_i) * bc.x, (a_nb.y - f_i) * bc.y, (a_nb.z - f_i) * bc.z));
            } else {
                s_u = vadd(s_u, vzero());
            }
        } else {
            const int slot = m.cf_slot[q];
            const double a_ij_di = a.adi[slot];
            a.au[slot] = a_nb.x + a_ij_di;
            a.av[slot] = a_nb.y + a_ij_di;
            a.aw[slot] = a_nb.z + a_ij_di;
        }
    }
    const V3 source_total = vadd(vadd(s_u, s_u_dc), s_d_cross);
    a.bu[i] = source_total.x; a.bv[i] = source_total.y; a.bw[i] = source_total.z;
    const size_t N = (size_t)m.N;
    a.pe[i] = a_p.x / a_ii_di; a.pe[N + i] = a_p.y / a_ii_di; a.pe[2 * N + i] = a_p.z / a_ii_di;
    const double nu_ = a_p.x + a_ii_di, nv_ = a_p.y + a_ii_di, nw_ = a_p.z + a_ii_di;
    a.au[di] = nu_; a.av[di] = nv_; a.aw[di] = nw_;
    if (COHERENT) { __stcg(a.du_out + i, nu_); __stcg(a.dv_out + i, nv_); __stcg(a.dw_out + i, nw_); }
    else { a.du_out[i] = nu_; a.dv_out[i] = nv_; a.dw_out[i] = nw_; }
}

// The same cell with EIGHT lanes: lane k computes face k's flux and coefficients (the loads of the faces overlap instead
// of forming one chain per thread: the level kernel below is latency bound, 382 dependent levels at 128^3), then every lane
// of the group replays the reference's accumulation over the faces in ascending order from shuffled values — the sums are
// the sequential sums, bit for bit. `gmask`: the group's eight lanes, `gl`: lane within the group.
template <bool COHERENT>
__device__ __forceinline__ void momentum_cell8(const MomArgs& a, int i, unsigned gmask, int gl) {
    const MV& m = a.m;
    V3 s_u = vzero();                      // get_momentum_source_term == 0 (solver.rs:698-701)
    const V3 s_u_dc = vzero(), s_d_cross = vzero();
    const int di = m.diag[i];
    const double a_ii_di = a.adi[di];
    V3 a_p = vzero();
    const V3 diag_i = v3(ld_diag<COHERENT>(a.du_in, i), ld_diag<COHERENT>(a.dv_in, i), ld_diag<COHERENT>(a.dw_in, i));
    const V3 cvel = vel(a.in.u, a.in.v, a.in.w, i);
    const int q0 = m.cf_ptr[i], q1 = m.cf_ptr[i + 1];
    for (int base = q0; base < q1; base += 8) {
        const int q = base + gl;
        // per-face terms of this lane (kind: 0 interior, 1 wall / velocity inlet, 2 other boundary, -1 no face)
        double f_i = 0.;
        V3 a_nb = vzero(), press = vzero(), bct = vzero();
        int kind = -1;
        if (q < q1) {
            const int f = m.cf_face[q];
            const int nb = m.cf_nb[q];
            const V3 n_out = outward(m, f, i);
            const double area = m.area[f];
            const double face_flux_v = face_flux<COHERENT>(m, a.in, f, i, n_out, diag_i, a.du_in, a.dv_in, a.dw_in, a.flags);
            f_i = face_flux_v * area * a.rho;
            const double face_pressure = a.pface[f];
            a_nb = neighbour_coefficient(a, i, nb, f_i, cvel);
            press = vmuls(vmuls(vneg(n_out), face_pressure), area);
            if (nb < 0) {
                const int z = m.fz[f], zt = m.zt[z];
                if (zt == ORC_BC_WALL || zt == ORC_BC_VELOCITY_INLET) {
                    const V3 bc = zvec(m, z);
                    bct = v3((a_nb.x - f_i) * bc.x, (a_nb.y - f_i) * bc.y, (a_nb.z - f_i) * bc.z);
                    kind = 1;
                } else {
                    kind = 2;
                }
            } else {
                kind = 0;
                const int slot = m.cf_slot[q];
                const double a_ij_di = a.adi[slot];
                a.au[slot] = a_nb.x + a_ij_di;
                a.av[slot] = a_nb.y + a_ij_di;
                a.aw[slot] = a_nb.z + a_ij_di;
            }
        }
        // the reference's accumulation, face by face in ascending order (every lane of the group computes the same sums)
        const int nfac = min(8, q1 - base);
        for (int k = 0; k < nfac; ++k) {
            const double fk = __shfl_sync(gmask, f_i, k, 8);
            const V3 ak = v3(__shfl_sync(gmask, a_nb.x, k, 8), __shfl_sync(gmask, a_nb.y, k, 8), __shfl_sync(gmask, a_nb.z, k, 8));
            const V3 pk = v3(__shfl_sync(gmask, press.x, k, 8), __shfl_sync(gmask, press.y, k, 8), __shfl_sync(gmask, press.z, k, 8));
            const V3 bk = v3(__shfl_sync(gmask, bct.x, k, 8), __shfl_sync(gmask, bct.y, k, 8), __shfl_sync(gmask, bct.z, k, 8));
            const int kk = __shfl_sync(gmask, kind, k, 8);
            a_p = vadd(a_p, vadds(vneg(ak), fk));
            s_u = vadd(s_u, pk);
            if (kk == 1) s_u = vadd(s_u, bk);
            else if (kk == 2) s_u = vadd(s_u, vzero());
        }
    }
    if (gl != 0) return;
    const V3 source_total = vadd(vadd(s_u, s_u_dc), s_d_cross);
    a.bu[i] = source_total.x; a.bv[i] = source_total.y; a.bw[i] = source_total.z;
    const size_t N = (size_t)m.N;
    a.pe[i] = a_p.x / a_ii_di; a.pe[N + i] = a_p.y / a_ii_di; a.pe[2 * N + i] = a_p.z / a_ii_di;
    const double nu_ = a_p.x + a_ii_di, nv_ = a_p.y + a_ii_di, nw_ = a_p.z + a_ii_di;
    a.au[di] = nu_; a.av[di] = nv_; a.aw[di] = nw_;
    if (COHERENT) { __stcg(a.du_out + i, nu_); __stcg(a.dv_out + i, nv_); __stcg(a.dw_out + i, nw_); }
    else { a.du_out[i] = nu_; a.dv_out[i] = nv_; a.dw_out[i] = nw_; }
}

// Exact mode: cells grouped by dependency level (level(i) = 1 + max level of neighbours j < i); one
// cooperative launch walks the levels with a grid barrier in between, so cell i sees NEW diagonals of
// every neighbour j < i and OLD ones of j > i — the reference's sequential in-place order (Q2).
__global__ void __launch_bounds__(128) k_momentum_levels(MomArgs a, const int* __restrict__ level_ptr, const int* __restrict__ level_order,
                                                         int nlevels) {
    cg::grid_group grid = cg::this_grid();
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    const int gl = threadIdx.x & 7;
    const unsigned gmask = 0xffu << (threadIdx.x & 24);   // this thread's group of eight lanes within its warp
    for (int L = 0; L < nlevels; ++L) {
        const int b = level_ptr[L], e = level_ptr[L + 1];
        for (int idx = b + (gtid >> 3); idx < e; idx += (gsz >> 3)) momentum_cell8<true>(a, level_order[idx], gmask, gl);
        grid.sync();
    }
}
// No recurrence (Linear / LinearWeighted face velocity, or frozen mode): plain cell-parallel launch.
__global__ void __launch_bounds__(128) k_momentum_flat(MomArgs a) {
    for (int i = a.m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < a.m.hi; i += gridDim.x * blockDim.x) momentum_cell<false>(a, i);
}

// Peclet statistics (discretization.rs:331-338): avg of per-cell means, min/max by f64::total_cmp.
__device__ __forceinline__ long long total_key(double x) {
    long long b = __double_as_longlong(x);
    return b ^ (long long)(((unsigned long long)(b >> 63)) >> 1);
}
__device__ __forceinline__ double key_to_double(long long k) {
    return __longlong_as_double(k ^ (long long)(((unsigned long long)(k >> 63)) >> 1));
}
__global__ void k_peclet(int N, int lo, int hi, const double* __restrict__ pe, double* partials, unsigned int* counter, double* out3) {
    // out3 = {sum of per-cell means (NOT yet divided by the cell count), min, max} over the owned cells
    __shared__ double sh[32];
    __shared__ long long shk[32];
    double avg = 0.;
    long long kmin = total_key(INFINITY), kmax = total_key(-INFINITY);
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        double x = pe[i], y = pe[(size_t)N + i], z = pe[2 * (size_t)N + i];
        avg += (((0. + x) + y) + z) / 3.;
        long long kx = total_key(x), ky = total_key(y), kz = total_key(z);
        kmin = min(kmin, min(kx, min(ky, kz)));
        kmax = max(kmax, max(kx, max(ky, kz)));
    }
    double s = block_sum(avg, sh);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    for (int o = 16; o > 0; o >>= 1) { kmin = min(kmin, __shfl_down_sync(0xffffffffu, kmin, o)); kmax = max(kmax, __shfl_down_sync(0xffffffffu, kmax, o)); }
    __syncthreads();
    if (lane == 0) shk[wid] = kmin;
    __syncthreads();
    if (threadIdx.x == 0) { long long r = shk[0]; for (int q = 1; q < nw; ++q) r = min(r, shk[q]); partials[Ctx::kMaxBlocks + blockIdx.x] = __longlong_as_double(r); }
    __syncthreads();
    if (lane == 0) shk[wid] = kmax;
    __syncthreads();
    if (threadIdx.x == 0) { long long r = shk[0]; for (int q = 1; q < nw; ++q) r = max(r, shk[q]); partials[2 * Ctx::kMaxBlocks + blockIdx.x] = __longlong_as_double(r); partials[blockIdx.x] = s; }
    if (last_block_done(counter)) {
        double T = sum_partials(partials, gridDim.x, sh);
        if (threadIdx.x == 0) {
            long long mn = __double_as_longlong(partials[Ctx::kMaxBlocks]), mx = __double_as_longlong(partials[2 * Ctx::kMaxBlocks]);
            for (int q = 1; q < (int)gridDim.x; ++q) {
                mn = min(mn, __double_as_longlong(__ldcg(partials + Ctx::kMaxBlocks + q)));
                mx = max(mx, __double_as_longlong(__ldcg(partials + 2 * Ctx::kMaxBlocks + q)));
            }
            out3[0] = T;
            out3[1] = key_to_double(mn);
            out3[2] = key_to_double(mx);
        }
    }
}

void build_momentum_advection(Ctx& c, const DMesh& d, AsmWork& w, const AsmSettings& s, double rho, DCsr& a_u, DCsr& a_v, DCsr& a_w,
                              const DCsr& a_di, double* du, double* dv, double* dw, const double* u, const double* v, const double* wv,
                              const double* p, double* b_u, double* b_v, double* b_w, double* peclet3_dev) {
    validate_settings(s);
    if (d.N == 0) return;
    w.ensure(c, d, s);
    const MV m = view(d);
    const int cg_ = grid_for(d.N, 128, c.sm_count * 16), fg = grid_for(d.F, 128, c.sm_count * 16);
    const bool need_gradp = (s.v_interp == ORC_V_RHIE_CHOW) || (s.p_interp == ORC_P_SECOND_ORDER);
    if (need_gradp) {
        launch_grad_p(c, m, s.gradient, p, w.gpx, w.gpy, w.gpz);
        if (w.halo_exchange) { double* g[3] = {w.gpx.p, w.gpy.p, w.gpz.p}; w.halo_exchange(g, 3); }  // neighbours' grad p (Rhie-Chow, SecondOrder)
    }
    if (s.momentum == ORC_MOM_TVD) launch_grad_u(c, m, s.gradient, u, v, wv, w.gu);
    k_face_pressure<<<fg, 128, 0, c.stream>>>(m, p, w.gpx, w.gpy, w.gpz, s.p_interp, w.pface, c.d_flags);
    c.after_launch("k_face_pressure");

    MomArgs a;
    a.m = m;
    a.in.u = u; a.in.v = v; a.in.w = wv; a.in.p = p; a.in.gx = w.gpx; a.in.gy = w.gpy; a.in.gz = w.gpz; a.in.v_interp = s.v_interp;
    a.pface = w.pface; a.gu = w.gu; a.adi = a_di.val;
    a.au = a_u.val; a.av = a_v.val; a.aw = a_w.val;
    a.du_out = du; a.dv_out = dv; a.dw_out = dw;
    a.bu = b_u; a.bv = b_v; a.bw = b_w; a.pe = w.pe;
    a.momentum = s.momentum; a.limiter = s.limiter; a.rho = rho; a.flags = c.d_flags;
    const bool recurrence = (s.v_interp == ORC_V_RHIE_CHOW);
    if (recurrence && s.assembly_mode == ORC_ASSEMBLY_EXACT) {
        a.du_in = du; a.dv_in = dv; a.dw_in = dw;
        int per_sm = 0;
        ORC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_momentum_levels, 128, 0));
        ORC_REQUIRE(per_sm > 0, ORC_E_CUDA, "k_momentum_levels cannot be made resident");
        int grid = std::min(per_sm * c.sm_count, std::max(1, (8 * d.max_level_width + 127) / 128));   // eight lanes per cell
        const int* lp = d.level_ptr.p;
        const int* lo = d.level_order.p;
        int nl = d.nlevels;
        void* args[] = {(void*)&a, (void*)&lp, (void*)&lo, (void*)&nl};
        ORC_CUDA(cudaLaunchCooperativeKernel((void*)k_momentum_levels, dim3(grid), dim3(128), args, 0, c.stream));
        c.after_launch("k_momentum_levels");
    } else {
        if (recurrence) {  // frozen: every face sees the previous iteration's diagonals
            ORC_CUDA(cudaMemcpyAsync(w.du_old.p, du, sizeof(double) * d.N, cudaMemcpyDeviceToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(w.dv_old.p, dv, sizeof(double) * d.N, cudaMemcpyDeviceToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(w.dw_old.p, dw, sizeof(double) * d.N, cudaMemcpyDeviceToDevice, c.stream));
            a.du_in = w.du_old; a.dv_in = w.dv_old; a.dw_in = w.dw_old;
        } else {
            a.du_in = du; a.dv_in = dv; a.dw_in = dw;  // never read for neighbours
        }
        k_momentum_flat<<<cg_, 128, 0, c.stream>>>(a);
        c.after_launch("k_momentum_flat");
    }
    if (peclet3_dev) {
        k_peclet<<<grid_for(d.N, 256, c.sm_count * 4), 256, 0, c.stream>>>((int)d.N, (int)d.own_lo, (int)d.own_hi, w.pe, c.d_partials, c.d_counter, peclet3_dev);
        c.after_launch("k_peclet");
    }
}

// -------------------------------------------------------------------------------------------------
// A4: build_pressure_correction_matrices (discretization.rs:359-448). No recurrence: reads only.
// The reference rebuilds COO -> CSR every iteration; here values go straight into the fixed pattern.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_pressure_correction(MV m, FluxIn in, const double* __restrict__ du, const double* __restrict__ dv,
                                                             const double* __restrict__ dw, double rho, double* val, double* b, int* flags) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        double a_p = 0., b_p = 0.;
        const V3 diag_i = v3(du[i], dv[i], dw[i]);
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) if (m.cf_slot[q] >= 0) val[m.cf_slot[q]] = 0.;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int nb = m.cf_nb[q];
            const V3 n_out = outward(m, f, i);
            const double area = m.area[f];
            const double flux = face_flux<false>(m, in, f, i, n_out, diag_i, du, dv, dw, flags);
            const V3 n_in = vmuls(n_out, -1.);  // get_inward_face_normal = outward * -1. (mesh.rs:224-226)
            b_p += rho * (-flux) * area;
            if (nb >= 0) {
                const double a_mag = 0.5 * vnorm(v3((diag_i.x + du[nb]) * n_in.x, (diag_i.y + dv[nb]) * n_in.y, (diag_i.z + dw[nb]) * n_in.z));
                const double a_nb = rho * (area * area) / a_mag;
                const int slot = m.cf_slot[q];
                val[slot] = val[slot] + (-a_nb);
                a_p += a_nb;
            } else {
                const double a_ii_norm = vnorm(v3(diag_i.x * n_in.x, diag_i.y * n_in.y, diag_i.z * n_in.z));
                const double a_nb = rho * (area * area) / a_ii_norm;
                a_p += a_nb / 2.;
            }
        }
        val[m.diag[i]] = a_p;
        b[i] = b_p;
    }
}
void build_pressure_correction(Ctx& c, const DMesh& d, AsmWork& w, const AsmSettings& s, double rho, const double* du, const double* dv,
                               const double* dw, const double* u, const double* v, const double* wv, const double* p, DCsr& a, double* b) {
    validate_settings(s);
    if (d.N == 0) return;
    w.ensure(c, d, s);
    const MV m = view(d);
    const int cg_ = grid_for(d.N, 128, c.sm_count * 16);
    if (s.v_interp == ORC_V_RHIE_CHOW) {  // u, v, w changed since the momentum assembly but p did not: grad p could be
        launch_grad_p(c, m, s.gradient, p, w.gpx, w.gpy, w.gpz);  // reused; recomputed so the entry is self-contained
        if (w.halo_exchange) { double* g[3] = {w.gpx.p, w.gpy.p, w.gpz.p}; w.halo_exchange(g, 3); }
    }
    FluxIn in;
    in.u = u; in.v = v; in.w = wv; in.p = p; in.gx = w.gpx; in.gy = w.gpy; in.gz = w.gpz; in.v_interp = s.v_interp;
    k_pressure_correction<<<cg_, 128, 0, c.stream>>>(m, in, du, dv, dw, rho, a.val, b, c.d_flags);
    c.after_launch("k_pressure_correction");
}

// -------------------------------------------------------------------------------------------------
// A10: apply_pressure_correction (solver.rs:1170-1227) + the field sums of solver.rs:206-208
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_apply_correction(MV m, const double* __restrict__ du, const double* __restrict__ dv,
                                                          const double* __restrict__ dw, const double* __restrict__ pp, double* u, double* v,
                                                          double* w, double* p, double p_relax, double u_relax, double* partials,
                                                          unsigned int* counter, double* out8, int* flags) {
    __shared__ double sh[32];
    double s_pp = 0., s_vc = 0., s_u = 0., s_v = 0., s_w = 0.;
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        const double ppi = pp[i];
        p[i] = p[i] + p_relax * ppi;
        V3 acc = vzero();
        const double aui = du[i], avi = dv[i], awi = dw[i];
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int zt = m.zt[m.fz[f]];
            const V3 n = outward(m, f, i);
            double pn;
            switch (zt) {
                case ORC_BC_WALL: case ORC_BC_SYMMETRY: case ORC_BC_VELOCITY_INLET: pn = ppi; break;
                case ORC_BC_PRESSURE_INLET: case ORC_BC_PRESSURE_OUTLET: pn = 0.; break;
                case ORC_BC_INTERIOR: pn = pp[(m.c0[f] == i) ? m.c1[f] : m.c0[f]]; break;
                default: atomicOr(flags, DF_UNSUPPORTED_BC); pn = 0.;
            }
            const V3 scaled = v3(n.x / aui, n.y / avi, n.z / awi);
            acc = vadd(acc, vmuls(vmuls(scaled, ppi - pn), m.area[f]));
        }
        const double un = u[i] + acc.x * u_relax, vn = v[i] + acc.y * u_relax, wn = w[i] + acc.z * u_relax;
        u[i] = un; v[i] = vn; w[i] = wn;
        const double nn = vnorm(acc);
        s_vc += nn * nn;     // velocity_correction.norm().powi(2)
        s_pp += ppi * ppi;   // p_prime.norm()
        s_u += un; s_v += vn; s_w += wn;
    }
    double r;
    r = block_sum(s_pp, sh); if (threadIdx.x == 0) partials[blockIdx.x] = r;
    r = block_sum(s_vc, sh); if (threadIdx.x == 0) partials[Ctx::kMaxBlocks + blockIdx.x] = r;
    r = block_sum(s_u, sh);  if (threadIdx.x == 0) partials[2 * Ctx::kMaxBlocks + blockIdx.x] = r;
    r = block_sum(s_v, sh);  if (threadIdx.x == 0) partials[3 * Ctx::kMaxBlocks + blockIdx.x] = r;
    r = block_sum(s_w, sh);  if (threadIdx.x == 0) partials[4 * Ctx::kMaxBlocks + blockIdx.x] = r;
    if (last_block_done(counter)) {
        const int G = gridDim.x;
        double t0 = sum_partials(partials, G, sh);
        double t1 = sum_partials(partials + Ctx::kMaxBlocks, G, sh);
        double t2 = sum_partials(partials + 2 * Ctx::kMaxBlocks, G, sh);
        double t3 = sum_partials(partials + 3 * Ctx::kMaxBlocks, G, sh);
        double t4 = sum_partials(partials + 4 * Ctx::kMaxBlocks, G, sh);
        if (threadIdx.x == 0) { out8[0] = t0; out8[1] = t1; out8[2] = t2; out8[3] = t3; out8[4] = t4; }  // sums; sqrt by the caller
    }
}
void apply_pressure_correction(Ctx& c, const DMesh& d, const double* du, const double* dv, const double* dw, const double* p_prime,
                               double* u, double* v, double* wv, double* p, double p_relax, double u_relax, double* out8_dev) {
    if (d.N == 0) return;
    k_apply_correction<<<grid_for(d.N, 256, c.sm_count * 8), 256, 0, c.stream>>>(view(d), du, dv, dw, p_prime, u, v, wv, p, p_relax, u_relax,
                                                                                  c.d_partials, c.d_counter, out8_dev, c.d_flags);
    c.after_launch("k_apply_correction");
}

__global__ void k_extract_diag(int n, const int* __restrict__ rowptr, const int* __restrict__ diag, const double* __restrict__ val, double* d, int* flags) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (rowptr && rowptr[i] == rowptr[i + 1]) { d[i] = 0.; continue; }  // halo row of a partition
        int k = diag[i];
        if (k < 0) { atomicOr(flags, DF_MISSING_ENTRY); d[i] = 0.; } else d[i] = val[k];
    }
}
void extract_diagonal(Ctx& c, const DCsr& a, double* d) {
    if (a.nrows == 0) return;
    ORC_REQUIRE(a.diag != nullptr, ORC_E_INTERNAL, "extract_diagonal: diagonal index not built");
    k_extract_diag<<<grid_for(a.nrows, 256, c.sm_count * 8), 256, 0, c.stream>>>((int)a.nrows, a.rowptr, a.diag, a.val, d, c.d_flags);
    c.after_launch("k_extract_diag");
}

// -------------------------------------------------------------------------------------------------
// S1-S3: passive scalar transport, div(rho u phi) - div(Gamma grad phi) = 0 on the resident flow. Not in the reference: the
// discretisation below is its own specification (DESIGN.md §1), restated operator for operator by tests/scalar_oracle.
// -------------------------------------------------------------------------------------------------
void validate_scalar_settings(const AsmSettings& s) {
    if (s.momentum != ORC_MOM_UD && s.momentum != ORC_MOM_CD1 && s.momentum != ORC_MOM_TVD)
        throw Error(ORC_E_UNSUPPORTED, "unsupported convection scheme");
    if (s.momentum == ORC_MOM_TVD && (s.limiter < ORC_PSI_UD || s.limiter > ORC_PSI_UMIST)) throw Error(ORC_E_INVALID, "unknown TVD limiter");
    if (s.v_interp != ORC_V_LINEAR && s.v_interp != ORC_V_LINEAR_WEIGHTED && s.v_interp != ORC_V_RHIE_CHOW)
        throw Error(ORC_E_UNSUPPORTED, "`None` VelocityInterpolation cannot be used for interior faces");
    if (s.gradient != ORC_G_GREEN_GAUSS_CELL && s.gradient != ORC_G_LEAST_SQUARES) throw Error(ORC_E_UNSUPPORTED, "unsupported gradient scheme");
}

// S1: F_f once per face, from the side of c0 (the outward normal of c0 is the face normal). Cell c1 uses -F_f, which is bit for bit
// what face_flux evaluates from c1's side: every sum in it commutes, vunit(-d) == -vunit(d) and the norms ignore the sign.
__global__ void __launch_bounds__(128) k_scalar_face_flux(MV m, FluxIn in, const double* __restrict__ du, const double* __restrict__ dv,
                                                          const double* __restrict__ dw, double* F, int* flags) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < m.F; f += gridDim.x * blockDim.x) {
        const int c0 = m.c0[f];
        F[f] = face_flux<false>(m, in, f, c0, fnormal(m, f), v3(du[c0], dv[c0], dw[c0]), du, dv, dw, flags);
    }
}

// the value of phi on face f as the gradient sees it from cell i: mean of the two cells, the fixed value, or phi_i
__device__ __forceinline__ double scalar_face_value(const MV& m, const int* zk, const double* zval, const double* phi, int f, int i) {
    const int z = m.fz[f];
    if (m.zt[z] == ORC_BC_INTERIOR) return (phi[m.c0[f]] + phi[m.c1[f]]) * 0.5;
    return (zk[z] == ORC_SBC_FIXED) ? zval[z] : phi[i];
}
// S2 (TVD only): Green-Gauss cell-based grad phi = sum n_out * ((phi_f * A_f) / V_P), plain Vector * Float products
__global__ void __launch_bounds__(128) k_scalar_grad(MV m, const int* __restrict__ zk, const double* __restrict__ zval, const double* __restrict__ phi,
                                                     double* gx, double* gy, double* gz) {
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        V3 acc = vzero();
        const double vol = m.vol[i];
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const double s = scalar_face_value(m, zk, zval, phi, f, i) * m.area[f] / vol;
            acc = vadd(acc, vmuls(outward(m, f, i), s));
        }
        gx[i] = acc.x; gy[i] = acc.y; gz[i] = acc.z;
    }
}

struct ScalarArgs {
    MV m;
    const double *F, *phi, *gx, *gy, *gz;
    const int* zk;
    const double* zval;
    double gamma, rho;
    int scheme, limiter;
    double *val, *b;
};
// min(f, 0) and max(f, 0) as comparisons: both cells of a face see the same zero whatever the sign of a zero flux
__device__ __forceinline__ double neg_part(double f) { return f < 0. ? f : 0.; }
__device__ __forceinline__ double pos_part(double f) { return f > 0. ? f : 0.; }

// S3: one thread per owned cell, faces in ascending order, values straight into the mesh pattern through cf_slot. f is the mass
// flux out of P: (rho * A_f) * (+-F_f). Interior face: a_P += d, a_N -= d (d = Gamma A_f / |x_N - x_P|), then the convective
// coefficients of the face value. TVD decides the upwind cell U on the sign of the c0-side flux, so both cells of a face use the
// same U, D and w = psi(r) / 2 (conservative). Boundary: FIXED a_P += d_b + max(f, 0), b += (d_b - min(f, 0)) phi_b with
// d_b = Gamma A_f / |x_f - x_P|; ZERO_GRADIENT a_P += f.
__global__ void __launch_bounds__(128) k_scalar_transport(ScalarArgs a) {
    const MV& m = a.m;
    for (int i = m.lo + blockIdx.x * blockDim.x + threadIdx.x; i < m.hi; i += gridDim.x * blockDim.x) {
        double a_p = 0., b_p = 0.;
        const V3 cc = ccentroid(m, i);
        // duplicate (i, nb) pairs add up: clear the off-diagonals first
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) if (m.cf_slot[q] >= 0) a.val[m.cf_slot[q]] = 0.;
        for (int q = m.cf_ptr[i]; q < m.cf_ptr[i + 1]; ++q) {
            const int f = m.cf_face[q];
            const int z = m.fz[f];
            const int c0 = m.c0[f];
            const double area = m.area[f];
            const double Ff = a.F[f];
            const double fl = (a.rho * area) * ((c0 == i) ? Ff : -Ff);
            if (m.zt[z] == ORC_BC_INTERIOR) {
                const int nb = (c0 == i) ? m.c1[f] : c0;
                const int slot = m.cf_slot[q];
                const double d = a.gamma * area / vnorm(vsub(ccentroid(m, nb), cc));
                double c_p, c_n;
                if (a.scheme == ORC_MOM_UD) {
                    c_n = neg_part(fl);
                    c_p = fl - c_n;
                } else if (a.scheme == ORC_MOM_CD1) {
                    c_n = fl / 2.;
                    c_p = fl - c_n;
                } else {
                    const int up = (Ff >= 0.) ? c0 : m.c1[f];
                    const int dn = (up == c0) ? m.c1[f] : c0;
                    const double phi_u = a.phi[up], phi_d = a.phi[dn];
                    double w = 0.5;
                    if (phi_d != phi_u) {
                        const V3 g_u = v3(a.gx[up], a.gy[up], a.gz[up]);
                        const double r = 2. * vdot(g_u, vsub(ccentroid(m, dn), ccentroid(m, up))) / (phi_d - phi_u) - 1.;
                        w = psi(a.limiter, r) / 2.;
                    }
                    const double c_up = (1. - w) * fl, c_dn = w * fl;
                    if (up == i) { c_p = c_up; c_n = c_dn; } else { c_p = c_dn; c_n = c_up; }
                }
                a_p = a_p + d;
                a_p = a_p + c_p;
                a.val[slot] = a.val[slot] - d;
                a.val[slot] = a.val[slot] + c_n;
            } else if (a.zk[z] == ORC_SBC_FIXED) {
                const double d_b = a.gamma * area / vnorm(vsub(fcentroid(m, f), cc));
                a_p = a_p + (d_b + pos_part(fl));
                b_p = b_p + (d_b - neg_part(fl)) * a.zval[z];
            } else {
                a_p = a_p + fl;
            }
        }
        a.val[m.diag[i]] = a_p;
        a.b[i] = b_p;
    }
}

void scalar_face_flux(Ctx& c, const DMesh& d, ScalarWork& w, const AsmSettings& s, const double* du, const double* dv, const double* dw,
                      const double* u, const double* v, const double* wv, const double* p) {
    validate_scalar_settings(s);
    const size_t N = (size_t)std::max<int64_t>(d.N, 1), F = (size_t)std::max<int64_t>(d.F, 1);
    if (w.F.n != F) w.F.alloc(&c, F);
    if (w.gpx.n != N) { w.gpx.alloc(&c, N); w.gpy.alloc(&c, N); w.gpz.alloc(&c, N); w.gpx.zero(); w.gpy.zero(); w.gpz.zero(); }
    if (d.F == 0) return;
    const MV m = view(d);
    if (s.v_interp == ORC_V_RHIE_CHOW) {
        if (d.N > 0) launch_grad_p(c, m, s.gradient, p, w.gpx, w.gpy, w.gpz);
        if (w.halo_exchange) { double* g[3] = {w.gpx.p, w.gpy.p, w.gpz.p}; w.halo_exchange(g, 3); }
    }
    FluxIn in;
    in.u = u; in.v = v; in.w = wv; in.p = p; in.gx = w.gpx; in.gy = w.gpy; in.gz = w.gpz; in.v_interp = s.v_interp;
    ProfScope ps(c, PC_ASSEMBLY, 0.);
    k_scalar_face_flux<<<grid_for(d.F, 128, c.sm_count * 16), 128, 0, c.stream>>>(m, in, du, dv, dw, w.F, c.d_flags);
    c.after_launch("k_scalar_face_flux");
}

void build_scalar_transport(Ctx& c, const DMesh& d, ScalarWork& w, const AsmSettings& s, double gamma, double rho, const double* phi,
                            DCsr& a, double* b) {
    validate_scalar_settings(s);
    ORC_REQUIRE(w.F.n == (size_t)std::max<int64_t>(d.F, 1), ORC_E_INTERNAL, "build_scalar_transport: face fluxes not computed");
    const size_t N = (size_t)std::max<int64_t>(d.N, 1);
    if (w.hx.n != N) { w.hx.alloc(&c, N); w.hy.alloc(&c, N); w.hz.alloc(&c, N); w.hx.zero(); w.hy.zero(); w.hz.zero(); }
    if (d.N == 0) return;
    const MV m = view(d);
    const int g = grid_for(d.N, 128, c.sm_count * 16);
    if (s.momentum == ORC_MOM_TVD) {
        {
            ProfScope ps(c, PC_ASSEMBLY, 0.);
            k_scalar_grad<<<g, 128, 0, c.stream>>>(m, d.zone_sbc_kind, d.zone_sbc_value, phi, w.hx, w.hy, w.hz);
            c.after_launch("k_scalar_grad");
        }
        if (w.halo_exchange) { double* h[3] = {w.hx.p, w.hy.p, w.hz.p}; w.halo_exchange(h, 3); }   // the upwind cell may be a halo cell
    }
    ScalarArgs sa;
    sa.m = m; sa.F = w.F; sa.phi = phi; sa.gx = w.hx; sa.gy = w.hy; sa.gz = w.hz; sa.zk = d.zone_sbc_kind; sa.zval = d.zone_sbc_value;
    sa.gamma = gamma; sa.rho = rho; sa.scheme = s.momentum; sa.limiter = s.limiter; sa.val = a.val; sa.b = b;
    ProfScope ps(c, PC_ASSEMBLY, 0.);
    k_scalar_transport<<<g, 128, 0, c.stream>>>(sa);
    c.after_launch("k_scalar_transport");
}

// S4: Boussinesq body force -rho beta (phi - phi_ref) g, fused with the b += b_di of the momentum right-hand sides: one pass of
// 88 B per owned cell (reads b x3, b_di x3, phi, V; writes b x3). Halo rows get (b + b_di) only, as the three k_add_inplace give.
__global__ void k_momentum_source_buoyancy(int64_t n, int64_t lo, int64_t hi, double* bu, double* bv, double* bw, const double* __restrict__ bdu,
                                           const double* __restrict__ bdv, const double* __restrict__ bdw, const double* __restrict__ phi,
                                           const double* __restrict__ vol, double rho_beta, double phi_ref, double gx, double gy, double gz) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double x = bu[i] + bdu[i], y = bv[i] + bdv[i], z = bw[i] + bdw[i];
        if (i >= lo && i < hi) {
            const double s = (rho_beta * (phi[i] - phi_ref)) * vol[i];
            x = x - s * gx; y = y - s * gy; z = z - s * gz;
        }
        bu[i] = x; bv[i] = y; bw[i] = z;
    }
}
void momentum_source_buoyancy(Ctx& c, const DMesh& d, double* b_u, double* b_v, double* b_w, const double* b_u_di, const double* b_v_di,
                              const double* b_w_di, const double* phi, double rho_beta, double phi_ref, const double g[3]) {
    if (d.N <= 0) return;
    ProfScope ps(c, PC_ASSEMBLY, 0.);
    k_momentum_source_buoyancy<<<grid_for(d.N, 256, 1184), 256, 0, c.stream>>>(d.N, d.own_lo, d.own_hi, b_u, b_v, b_w, b_u_di, b_v_di, b_w_di, phi,
                                                                               d.cvol, rho_beta, phi_ref, g[0], g[1], g[2]);
    c.after_launch("k_momentum_source_buoyancy");
}

// S5: the outward flux of phi through every face of zone `zone` (zero elsewhere), from its cell c0 with mass flux
// f = (rho A_f) F_f: FIXED(phi_b) diffusive d_b (phi_P - phi_b), convective max(f, 0) phi_P + min(f, 0) phi_b; ZERO_GRADIENT 0 and
// f phi_P. out2: two planes of F doubles (diffusive, convective).
__global__ void __launch_bounds__(128) k_scalar_zone_flux(MV m, const int* __restrict__ zk, const double* __restrict__ zval, const double* __restrict__ F,
                                                          const double* __restrict__ phi, double gamma, double rho, int zone, double* diff, double* conv) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < m.F; f += gridDim.x * blockDim.x) {
        double dd = 0., cc = 0.;
        if (m.fz[f] == zone) {
            const int p = m.c0[f];
            const double area = m.area[f];
            const double fl = (rho * area) * F[f];
            if (zk[zone] == ORC_SBC_FIXED) {
                const double d_b = gamma * area / vnorm(vsub(fcentroid(m, f), ccentroid(m, p)));
                dd = d_b * (phi[p] - zval[zone]);
                cc = pos_part(fl) * phi[p] + neg_part(fl) * zval[zone];
            } else {
                cc = fl * phi[p];
            }
        }
        diff[f] = dd; conv[f] = cc;
    }
}
void scalar_zone_flux(Ctx& c, const DMesh& d, const ScalarWork& w, double gamma, double rho, const double* phi, int zone, double* out2F) {
    ORC_REQUIRE(w.F.n == (size_t)std::max<int64_t>(d.F, 1), ORC_E_INTERNAL, "scalar_zone_flux: face fluxes not computed");
    if (d.F == 0) return;
    ProfScope ps(c, PC_ASSEMBLY, 0.);
    k_scalar_zone_flux<<<grid_for(d.F, 128, c.sm_count * 16), 128, 0, c.stream>>>(view(d), d.zone_sbc_kind, d.zone_sbc_value, w.F, phi, gamma, rho,
                                                                                 zone, out2F, out2F + d.F);
    c.after_launch("k_scalar_zone_flux");
}

}  // namespace orc
