// TEST INFRASTRUCTURE ONLY. NOT PART OF THE PRODUCT PATH.
//
// Sequential CPU model of the passive scalar transport (DESIGN.md §1, "Passive scalar"): steady div(rho u phi) - div(Gamma grad phi)
// = 0 on a given flow state. The reference has no such equation, so the discretisation written in DESIGN.md is the specification;
// this file restates it operator for operator (C++17, -O2 -ffp-contract=off) over the oracle's own mesh, face flux, pressure gradient
// and iterative_solve (oracle/orc_oracle.hpp, linked from oracle/_build/liborc_oracle.so, so its partition emulation applies to the
// solves here as well). tests/scalar_oracle.py builds and drives it.
//
// Unlike the GPU path, the face flux is evaluated here from BOTH sides of a face (so_face_flux side 1), and the assembly uses the c0
// side; tests/test_scalar_transport.py checks that the c1 side is exactly the negation.
#include <cmath>
#include <cstring>
#include <limits>
#include <map>
#include <string>
#include <vector>

#include "orc_oracle.hpp"

using namespace orc_oracle;

namespace {

std::string g_err;

Vec3 vsub(Vec3 a, Vec3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
Vec3 vadd(Vec3 a, Vec3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
Vec3 vmuls(Vec3 a, Float s) { return {a.x * s, a.y * s, a.z * s}; }
Float vdot(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
Float vnorm(Vec3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }

// psi(r) of src/lib.rs:107-118, as the momentum assembly uses it (Rust f64::min / max == fmin / fmax)
Float psi(int limiter, Float r) {
    switch (limiter) {
        case PSI_UD: return 0.;
        case PSI_CD1: return 1.;
        case PSI_LUD: return r;
        case PSI_QUICK: return (3. + r) / 4.;
        default: {
            Float acc = std::numeric_limits<Float>::infinity();
            acc = std::fmin(acc, 2. * r);
            acc = std::fmin(acc, (1. + 3. * r) / 4.);
            acc = std::fmin(acc, (3. + r) / 4.);
            acc = std::fmin(acc, 2.);
            return std::fmax(0., acc);
        }
    }
}
Float neg_part(Float f) { return f < 0. ? f : 0.; }
Float pos_part(Float f) { return f > 0. ? f : 0.; }

enum { SBC_ZERO_GRADIENT = 0, SBC_FIXED = 1 };

struct Problem {
    const Mesh& m;
    std::map<uint64_t, size_t> zone_index;   // zone id -> position in ascending id order
    const int64_t* kind;                     // per zone (ascending id)
    const double* value;
    Problem(const Mesh& m_, const int64_t* k, const double* v) : m(m_), kind(k), value(v) {
        size_t q = 0;
        for (auto& kv : m.face_zones) zone_index[kv.first] = q++;
    }
    int zone_type(size_t f) const { return m.face_zones.at(m.faces[f].zone).zone_type; }
    size_t zidx(size_t f) const { return zone_index.at(m.faces[f].zone); }
};

// F_f from the side of `cell` (the oracle's get_face_flux: solver.rs:1007-1102)
Float flux(const Problem& pr, const DVec& u, const DVec& v, const DVec& w, const DVec& p, size_t f, size_t cell, int vel_interp, int gradient,
           const Csr& a_u, const Csr& a_v, const Csr& a_w) {
    return get_face_flux(pr.m, u, v, w, p, f, cell, vel_interp, gradient, a_u, a_v, a_w);
}

// Green-Gauss cell based: sum n_out * ((phi_f * A_f) / V_P)
Vec3 scalar_gradient(const Problem& pr, const DVec& phi, size_t i) {
    const Mesh& m = pr.m;
    Vec3 acc{0., 0., 0.};
    const Float vol = m.cells[i].volume;
    for (size_t f : m.cells[i].face_indices) {
        const Face& face = m.faces[f];
        Float pf;
        if (pr.zone_type(f) == Interior) pf = (phi[face.cell_indices[0]] + phi[face.cell_indices[1]]) * 0.5;
        else pf = (pr.kind[pr.zidx(f)] == SBC_FIXED) ? pr.value[pr.zidx(f)] : phi[i];
        const Float s = pf * face.area / vol;
        acc = vadd(acc, vmuls(get_outward_face_normal(face, i), s));
    }
    return acc;
}

// the system of one sweep in the mesh pattern (diagonal + face neighbours, ascending columns); F: c0-side face fluxes
void assemble(const Problem& pr, const DVec& F, const DVec& phi, Float gamma, Float rho, int scheme, int limiter, Csr& a, DVec& b) {
    const Mesh& m = pr.m;
    const size_t n = m.cells.size();
    std::vector<Vec3> g(n);
    if (scheme == TVD)
        for (size_t i = 0; i < n; ++i) g[i] = scalar_gradient(pr, phi, i);
    a = Csr();
    a.nrows = a.ncols = n;
    a.rowptr.assign(1, 0);
    b.assign(n, 0.);
    for (size_t i = 0; i < n; ++i) {
        std::map<size_t, Float> row;
        Float a_p = 0., b_p = 0.;
        const Vec3 cc = m.cells[i].centroid;
        for (size_t f : m.cells[i].face_indices) {
            const Face& face = m.faces[f];
            const size_t c0 = face.cell_indices[0];
            const Float area = face.area;
            const Float fl = (rho * area) * ((c0 == i) ? F[f] : -F[f]);
            if (pr.zone_type(f) == Interior) {
                const size_t c1 = face.cell_indices[1];
                const size_t nb = (c0 == i) ? c1 : c0;
                const Float d = gamma * area / vnorm(vsub(m.cells[nb].centroid, cc));
                Float c_p, c_n;
                if (scheme == UD) {
                    c_n = neg_part(fl);
                    c_p = fl - c_n;
                } else if (scheme == CD1) {
                    c_n = fl / 2.;
                    c_p = fl - c_n;
                } else {
                    const size_t up = (F[f] >= 0.) ? c0 : c1;
                    const size_t dn = (up == c0) ? c1 : c0;
                    Float wgt = 0.5;
                    if (phi[dn] != phi[up]) {
                        const Float r = 2. * vdot(g[up], vsub(m.cells[dn].centroid, m.cells[up].centroid)) / (phi[dn] - phi[up]) - 1.;
                        wgt = psi(limiter, r) / 2.;
                    }
                    const Float c_up = (1. - wgt) * fl, c_dn = wgt * fl;
                    if (up == i) { c_p = c_up; c_n = c_dn; } else { c_p = c_dn; c_n = c_up; }
                }
                a_p = a_p + d;
                a_p = a_p + c_p;
                Float& e = row[nb];   // starts at 0
                e = e - d;
                e = e + c_n;
            } else if (pr.kind[pr.zidx(f)] == SBC_FIXED) {
                const Float d_b = gamma * area / vnorm(vsub(face.centroid, cc));
                a_p = a_p + (d_b + pos_part(fl));
                b_p = b_p + (d_b - neg_part(fl)) * pr.value[pr.zidx(f)];
            } else {
                a_p = a_p + fl;
            }
        }
        row[i] = a_p;
        for (auto& kv : row) { a.col.push_back(kv.first); a.val.push_back(kv.second); }
        a.rowptr.push_back(a.col.size());
        b[i] = b_p;
    }
}

struct Flow {
    DVec u, v, w, p;
};

DVec face_fluxes(const Problem& pr, const Flow& fl, int side, int vel_interp, int gradient, const Csr& a_u, const Csr& a_v, const Csr& a_w) {
    const Mesh& m = pr.m;
    DVec F(m.faces.size());
    for (size_t f = 0; f < m.faces.size(); ++f) {
        const Face& face = m.faces[f];
        const size_t cell = (side == 1 && face.cell_indices.size() > 1) ? face.cell_indices[1] : face.cell_indices[0];
        F[f] = flux(pr, fl.u, fl.v, fl.w, fl.p, f, cell, vel_interp, gradient, a_u, a_v, a_w);
    }
    return F;
}

}  // namespace

#define SO_TRY(...)                 \
    try { __VA_ARGS__; return 0; }  \
    catch (const std::exception& e) { g_err = e.what(); return 1; }

extern "C" {

const char* so_last_error() { return g_err.c_str(); }

// face fluxes F_f of every face from the side of c0 (side 0) or of c1 (side 1; boundary faces: c0)
int so_face_flux(void* mp, const double* u, const double* v, const double* w, const double* p, void* a_u, void* a_v, void* a_w,
                 int64_t vel_interp, int64_t gradient, int64_t side, double* F_out) {
    SO_TRY({
        const Mesh& m = *static_cast<Mesh*>(mp);
        const size_t n = m.cells.size();
        Problem pr(m, nullptr, nullptr);
        Flow fl{DVec(u, u + n), DVec(v, v + n), DVec(w, w + n), DVec(p, p + n)};
        DVec F = face_fluxes(pr, fl, int(side), int(vel_interp), int(gradient), *static_cast<Csr*>(a_u), *static_cast<Csr*>(a_v),
                             *static_cast<Csr*>(a_w));
        std::memcpy(F_out, F.data(), 8 * F.size());
    });
}

// the system of one sweep with the given phi. iv: scheme (UD/CD1/TVD), limiter, velocity interpolation, gradient
int so_build(void* mp, const double* u, const double* v, const double* w, const double* p, const double* phi, void* a_u, void* a_v,
             void* a_w, double gamma, double rho, const int64_t* iv, const int64_t* zone_kind, const double* zone_value, void** a_out,
             double* b_out) {
    SO_TRY({
        const Mesh& m = *static_cast<Mesh*>(mp);
        const size_t n = m.cells.size();
        Problem pr(m, zone_kind, zone_value);
        Flow fl{DVec(u, u + n), DVec(v, v + n), DVec(w, w + n), DVec(p, p + n)};
        DVec F = face_fluxes(pr, fl, 0, int(iv[2]), int(iv[3]), *static_cast<Csr*>(a_u), *static_cast<Csr*>(a_v), *static_cast<Csr*>(a_w));
        Csr a; DVec b;
        assemble(pr, F, DVec(phi, phi + n), gamma, rho, int(iv[0]), int(iv[1]), a, b);
        *a_out = new Csr(a);
        std::memcpy(b_out, b.data(), 8 * n);
    });
}

// `sweeps` assemble + iterative_solve sweeps. iv: scheme, limiter, velocity interpolation, gradient, solver type, iterations,
// preconditioner, mg_smoother, mg_levels; dv: relaxation, threshold. phi in/out.
int so_solve(void* mp, const double* u, const double* v, const double* w, const double* p, void* a_u, void* a_v, void* a_w, double gamma,
             double rho, const int64_t* iv, const double* dv, const int64_t* zone_kind, const double* zone_value, int64_t sweeps, double* phi) {
    SO_TRY({
        const Mesh& m = *static_cast<Mesh*>(mp);
        const size_t n = m.cells.size();
        Problem pr(m, zone_kind, zone_value);
        Flow fl{DVec(u, u + n), DVec(v, v + n), DVec(w, w + n), DVec(p, p + n)};
        DVec F = face_fluxes(pr, fl, 0, int(iv[2]), int(iv[3]), *static_cast<Csr*>(a_u), *static_cast<Csr*>(a_v), *static_cast<Csr*>(a_w));
        DVec x(phi, phi + n);
        SolveOpts o;
        o.gs_intended = true; o.mg_smoother = int(iv[7]); o.mg_levels = uint64_t(iv[8]);
        for (int64_t k = 0; k < sweeps; ++k) {
            Csr a; DVec b;
            assemble(pr, F, x, gamma, rho, int(iv[0]), int(iv[1]), a, b);
            iterative_solve(a, b, x, uint64_t(iv[5]), int(iv[4]), dv[0], dv[1], int(iv[6]), o);
        }
        std::memcpy(phi, x.data(), 8 * n);
    });
}

}  // extern "C"
