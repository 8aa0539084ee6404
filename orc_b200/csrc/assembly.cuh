// assembly.cuh — device mesh mirror + the assembly half of the SIMPLE loop
// (src/discretization.rs, src/solver.rs:774-1227 of the reference).
#pragma once
#include <functional>

#include "linalg.cuh"
#include "mesh_host.hpp"

namespace orc {

// Device-resident SoA mirror of HostMesh (HBM layout: DESIGN.md §3).
struct DMesh {
    Ctx* ctx = nullptr;
    int64_t N = 0, F = 0, S = 0, nnz = 0;
    int64_t own_lo = 0, own_hi = 0;  // owned cell range ([0, N) unless this is a partition)
    int nlevels = 0, nzones = 0;
    // faces
    DBuf<int> face_c0, face_c1, face_zone;
    DBuf<double> face_area, fnx, fny, fnz, fcx, fcy, fcz;
    // cells
    DBuf<double> cvol, ccx, ccy, ccz;
    double cc_lo[3] = {0., 0., 0.}, cc_hi[3] = {0., 0., 0.};   // bounding box of the cell centroids (PosHint of the mesh matrices)
    DBuf<int> cf_ptr, cf_face, cf_nb, cf_slot;
    // shared pattern
    DBuf<int> rowptr, col, diag;
    int max_row = 0;   // longest row of the pattern
    // level schedule of the momentum recurrence
    DBuf<int> level_ptr, level_order;
    int max_level_width = 0;
    // zone table (refreshed when the host table changes)
    DBuf<int> zone_type;
    DBuf<double> zone_scalar, zone_vec;
    DBuf<int> zone_sbc_kind;          // passive scalar condition per zone (ORC_SBC_*), uploaded with the zone table
    DBuf<double> zone_sbc_value;
    uint64_t zone_epoch = 0;
};

std::unique_ptr<DMesh> mesh_upload(Ctx& c, const HostMesh& m);
void mesh_refresh_zones(Ctx& c, DMesh& d, const HostMesh& m);  // also validates the BC types reachable on the path

CsrPtr mesh_matrix(Ctx& c, const DMesh& d);  // CSR sharing the mesh pattern, own (uninitialised) values
// face / cell geometry of src/io.rs:289-438 computed on the device from the node coordinates (bit-identical to the host pass)
void mesh_geometry_device(Ctx& c, const HostMesh& m, double* face_area, double* face_normal3, double* face_centroid3, double* cell_volume,
                          double* cell_centroid3, double* device_ms);

struct AsmSettings {
    int momentum, limiter, p_interp, v_interp, gradient, assembly_mode;
};
void validate_settings(const AsmSettings& s);  // the reference's panics on unsupported schemes -> ORC_E_UNSUPPORTED

// scratch that lives as long as a steady solve (or one fine-grained call)
struct AsmWork {
    DBuf<double> gpx, gpy, gpz;      // Green-Gauss grad p per cell
    DBuf<double> gu;                 // 9 N: Green-Gauss grad u (TVD only)
    DBuf<double> pface;              // face pressure per face
    DBuf<double> du_old, dv_old, dw_old;  // frozen-mode snapshot of the diagonals
    DBuf<double> pe;                 // 3 N Peclet terms
    // multi-GPU: fills the halo entries of up to 4 cell vectors from their owners (empty on one GPU)
    std::function<void(double* const*, int)> halo_exchange;
    void ensure(Ctx& c, const DMesh& d, const AsmSettings& s);
};

// build_momentum_diffusion_matrix (discretization.rs:39-131)
void build_momentum_diffusion(Ctx& c, const DMesh& d, double mu, DCsr& a_di, double* b_u, double* b_v, double* b_w);
// the Laplace system of initialize_pressure_field (solver.rs:437-494): a shares the mesh pattern, b is a device vector
void build_pressure_laplace(Ctx& c, const DMesh& d, DCsr& a, double* b);
// initialize_momentum_matrix (discretization.rs:450-472)
void init_momentum_matrix(Ctx& c, const DMesh& d, DCsr& a);
// calculate_pressure_gradient / calculate_velocity_gradient for all cells (solver.rs:774-949); `gradient`: ORC_G_GREEN_GAUSS_CELL or
// ORC_G_LEAST_SQUARES. gu9: nine planes of N doubles, row-major tensor (d u / d x, d u / d y, ... d w / d z).
void pressure_gradient(Ctx& c, const DMesh& d, const double* p, double* gx, double* gy, double* gz, int gradient = ORC_G_GREEN_GAUSS_CELL);
void velocity_gradient(Ctx& c, const DMesh& d, const double* u, const double* v, const double* w, double* gu9, int gradient = ORC_G_GREEN_GAUSS_CELL);
// the potential system of initialize_velocity_field (solver.rs:524-590) and the least-squares gradient of psi (:624-693)
void build_velocity_potential(Ctx& c, const DMesh& d, DCsr& a, double* b);
void potential_gradient(Ctx& c, const DMesh& d, const double* psi, double* u, double* v, double* w);
// build_momentum_advection_matrices (discretization.rs:134-356). du/dv/dw are the diagonals of a_u/a_v/a_w
// (in/out state, SURVEY.md Q2); the matrices' diagonal entries are written as well. peclet3 is a device triple.
void build_momentum_advection(Ctx& c, const DMesh& d, AsmWork& w, const AsmSettings& s, double rho, DCsr& a_u, DCsr& a_v, DCsr& a_w,
                              const DCsr& a_di, double* du, double* dv, double* dw, const double* u, const double* v, const double* wv,
                              const double* p, double* b_u, double* b_v, double* b_w, double* peclet3_dev);
// build_pressure_correction_matrices (discretization.rs:359-448)
void build_pressure_correction(Ctx& c, const DMesh& d, AsmWork& w, const AsmSettings& s, double rho, const double* du, const double* dv,
                               const double* dw, const double* u, const double* v, const double* wv, const double* p, DCsr& a, double* b);
// apply_pressure_correction (solver.rs:1170-1227) fused with the iteration scalars of solver.rs:206-208:
// out8_dev = {sum p'^2, sum |du|^2, sum u, sum v, sum w, -, -, -} over the owned cells (sqrt / division by the caller)
void apply_pressure_correction(Ctx& c, const DMesh& d, const double* du, const double* dv, const double* dw, const double* p_prime,
                               double* u, double* v, double* wv, double* p, double p_relax, double u_relax, double* out8_dev);
void extract_diagonal(Ctx& c, const DCsr& a, double* d);  // d[i] = a(i,i); missing -> DF_MISSING_ENTRY

// ---- passive scalar transport on the converged flow (an extension: the reference has no such equation; DESIGN.md §1) ----
// steady div(rho u phi) - div(Gamma grad phi) = 0 in the mesh pattern, a_P phi_P + sum a_N phi_N = b
struct ScalarWork {
    DBuf<double> F;                  // face flux per face, from the side of c0 (k_scalar_face_flux)
    DBuf<double> gpx, gpy, gpz;      // grad p (Rhie-Chow)
    DBuf<double> hx, hy, hz;         // grad phi (TVD)
    std::function<void(double* const*, int)> halo_exchange;   // multi-GPU: as AsmWork::halo_exchange (empty on one GPU)
};
// momentum UD / CD1 / TVD(limiter), velocity interpolation other than None, gradient Green-Gauss cell or least squares
void validate_scalar_settings(const AsmSettings& s);
// F_f of every face with the resident u, v, w, p, grad p of the settings' scheme and the frozen diagonals du, dv, dw (the halo
// cells of a partition must hold their owners' values; grad p is exchanged here)
void scalar_face_flux(Ctx& c, const DMesh& d, ScalarWork& w, const AsmSettings& s, const double* du, const double* dv, const double* dw,
                      const double* u, const double* v, const double* wv, const double* p);
// one sweep's system with the current phi (its halo cells filled) and w.F; a shares the mesh pattern, b is a device vector
void build_scalar_transport(Ctx& c, const DMesh& d, ScalarWork& w, const AsmSettings& s, double gamma, double rho, const double* phi,
                            DCsr& a, double* b);
// Boussinesq coupling (DESIGN.md §1): b_k <- (b_k + b_di,k) - (s_P * g_k) with s_P = ((rho * beta) * (phi_P - phi_ref)) * V_P on the
// owned rows, b_k + b_di,k on the halo rows, k = u, v, w (one launch)
void momentum_source_buoyancy(Ctx& c, const DMesh& d, double* b_u, double* b_v, double* b_w, const double* b_u_di, const double* b_v_di,
                              const double* b_w_di, const double* phi, double rho_beta, double phi_ref, const double g[3]);
// outward diffusive / convective flux of phi through each face of zone index `zone` with w.F (zero on other faces): out2F = two
// planes of d.F doubles
void scalar_zone_flux(Ctx& c, const DMesh& d, const ScalarWork& w, double gamma, double rho, const double* phi, int zone, double* out2F);

}  // namespace orc
