//! UNBUILT / UNTESTED (no Rust toolchain in the build image). FFI declarations for include/orc_b200.h and a
//! `solve_steady` with the reference's exact signature (src/solver.rs:26-37) that routes the hot path to the B200.
#![allow(non_camel_case_types)]
use nalgebra::DVector;
use orc::mesh::Mesh;
use orc::numerical_types::{Float, Uint};
use orc::settings::*;
use std::ffi::{c_char, c_void, CStr, CString};

#[repr(C)] pub struct orc_ctx { _p: [u8; 0] }
#[repr(C)] pub struct orc_mesh { _p: [u8; 0] }
#[repr(C)] pub struct orc_steady { _p: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct orc_settings {
    pub momentum: i32, pub limiter: i32, pub pressure_interpolation: i32, pub velocity_interpolation: i32, pub gradient: i32,
    pub solver_type: i32, pub preconditioner: i32, pub mg_smoother: i32, pub mg_levels: i32, pub gs_mode: i32,
    pub assembly_mode: i32, pub reduction_mode: i32, pub iterations: u64, pub pressure_relaxation: f64,
    pub momentum_relaxation: f64, pub relaxation: f64, pub threshold: f64,
}
#[repr(C)]
pub struct orc_report {
    pub iteration: u64, pub u_avg: f64, pub v_avg: f64, pub w_avg: f64, pub peclet_avg: f64, pub peclet_min: f64,
    pub peclet_max: f64, pub velocity_correction: f64, pub pressure_correction: f64, pub ms_per_iter: f64,
}
pub type orc_report_cb = Option<extern "C" fn(*const orc_report, *mut c_void)>;

extern "C" {
    pub fn orc_settings_default(s: *mut orc_settings);
    pub fn orc_ctx_create(device: i32, stream: *mut c_void, out: *mut *mut orc_ctx) -> i32;
    pub fn orc_ctx_destroy(ctx: *mut orc_ctx);
    pub fn orc_last_error() -> *const c_char;
    pub fn orc_mesh_from_arrays(dims: i32, n_nodes: i64, xyz: *const f64, n_faces: i64, face_node_offsets: *const i64,
        face_nodes: *const i64, c0: *const i64, c1: *const i64, face_zone: *const i64, n_zones: i64, zone_ids: *const i64,
        zone_types: *const i64, zone_names: *const *const c_char, out: *mut *mut orc_mesh) -> i32;
    pub fn orc_mesh_from_geometry(dimensions: i32, n_cells: i64, n_faces: i64, face_c0: *const i64, face_c1: *const i64,
        face_zone: *const i64, face_area: *const f64, face_normal3: *const f64, face_centroid3: *const f64, cell_volume: *const f64,
        cell_centroid3: *const f64, cell_face_offsets: *const i64, cell_face_indices: *const i64, n_zones: i64, zone_ids: *const i64,
        zone_types: *const i64, zone_names: *const *const c_char, out: *mut *mut orc_mesh) -> i32;
    pub fn orc_mesh_set_zone(m: *mut orc_mesh, name: *const c_char, zone_type: i64, scalar: f64, vx: f64, vy: f64, vz: f64) -> i32;
    pub fn orc_mesh_free(m: *mut orc_mesh);
    pub fn orc_solve_steady(ctx: *mut orc_ctx, m: *mut orc_mesh, u: *mut f64, v: *mut f64, w: *mut f64, p: *mut f64,
        s: *const orc_settings, rho: f64, mu: f64, iteration_count: u64, reporting_interval: u64, cb: orc_report_cb,
        user: *mut c_void) -> i32;
    // initialize_flow (src/solver.rs:246-352); reduction_mode: 0 = ORC_REDUCE_FAST, 1 = ORC_REDUCE_REFERENCE_ORDER
    pub fn orc_initialize_flow(ctx: *mut orc_ctx, m: *mut orc_mesh, mu: f64, rho: f64, iteration_count: u64, reduction_mode: i32,
        u: *mut f64, v: *mut f64, w: *mut f64, p: *mut f64) -> i32;
    // calculate_*_gradient (src/solver.rs:774-949) of the steady handle's resident fields: n x 3 and n x 9 row-major, either may be null
    pub fn orc_steady_gradients(st: *mut orc_steady, gradient: i32, grad_p3n: *mut f64, grad_u9n: *mut f64) -> i32;
    // check_boundary_conditions (src/solver.rs:710-770): 0 PressureOnly, 1 VelocityOnly, 2 Hybrid
    pub fn orc_check_boundary_conditions(m: *const orc_mesh, constraint_type: *mut i32) -> i32;
    // passive scalar transport (not in the reference): zone condition (0 zero gradient, 1 fixed), and `sweeps` assemble + solve
    // sweeps on the steady handle's resident flow; phi in/out
    pub fn orc_mesh_set_zone_scalar(m: *mut orc_mesh, name: *const c_char, kind: i32, value: f64) -> i32;
    pub fn orc_steady_solve_scalar(st: *mut orc_steady, gamma: f64, sweeps: u64, phi: *mut f64) -> i32;
    // Boussinesq coupling of the scalar into the loop (sweeps = 0 uncouples), the resident phi of the owned cells, and the
    // (diffusive, convective) outward flux of phi through a zone
    pub fn orc_steady_couple_scalar(st: *mut orc_steady, gamma: f64, beta: f64, phi_ref: f64, gx: f64, gy: f64, gz: f64, sweeps: u64) -> i32;
    pub fn orc_steady_set_scalar(st: *mut orc_steady, phi: *const f64) -> i32;
    pub fn orc_steady_get_scalar(st: *mut orc_steady, phi: *mut f64) -> i32;
    pub fn orc_steady_scalar_zone_flux(st: *mut orc_steady, name: *const c_char, out2: *mut f64) -> i32;
}

fn settings_to_c(ns: &NumericalSettings) -> orc_settings {
    let mut s = orc_settings::default();
    unsafe { orc_settings_default(&mut s) };
    // MomentumDiscretization::TVD carries a bare fn(Float)->Float (src/lib.rs:104): identify the presets by pointer
    (s.momentum, s.limiter) = match ns.momentum {
        MomentumDiscretization::UD => (0, 0),
        MomentumDiscretization::CD1 => (1, 1),
        MomentumDiscretization::CD2 => (2, 1),
        MomentumDiscretization::TVD(psi) if psi as usize == TVD_LUD as usize => (3, 2),
        MomentumDiscretization::TVD(psi) if psi as usize == TVD_QUICK as usize => (3, 3),
        MomentumDiscretization::TVD(psi) if psi as usize == TVD_UMIST as usize => (3, 4),
        MomentumDiscretization::TVD(_) => panic!("orc-b200: custom TVD limiter functions cannot cross the FFI"),
    };
    // GradientReconstructionMethods (src/lib.rs:155-162) -> ORC_G_* (include/orc_b200.h); node-based Green-Gauss is unimplemented in
    // the reference too: the library answers ORC_E_UNSUPPORTED where ORC panics
    s.gradient = match ns.gradient_reconstruction {
        GradientReconstructionMethods::GreenGauss(GreenGaussVariants::CellBased) => 0,
        GradientReconstructionMethods::GreenGauss(GreenGaussVariants::NodeBased) => 1,
        GradientReconstructionMethods::LeastSquares => 2,
        GradientReconstructionMethods::None => 3,
    };
    s.pressure_interpolation = ns.pressure_interpolation as i32;
    s.velocity_interpolation = ns.velocity_interpolation as i32;
    s.pressure_relaxation = ns.pressure_relaxation;
    s.momentum_relaxation = ns.momentum_relaxation;
    s.solver_type = ns.matrix_solver.solver_type as i32;
    s.iterations = ns.matrix_solver.iterations;
    s.relaxation = ns.matrix_solver.relaxation;
    s.threshold = ns.matrix_solver.relative_convergence_threshold;
    s.preconditioner = ns.matrix_solver.preconditioner as i32;
    s
}

/// Flattens the AoS `Mesh` (src/mesh.rs:181-187) into TGRID-style arrays. Geometry is recomputed by the library with
/// the same operation order as io.rs:289-438, so it is bit-identical to what `read_mesh` stored in `mesh`.
/// Flattens ORC's `Mesh` (src/mesh.rs:181-187) WITH the geometry `io::read_mesh` computed (io.rs:289-438), so that the device
/// path assembles from the reference's own areas, normals and volumes (include/orc_b200.h: orc_mesh_from_geometry).
fn upload_mesh(mesh: &Mesh) -> *mut orc_mesh {
    let (mut c0, mut c1, mut fz, mut area, mut normal, mut fcent) = (vec![], vec![], vec![], vec![], vec![], vec![]);
    for f in &mesh.faces {
        c0.push(f.cell_indices[0] as i64);
        c1.push(f.cell_indices.get(1).map_or(-1, |&c| c as i64));
        fz.push(f.zone as i64);
        area.push(f.area);
        normal.extend([f.normal.x, f.normal.y, f.normal.z]);
        fcent.extend([f.centroid.x, f.centroid.y, f.centroid.z]);
    }
    let (mut vol, mut ccent, mut offs, mut cfaces) = (vec![], vec![], vec![0i64], vec![]);
    for cell in &mesh.cells {
        vol.push(cell.volume);
        ccent.extend([cell.centroid.x, cell.centroid.y, cell.centroid.z]);
        cfaces.extend(cell.face_indices.iter().map(|&f| f as i64));
        offs.push(cfaces.len() as i64);
    }
    let mut ids: Vec<i64> = mesh.face_zones.keys().map(|&k| k as i64).collect();
    ids.sort();
    let types: Vec<i64> = ids.iter().map(|i| Uint::from(mesh.face_zones[&(*i as Uint)].zone_type) as i64).collect();
    let names: Vec<CString> = ids.iter().map(|i| CString::new(mesh.face_zones[&(*i as Uint)].name.clone()).unwrap()).collect();
    let name_ptrs: Vec<*const c_char> = names.iter().map(|n| n.as_ptr()).collect();
    let mut out = std::ptr::null_mut();
    let rc = unsafe {
        orc_mesh_from_geometry(3, vol.len() as i64, c0.len() as i64, c0.as_ptr(), c1.as_ptr(), fz.as_ptr(), area.as_ptr(), normal.as_ptr(),
            fcent.as_ptr(), vol.as_ptr(), ccent.as_ptr(), offs.as_ptr(), cfaces.as_ptr(), ids.len() as i64, ids.as_ptr(), types.as_ptr(),
            name_ptrs.as_ptr(), &mut out)
    };
    check(rc);
    for (i, name) in ids.iter().zip(&names) {
        let z = &mesh.face_zones[&(*i as Uint)];
        check(unsafe { orc_mesh_set_zone(out, name.as_ptr(), Uint::from(z.zone_type) as i64, z.scalar_value, z.vector_value.x,
            z.vector_value.y, z.vector_value.z) });
    }
    out
}

fn check(rc: i32) {
    if rc != 0 {
        // the reference's error channel is panic!(): keep it on the Rust side of the boundary
        panic!("{}", unsafe { CStr::from_ptr(orc_last_error()) }.to_string_lossy());
    }
}

/// Drop-in for `orc::solver::solve_steady` (src/solver.rs:26-37): same arguments, same in-place update of u, v, w, p.
#[allow(clippy::too_many_arguments)]
pub fn solve_steady(mesh: &mut Mesh, u: &mut DVector<Float>, v: &mut DVector<Float>, w: &mut DVector<Float>, p: &mut DVector<Float>,
                    numerical_settings: &NumericalSettings, rho: Float, mu: Float, iteration_count: Uint, reporting_interval: Uint) {
    extern "C" fn report(r: *const orc_report, _u: *mut c_void) {
        let r = unsafe { &*r };
        println!("Iteration {}: avg velocity = ({:.2e}, {:.2e}, {:.2e})\tavg peclet = {:.1e}\tmin peclet = {:.1e}\tmax peclet = {:.1e}\tvelocity correction: {:.2e}\tpressure correction: {:.2e}\tms/iter: {:.1e}",
                 r.iteration, r.u_avg, r.v_avg, r.w_avg, r.peclet_avg, r.peclet_min, r.peclet_max, r.velocity_correction, r.pressure_correction, r.ms_per_iter);
    }
    println!("Solving...");
    let mut ctx = std::ptr::null_mut();
    check(unsafe { orc_ctx_create(0, std::ptr::null_mut(), &mut ctx) });
    let m = upload_mesh(mesh);
    let s = settings_to_c(numerical_settings);
    let rc = unsafe { orc_solve_steady(ctx, m, u.as_mut_ptr(), v.as_mut_ptr(), w.as_mut_ptr(), p.as_mut_ptr(), &s, rho, mu,
                                       iteration_count, reporting_interval, Some(report), std::ptr::null_mut()) };
    unsafe { orc_mesh_free(m); orc_ctx_destroy(ctx); }
    check(rc);
    println!("Done solving.");
}
