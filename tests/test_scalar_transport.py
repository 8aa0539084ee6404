"""Passive scalar transport (DESIGN.md §1, "Passive scalar"): properties of the discretisation, checked on its sequential model
(tests/scalar_oracle), and the host-side checks of the product's zone conditions. No GPU needed."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import orc_b200
from orc_b200 import synthetic as syn

import scalar_oracle as so

RHO, MU = 1000.0, 1e-3
UD, CD1, TVD = 0, 1, 3
PSI_QUICK = 3
V_LINEAR, V_LINEAR_WEIGHTED, V_RHIE_CHOW = 0, 1, 2
MESHES = {"hex": lambda: syn.hex_box(6, 4, 3), "tet": lambda: syn.tet_box(3, 3, 2), "poly": lambda: syn.poly_box(6, 4, 3)}


def flowing_state(oracle, arrays, vel_interp, iterations=3):
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(om)
    s = oracle.Settings(velocity_interpolation=vel_interp, iterations=20)
    return om, so.simple_iterations(om, s, RHO, MU, iterations)


@pytest.mark.parametrize("vel_interp", [V_LINEAR, V_LINEAR_WEIGHTED, V_RHIE_CHOW])
@pytest.mark.parametrize("kind", sorted(MESHES))
def test_face_flux_from_c1_is_the_negated_flux_from_c0(oracle, kind, vel_interp):
    """The assembly evaluates F once per face from c0's side and gives c1 -F: that is exactly what c1's side computes."""
    om, (u, v, w, p, a_u, a_v, a_w) = flowing_state(oracle, MESHES[kind](), vel_interp)
    assert np.abs(u).max() > 0 and np.abs(p).max() > 0
    f0 = so.face_flux(om, u, v, w, p, a_u, a_v, a_w, vel_interp, 0, side=0)
    f1 = so.face_flux(om, u, v, w, p, a_u, a_v, a_w, vel_interp, 0, side=1)
    interior = om.export()["face_c1"] >= 0
    assert interior.sum() > 0 and np.abs(f0[interior]).max() > 0
    assert np.array_equal(f1[interior], -f0[interior])


@pytest.mark.parametrize("scheme", [UD, CD1, TVD])
def test_conduction_at_rest_is_the_linear_profile(oracle, scheme):
    """u = p = 0, walls y = 0 / y = H fixed at T0 / T1, everything else zero gradient: T = T0 + (T1 - T0) y / H in every cell."""
    arrays = so.split_walls(syn.hex_box(5, 6, 3, jitter=0.0))
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(om)
    bcs = so.ScalarBcs(om)
    t0, t1, h = 1.0, 3.0, arrays["extent"][1]
    bcs.set("WALL", so.FIXED, t0)
    bcs.set("WALL_TOP", so.FIXED, t1)
    n = om.n_cells
    z = np.zeros(n)
    a, b = so.build(om, bcs, z, z, z, z, z, *so.unit_diagonals(om), 0.7, RHO, scheme, PSI_QUICK, V_LINEAR, 0)
    t = spla.spsolve(a.to_scipy().tocsc(), b)
    y = om.export()["cell_centroid"][:, 1]
    exact = t0 + (t1 - t0) * y / h
    assert np.abs(t - exact).max() <= 1e-12 * np.abs(exact).max()


def test_uniform_stream_upwind_carries_the_inflow_value_exactly(oracle):
    """A uniform stream through a box of dyadic spacing, upwind, no diffusion: phi = phi_in everywhere solves the system exactly."""
    arrays = syn.hex_box(8, 4, 4, lx=1.0, ly=0.5, lz=0.5, jitter=0.0)
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    speed, phi_in = 0.25, 2.5
    om.set_zone("INLET", oracle.VELOCITY_INLET, 0.0, (speed, 0.0, 0.0))
    om.set_zone("OUTLET", oracle.PRESSURE_OUTLET, 0.0)
    om.set_zone("WALL", oracle.SYMMETRY, 0.0)
    om.set_zone("SYM", oracle.SYMMETRY, 0.0)
    bcs = so.ScalarBcs(om)
    bcs.set("INLET", so.FIXED, phi_in)
    n = om.n_cells
    z = np.zeros(n)
    a, b = so.build(om, bcs, np.full(n, speed), z, z, z, z, *so.unit_diagonals(om), 0.0, 1.0, UD, PSI_QUICK, V_LINEAR, 0)
    assert np.abs(b).max() > 0
    assert np.array_equal(a.spmv(np.full(n, phi_in)), b)


def boundary_terms(om, bcs, F, phi, gamma, rho):
    """The scalar flux out through every boundary face, summed independently of the assembly: (term list)."""
    g = om.export()
    zones = om.zones()
    kind_of = {int(i): int(k) for i, k in zip(zones["ids"], bcs.kind)}
    value_of = {int(i): float(v) for i, v in zip(zones["ids"], bcs.value)}
    types = {int(i): int(t) for i, t in zip(zones["ids"], zones["types"])}
    terms = []
    for f in range(F.size):
        zid = int(g["face_zone"][f])
        if types[zid] == 2:
            continue
        c = int(g["face_c0"][f])
        fl = (rho * g["face_area"][f]) * F[f]
        if kind_of[zid] == so.FIXED:
            d_b = gamma * g["face_area"][f] / np.linalg.norm(g["face_centroid"][f] - g["cell_centroid"][c])
            terms += [(d_b + max(fl, 0.0)) * phi[c], -(d_b - min(fl, 0.0)) * value_of[zid]]
        else:
            terms.append(fl * phi[c])
    return terms


@pytest.mark.parametrize("scheme", [UD, CD1, TVD])
def test_the_assembly_is_conservative(oracle, scheme):
    """sum_i (A phi - b)_i is what leaves through the boundary: interior faces cancel up to rounding. A sign flip on one side of one
    interior face breaks the bound."""
    arrays = so.split_walls(syn.hex_box(6, 4, 3))
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(om)
    om.set_zone("WALL_TOP", oracle.WALL, 0.0)
    s = oracle.Settings(iterations=20)
    u, v, w, p, a_u, a_v, a_w = so.simple_iterations(om, s, RHO, MU, 3)
    bcs = so.ScalarBcs(om)
    bcs.set("INLET", so.FIXED, 1.0)
    bcs.set("WALL_TOP", so.FIXED, 0.25)
    gamma = 2e-3
    phi = np.random.default_rng(7).uniform(0.0, 1.0, om.n_cells)
    a, b = so.build(om, bcs, u, v, w, p, phi, a_u, a_v, a_w, gamma, RHO, scheme, PSI_QUICK, V_RHIE_CHOW, 0)
    F = so.face_flux(om, u, v, w, p, a_u, a_v, a_w, V_RHIE_CHOW, 0)
    terms = boundary_terms(om, bcs, F, phi, gamma, RHO)
    rp, co, va = a.arrays()
    products = va * phi[co]
    every = np.concatenate([np.abs(products), np.abs(b), np.abs(terms)])
    gamma_m = every.size * np.finfo(float).eps / (1 - every.size * np.finfo(float).eps)
    bound = gamma_m * every.sum()

    def imbalance(values):
        return abs(np.sum(sp.csr_matrix((values, co, rp), shape=(om.n_cells,) * 2) @ phi - b) - sum(terms))

    assert imbalance(va) <= bound, (imbalance(va), bound)
    # one interior face seen with the wrong sign from one of its cells: the off-diagonal entry of that row flips
    row = int(np.argmax(np.diff(rp)))
    k = next(q for q in range(rp[row], rp[row + 1]) if co[q] != row and abs(va[q]) > 0)
    flipped = va.copy()
    flipped[k] = -flipped[k]
    assert imbalance(flipped) > 100 * bound


def test_zone_condition_errors():
    """Unknown zone names, kinds other than ZeroGradient / Fixed and non-finite values are refused on the host (no device)."""
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(3, 2, 2)))
    pm.set_zone_scalar("INLET", orc_b200.ScalarCondition.Fixed, 1.5)
    pm.set_zone_scalar("WALL", orc_b200.ScalarCondition.ZeroGradient)
    with pytest.raises(orc_b200.OrcError, match="should exist in mesh") as e:
        pm.set_zone_scalar("NO_SUCH_ZONE", orc_b200.ScalarCondition.Fixed, 1.0)
    assert e.value.code == orc_b200._lib.E_INVALID
    for bad in (2, -1):
        with pytest.raises(orc_b200.OrcError, match="kind") as e:
            pm.set_zone_scalar("INLET", bad, 1.0)
        assert e.value.code == orc_b200._lib.E_INVALID
    with pytest.raises(orc_b200.OrcError, match="finite") as e:
        pm.set_zone_scalar("INLET", orc_b200.ScalarCondition.Fixed, float("nan"))
    assert e.value.code == orc_b200._lib.E_INVALID
