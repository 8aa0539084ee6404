"""Buoyancy-driven flow (DESIGN.md §1, "Buoyancy"): the coupled model of tests/buoyancy_model.py against the exact fully developed
natural convection in a vertical slot, its wall heat flux against conduction, and with beta = 0 against the uncoupled loop. No GPU
needed."""
import math

import numpy as np
import pytest

import buoyancy_model as bm
import fast_simple as fs
import scalar_oracle as so
from orc_b200 import synthetic as syn

RHO, MU = 1000.0, 1e-3
# the slot: 16 x 32 cells, 4 mm long (x, along gravity) and H = 1 mm wide (y); walls at phi0 (y = 0) and phi1 (y = H), open ends at
# p = 0. K = rho beta g_x (phi1 - phi0) H^2 / mu = -0.125 m/s, |u|max = |K| / (72 sqrt 3) = 1.0e-3 m/s.
GAMMA, BETA, G0, PHI0, PHI1 = 1e-3, 0.0125, 10.0, 0.0, 1.0
H, LX, AREA = 1e-3, 4e-3, 4e-3 * 1e-3
ITERATIONS = 150
# measured on the model: the converged profile is 0.741 % of |u|max from the analytic one on the middle columns (a 32-cell
# two-point discretisation of a cubic), the wall fluxes are 4.9e-5 from conduction, each other's negation to 3.2e-8 and the end
# fluxes each other's negation to 7.3e-7 (relative).
PROFILE_BOUND, CONDUCTION_BOUND, WALL_BALANCE_BOUND, END_BALANCE_BOUND = 0.01, 1e-4, 1e-6, 1e-5


def slot_settings(oracle):
    return oracle.Settings(iterations=100, pressure_relaxation=0.1, solver_type=oracle.JACOBI)


def slot_mesh(mesh):
    """INLET / OUTLET pressure zones at 0, WALL and WALL_TOP no-slip walls, SYM symmetry: on the product or the oracle mesh."""
    syn.channel_bcs(mesh, inlet_pressure=0.0)
    mesh.set_zone("WALL_TOP", 3, 0.0, (0.0, 0.0, 0.0))
    return mesh


def slot_arrays():
    return so.split_walls(syn.hex_box(16, 32, 1))


def slot_analytic(cell_centroid, beta=BETA, g_x=-G0):
    """u(y) = (K / 6)(eta^3 - eta / 4), eta = y / H - 1/2, and |u|max"""
    k = RHO * beta * g_x * (PHI1 - PHI0) * H * H / MU
    eta = cell_centroid[:, 1] / H - 0.5
    return k / 6.0 * (eta ** 3 - eta / 4.0), abs(k) / (72.0 * math.sqrt(3.0))


def profile_misfit(cell_centroid, u):
    """max |u - u_exact| over the middle half of the slot's length, as a fraction of the exact |u|max"""
    exact, umax = slot_analytic(cell_centroid)
    mid = (cell_centroid[:, 0] > 0.25 * LX) & (cell_centroid[:, 0] < 0.75 * LX)
    return float(np.abs(u[mid] - exact[mid]).max() / umax)


def run_slot(oracle, beta=BETA, g_x=-G0, iterations=ITERATIONS):
    om = slot_mesh(oracle.Mesh.from_arrays(*syn.mesh_args(slot_arrays())))
    bcs = so.ScalarBcs(om)
    bcs.set("WALL", so.FIXED, PHI0)
    bcs.set("WALL_TOP", so.FIXED, PHI1)
    s = slot_settings(oracle)
    z = np.zeros(om.n_cells)
    state = fs.State(om, MU)
    out = bm.coupled_iterations(om, bcs, s, RHO, MU, (z, z, z, z), z, iterations, fs.oracle_solve(s), GAMMA, beta, (PHI0 + PHI1) / 2,
                                (g_x, 0.0, 0.0), state=state)
    return om, bcs, s, state, out[-1]


@pytest.fixture(scope="module")
def slot(oracle):
    return run_slot(oracle)


def test_the_slot_converges_to_the_analytic_profile(oracle, slot):
    om, _, _, _, rec = slot
    cc = om.export()["cell_centroid"]
    _, umax = slot_analytic(cc)
    assert profile_misfit(cc, rec["u"]) <= PROFILE_BOUND
    assert np.abs(rec["v"]).max() <= 0.002 * umax and np.abs(rec["w"]).max() <= 1e-6 * umax   # w: the mesh's 1e-7 jitter
    assert np.abs(rec["phi"] - (PHI0 + (PHI1 - PHI0) * cc[:, 1] / H)).max() <= 1e-4
    assert rec["report"][-2] <= 1e-7 * umax   # the velocity correction (1.7e-8 |u|max measured): converged


@pytest.mark.parametrize("beta,g_x", [(0.0, -G0), (BETA, G0)], ids=["no-buoyancy", "gravity-flipped"])
def test_the_profile_bound_is_tight(oracle, beta, g_x):
    om, _, _, _, rec = run_slot(oracle, beta=beta, g_x=g_x)
    assert profile_misfit(om.export()["cell_centroid"], rec["u"]) > 10 * PROFILE_BOUND


def test_wall_heat_flux_is_conduction(oracle, slot):
    om, bcs, s, state, rec = slot
    flux = {name: bm.zone_flux(om, bcs, rec, state, s, GAMMA, RHO, name) for name in ("WALL", "WALL_TOP", "INLET", "OUTLET")}
    conduction = GAMMA * (PHI0 - PHI1) * AREA / H
    wall, top = flux["WALL"][0], flux["WALL_TOP"][0]
    assert abs(top - conduction) <= CONDUCTION_BOUND * abs(conduction)
    assert abs(wall + top) <= WALL_BALANCE_BOUND * abs(conduction)
    assert flux["WALL"][1] == 0.0 and flux["WALL_TOP"][1] == 0.0   # no flow through a wall
    cin, cout = flux["INLET"][1], flux["OUTLET"][1]
    assert abs(cin) > 0.01 * abs(conduction)   # hot fluid leaves at the top of one end, cold enters at the bottom of the other
    assert abs(cin + cout) <= END_BALANCE_BOUND * abs(cin)


def test_zero_beta_is_the_uncoupled_loop(oracle):
    """beta = 0: the source adds exact zeros, so u, v, w, p are those of fast_simple.simple_iterations bit for bit."""
    arrays = syn.hex_box(8, 6, 4)
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(om)
    bcs = so.ScalarBcs(om)
    bcs.set("WALL", so.FIXED, 0.25)
    s = oracle.Settings(iterations=10)
    z = np.zeros(om.n_cells)
    coupled = bm.coupled_iterations(om, bcs, s, RHO, MU, (z, z, z, z), z, 3, fs.oracle_solve(s), 2e-3, 0.0, 0.5, (0.0, -9.81, 0.0))
    plain = fs.simple_iterations(om, s, RHO, MU, (z, z, z, z), 3, fs.oracle_solve(s))
    for a, b in zip(coupled, plain):
        for k in "uvwp":
            assert np.array_equal(a[k], b[k]), k
        assert np.abs(a["phi"]).max() > 0
