"""Passive scalar transport on one B200 (DESIGN.md §1, "Passive scalar"): the device assembly bit for bit against the sequential
model (tests/scalar_oracle), the sweeps of SteadySolver.solve_scalar against the model's sweeps (reference-order reductions) and
against tests/fast_model.py (fast mode), and the resident flow left as it was."""
import numpy as np
import pytest

import fast_model as fm
import orc_b200
import scalar_oracle as so
from cases import load_mesh_arrays, settings_pair, smooth_fields
from orc_b200 import discretization as disc
from orc_b200 import linear_algebra as la
from orc_b200 import synthetic as syn
from orc_b200.settings import ReductionMode

pytestmark = pytest.mark.gpu
RHO, MU, GAMMA = 1000.0, 1e-3, 2e-3
UD, CD1, CD2, TVD = 0, 1, 2, 3
PSI_LUD, PSI_QUICK, PSI_UMIST = 2, 3, 4
V_LINEAR, V_LINEAR_WEIGHTED, V_RHIE_CHOW, V_NONE = 0, 1, 2, 3
G_GG, G_LSQ = 0, 2
FIXED = orc_b200.ScalarCondition.Fixed


def scalar_bcs(pm, om, names):
    """INLET fixed at 1, WALL fixed at 0.25 (where the mesh has them), every other zone zero gradient: on both meshes."""
    bcs = so.ScalarBcs(om)
    for name, value in (("INLET", 1.0), ("WALL", 0.25)):
        if name in names:
            pm.set_zone_scalar(name, FIXED, value)
            bcs.set(name, so.FIXED, value)
    return bcs


def mesh_case(oracle, kind):
    if kind == "channel_flow":
        arrays = load_mesh_arrays("channel_flow")
    else:
        arrays = {"hex": lambda: syn.hex_box(8, 6, 4), "tet": lambda: syn.tet_box(4, 3, 3), "hex48": lambda: syn.hex_box(48, 48, 48)}[kind]()
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    names = list(arrays["zone_names"])
    for m in (pm, om):
        if "SYM" in names:
            syn.channel_bcs(m)
        else:   # channel_flow.msh: pressure-driven channel between walls, periodic sides as symmetry planes
            m.set_zone("INLET", 4, -0.02, (0.0, 0.0, 0.0))
            m.set_zone("OUTLET", 5, 0.0, (0.0, 0.0, 0.0))
            m.set_zone("WALL", 3, 0.0, (0.0, 0.0, 0.0))
            m.set_zone("PERIODIC_-Z", 7, 0.0, (0.0, 0.0, 0.0))
            m.set_zone("PERIODIC_+Z", 7, 0.0, (0.0, 0.0, 0.0))
    return pm, om, scalar_bcs(pm, om, names)


def flow_state(oracle, pm, om, ctx, ps, os_):
    """Smooth fields and the momentum matrices of one advection assembly on them (non-trivial Rhie-Chow diagonals), on both sides."""
    u, v, w, p = smooth_fields(om.export())
    a_di, *_ = om.build_momentum_diffusion(MU)
    oa = [om.init_momentum_matrix() for _ in range(3)]
    om.build_momentum_advection(*oa, a_di, u, v, w, p, os_, RHO)
    ga = []
    for a in oa:
        rp, co, va = a.arrays()
        ga.append(la.CsrMatrix.from_arrays(len(rp) - 1, len(rp) - 1, rp, co, va, ctx))
    return (u, v, w, p), oa, ga


def assemble_both(oracle, ctx, kind, seed=3, **kw):
    pm, om, bcs = mesh_case(oracle, kind)
    ps, os_ = settings_pair(oracle, **kw)
    (u, v, w, p), oa, ga = flow_state(oracle, pm, om, ctx, ps, os_)
    phi = np.random.default_rng(seed).uniform(0.0, 1.0, om.n_cells)
    a, b = disc.build_scalar_transport(pm, *ga, u, v, w, p, phi, GAMMA, RHO, ps)
    oa_, ob = so.build(om, bcs, u, v, w, p, phi, *oa, GAMMA, RHO, os_.momentum, os_.limiter, os_.velocity_interpolation, os_.gradient)
    return a.arrays(), oa_.arrays(), b, ob


SCHEMES = [dict(momentum=UD), dict(momentum=CD1), dict(momentum=TVD, limiter=PSI_LUD), dict(momentum=TVD, limiter=PSI_QUICK),
           dict(momentum=TVD, limiter=PSI_UMIST)]


def _id(kw):
    return "-".join(f"{k}{v}" for k, v in kw.items())


@pytest.mark.parametrize("kw", SCHEMES, ids=_id)
@pytest.mark.parametrize("kind", ["hex", "tet", "channel_flow"])
def test_assembly_equals_the_model(oracle, ctx, kind, kw):
    (grp, gco, gva), (orp, oco, ova), b, ob = assemble_both(oracle, ctx, kind, **kw)
    assert np.array_equal(grp, orp) and np.array_equal(gco, oco)
    assert np.array_equal(gva, ova), np.abs(gva - ova).max()
    assert np.array_equal(b, ob), np.abs(b - ob).max()
    assert np.abs(b).max() > 0


@pytest.mark.parametrize("gradient", [G_GG, G_LSQ])
@pytest.mark.parametrize("vel_interp", [V_LINEAR, V_LINEAR_WEIGHTED, V_RHIE_CHOW])
def test_assembly_equals_the_model_for_every_face_flux(oracle, ctx, vel_interp, gradient):
    for kind in ("hex", "tet"):
        (_, _, gva), (_, _, ova), b, ob = assemble_both(oracle, ctx, kind, momentum=TVD, limiter=PSI_QUICK, velocity_interpolation=vel_interp,
                                                         gradient=gradient)
        assert np.array_equal(gva, ova) and np.array_equal(b, ob), kind


def test_assembly_equals_the_model_at_48_cubed(oracle, ctx):
    """110 592 cells: every kernel runs more than one grid-stride pass."""
    (_, _, gva), (_, _, ova), b, ob = assemble_both(oracle, ctx, "hex48", momentum=TVD, limiter=PSI_UMIST)
    assert np.array_equal(gva, ova) and np.array_equal(b, ob)


def steady_pair(oracle, ctx, simple, reference_order, **kw):
    arrays = syn.hex_box(12, 8, 6)
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    om = oracle.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(pm)
    syn.channel_bcs(om)
    bcs = scalar_bcs(pm, om, arrays["zone_names"])
    ps, os_ = settings_pair(oracle, reference_order=reference_order, **kw)
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    st.set_fields(*(np.zeros(pm.n_cells) for _ in range(4)))
    if simple:
        st.iterate(simple)
    return pm, om, bcs, ps, os_, st


@pytest.mark.parametrize("kw,sweeps", [(dict(iterations=10), 1), (dict(momentum=UD, solver_type=3, iterations=10), 1),
                                       (dict(momentum=TVD, limiter=PSI_QUICK, iterations=10), 3), (dict(solver_type=1, iterations=20), 2)],
                         ids=["cd1-multigrid", "ud-bicgstab", "tvd-quick-x3", "cd1-jacobi-x2"])
def test_reference_order_sweeps_equal_the_model(oracle, ctx, kw, sweeps):
    """Three SIMPLE iterations (bit-identical to the oracle's in this mode), then the scalar sweeps on the resident flow."""
    pm, om, bcs, ps, os_, st = steady_pair(oracle, ctx, 3, True, **kw)
    u, v, w, p, a_u, a_v, a_w = so.simple_iterations(om, os_, RHO, MU, 3)
    for a, b in zip(st.get_fields(), (u, v, w, p)):
        assert np.array_equal(a, b)
    phi0 = np.full(pm.n_cells, 0.5)
    want = so.solve(om, bcs, u, v, w, p, phi0, a_u, a_v, a_w, GAMMA, RHO, os_, sweeps)
    got = st.solve_scalar(GAMMA, phi0, sweeps)
    assert np.isfinite(want).all() and np.abs(want - phi0).max() > 0
    assert np.array_equal(got, want), np.abs(got - want).max()


@pytest.mark.parametrize("solver_type", [3, 2], ids=["bicgstab", "multigrid"])
def test_fast_mode_sweep_equals_the_fast_model(oracle, ctx, solver_type):
    """Fast reductions: the sweep's solve is fast_model.iterative_solve on the system the device assembled."""
    pm, om, bcs, ps, os_, st = steady_pair(oracle, ctx, 0, False, solver_type=solver_type, iterations=10)
    assert ps.reduction_mode == ReductionMode.Fast
    u, v, w, p = smooth_fields(pm.export())
    st.set_fields(u, v, w, p)
    n = pm.n_cells
    unit = [disc.initialize_momentum_matrix(pm, ctx) for _ in range(3)]   # the diagonals of a handle that has not iterated yet
    a, b = disc.build_scalar_transport(pm, *unit, u, v, w, p, np.zeros(n), GAMMA, RHO, ps)
    A = fm.Mat.from_handle(a)
    kw = {}
    if solver_type == 2:
        _, glev = la.multigrid_trace(a, b, np.zeros(n), iteration_count=10)
        kw = dict(levels=[(fm.Mat.from_handle(r), fm.Mat.from_handle(q)) for r, q in glev], pos=fm.Positions(pm.export()["cell_centroid"]))
    want = fm.iterative_solve(A, b, np.zeros((1, n)), 10, fm.MULTIGRID if solver_type == 2 else fm.BICGSTAB, **kw)[0]
    got = st.solve_scalar(GAMMA, None, 1)
    assert np.array_equal(got, want), np.abs(got - want).max()


def test_the_resident_flow_is_untouched(oracle, ctx):
    """iterate(2), a TVD scalar solve, iterate(2) gives the fields of iterate(4)."""
    kw = dict(momentum=TVD, limiter=PSI_QUICK, iterations=20)
    _, _, _, _, _, st = steady_pair(oracle, ctx, 2, False, **kw)
    phi = st.solve_scalar(GAMMA, None, 3)
    assert np.isfinite(phi).all() and np.abs(phi).max() > 0
    st.iterate(2)
    _, _, _, _, _, ref = steady_pair(oracle, ctx, 4, False, **kw)
    for a, b in zip(st.get_fields(), ref.get_fields()):
        assert np.array_equal(a, b)


def test_errors(oracle, ctx):
    arrays = syn.hex_box(6, 4, 3)
    pm = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(pm)
    ps, _ = settings_pair(oracle)
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    n = pm.n_cells
    with pytest.raises(orc_b200.OrcError, match="undetermined") as e:
        st.solve_scalar(GAMMA)
    assert e.value.code == orc_b200._lib.E_INVALID
    pm.set_zone_scalar("INLET", FIXED, 1.0)
    for bad in (-1e-3, float("nan")):
        with pytest.raises(orc_b200.OrcError, match="gamma") as e:
            st.solve_scalar(bad)
        assert e.value.code == orc_b200._lib.E_INVALID
    assert np.isfinite(st.solve_scalar(GAMMA)).all()
    unit = [disc.initialize_momentum_matrix(pm, ctx) for _ in range(3)]
    z = np.zeros(n)
    for kw in (dict(momentum=CD2), dict(velocity_interpolation=V_NONE)):
        bad, _ = settings_pair(oracle, **kw)
        with pytest.raises(orc_b200.OrcError) as e:
            disc.build_scalar_transport(pm, *unit, z, z, z, z, z, GAMMA, RHO, bad)
        assert e.value.code == orc_b200._lib.E_UNSUPPORTED
