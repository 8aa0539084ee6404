"""Buoyancy-driven flow on one B200 (DESIGN.md §1, "Buoyancy"): coupled iterations of SteadySolver bit for bit against the coupled
model of tests/buoyancy_model.py (reference order and fast mode), the natural-convection slot run to convergence on the device, an
uncoupled or beta = 0 handle against the plain loop, the errors, and reset()."""
import numpy as np
import pytest

import bench
import buoyancy_model as bm
import fast_model as fm
import fast_simple as fs
import orc_b200
import scalar_oracle as so
import test_buoyancy as tb
from cases import couette_bcs, load_mesh_arrays, make_pair, settings_pair
from orc_b200 import synthetic as syn

pytestmark = pytest.mark.gpu
RHO, MU, GAMMA, BETA, PHI_REF = 1000.0, 1e-3, 2e-3, 0.0125, 0.5
FIXED = orc_b200.ScalarCondition.Fixed
CD2, TVD, PSI_UMIST, V_NONE = 2, 3, 4, 3


def case(oracle, kind):
    """(product mesh, oracle mesh, ScalarBcs, gravity) with the same flow and scalar conditions on both sides."""
    if kind == "slot":
        pm, om = make_pair(oracle, tb.slot_arrays())
        for m in (pm, om):
            tb.slot_mesh(m)
        fixed, g = (("WALL", tb.PHI0), ("WALL_TOP", tb.PHI1)), (-tb.G0, 0.0, 0.0)
    elif kind == "channel_flow":
        pm, om = make_pair(oracle, load_mesh_arrays("channel_flow"))
        for m in (pm, om):
            couette_bcs(m, u_wall=0.0, dp_dx=5.0, wall_zones=("WALL",), moving=None)
        fixed, g = (("INLET", 1.0), ("WALL", 0.25)), (0.0, -10.0, 0.0)
    else:   # "hex": hex_box(8, 6, 4) channel, gravity across the walls
        pm, om = make_pair(oracle, syn.hex_box(8, 6, 4))
        for m in (pm, om):
            syn.channel_bcs(m)
        fixed, g = (("INLET", 1.0), ("WALL", 0.0)), (0.0, -10.0, 0.0)
    bcs = so.ScalarBcs(om)
    for name, value in fixed:
        pm.set_zone_scalar(name, FIXED, value)
        bcs.set(name, so.FIXED, value)
    return pm, om, bcs, g


def run_pinned(oracle, ctx, pm, om, bcs, g, ps, os_, solve, iterations, sweeps, pos=None):
    """`iterations` coupled SteadySolver.iterate(1) calls from rest, each compared with the model's iteration: u, v, w, p, phi equal."""
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    n = pm.n_cells
    st.set_fields(*(np.zeros(n) for _ in range(4)))
    st.couple_scalar(GAMMA, BETA, PHI_REF, g, sweeps)
    batched = []

    def compare(rec):
        st.iterate(1)
        batched.append((st.batched, rec["batched"]))
        for got, name in zip((*st.get_fields(), st.get_scalar()), ("u", "v", "w", "p", "phi")):
            want = rec[name]
            assert np.isfinite(want).all()
            assert np.array_equal(got, want), (rec["iteration"], name, np.abs(got - want).max())

    z = np.zeros(n)
    model = bm.coupled_iterations(om, bcs, os_, RHO, MU, (z, z, z, z), z, iterations, solve, GAMMA, BETA, PHI_REF, g, sweeps, pos=pos,
                                  on_iteration=compare)
    assert np.abs(model[-1]["phi"]).max() > 0 and np.abs(model[-1]["u"]).max() > 0
    return st, batched


# Multigrid from rest diverges on the slot (in the model too): the hex box's TVD case runs it
REFERENCE_CASES = [("slot", dict(solver_type=1, iterations=20), 1),
                   ("hex", dict(solver_type=3, iterations=10), 1), ("hex", dict(iterations=10, momentum=TVD, limiter=PSI_UMIST), 2),
                   ("channel_flow", dict(solver_type=1, iterations=20), 1), ("hex", dict(solver_type=1, iterations=20), 1)]


@pytest.mark.parametrize("kind,kw,sweeps", REFERENCE_CASES,
                         ids=["slot-jacobi", "hex-bicgstab", "hex-tvd-umist-x2", "channel_flow-jacobi", "hex-jacobi"])
def test_reference_order_iterations_equal_the_model(oracle, ctx, kind, kw, sweeps):
    pm, om, bcs, g = case(oracle, kind)
    ps, os_ = settings_pair(oracle, reference_order=True, **kw)
    run_pinned(oracle, ctx, pm, om, bcs, g, ps, os_, fs.oracle_solve(os_), 3, sweeps)


def test_fast_mode_iterations_equal_the_fast_model(oracle, ctx):
    """24^3 jittered hex box, fast reductions forced, lockstep BiCGSTAB for u, v, w."""
    pm, om = make_pair(oracle, syn.hex_box(24, 24, 24))
    for m in (pm, om):
        syn.channel_bcs(m)
    bcs = so.ScalarBcs(om)
    for name, value in (("INLET", 1.0), ("WALL", 0.0)):
        pm.set_zone_scalar(name, FIXED, value)
        bcs.set(name, so.FIXED, value)
    ps, os_ = settings_pair(oracle, pressure_relaxation=bench.P_RELAX, solver_type=3)
    pos = fm.Positions(om.export()["cell_centroid"])
    _, batched = run_pinned(oracle, ctx, pm, om, bcs, (0.0, -10.0, 0.0), ps, os_, fs.model_solve(os_), 4, 1, pos=pos)
    assert batched == [(True, True)] * 4


def test_the_slot_on_the_device(oracle, ctx):
    """The natural-convection slot to convergence through SteadySolver: the bounds of test_buoyancy.py."""
    pm, _, _, g = case(oracle, "slot")
    ps, _ = settings_pair(oracle, reference_order=True, iterations=100, pressure_relaxation=0.1, solver_type=1)
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    st.set_fields(*(np.zeros(pm.n_cells) for _ in range(4)))
    st.couple_scalar(tb.GAMMA, tb.BETA, (tb.PHI0 + tb.PHI1) / 2, g, 1)
    st.iterate(tb.ITERATIONS)
    cc = pm.export()["cell_centroid"]
    u, v, _, _ = st.get_fields()
    misfit = tb.profile_misfit(cc, u)
    print(f"slot on the device: profile misfit {misfit:.5f} of |u|max")
    assert misfit <= tb.PROFILE_BOUND
    flux = {name: st.scalar_zone_flux(name) for name in ("WALL", "WALL_TOP", "INLET", "OUTLET")}
    print(f"slot zone fluxes (diffusive, convective): {flux}")
    conduction = tb.GAMMA * (tb.PHI0 - tb.PHI1) * tb.AREA / tb.H
    assert abs(flux["WALL_TOP"][0] - conduction) <= tb.CONDUCTION_BOUND * abs(conduction)
    assert abs(flux["WALL"][0] + flux["WALL_TOP"][0]) <= tb.WALL_BALANCE_BOUND * abs(conduction)
    cin, cout = flux["INLET"][1], flux["OUTLET"][1]
    assert abs(cin) > 0.01 * abs(conduction) and abs(cin + cout) <= tb.END_BALANCE_BOUND * abs(cin)


def test_zone_flux_equals_the_model(oracle, ctx):
    """Three coupled iterations on the hex box: the device's zone fluxes against the model's sums of the same terms."""
    pm, om, bcs, g = case(oracle, "hex")
    ps, os_ = settings_pair(oracle, reference_order=True, solver_type=1, iterations=20)
    st, _ = run_pinned(oracle, ctx, pm, om, bcs, g, ps, os_, fs.oracle_solve(os_), 3, 1)
    state = fs.State(om, MU)
    z = np.zeros(om.n_cells)
    rec = bm.coupled_iterations(om, bcs, os_, RHO, MU, (z, z, z, z), z, 3, fs.oracle_solve(os_), GAMMA, BETA, PHI_REF, g, state=state)[-1]
    names = ("INLET", "OUTLET", "WALL", "SYM")
    got = {name: st.scalar_zone_flux(name) for name in names}
    want = {name: bm.zone_flux(om, bcs, rec, state, os_, GAMMA, RHO, name) for name in names}
    scale = max(abs(x) for name in names for x in want[name])
    assert scale > 0
    for name in names:   # the same terms in the same order; d_b's distance may differ from numpy's norm in the last bit
        assert np.abs(np.subtract(got[name], want[name])).max() <= 1e-12 * scale, (name, got[name], want[name])


def test_zero_beta_and_uncoupled_handles_are_the_plain_loop(oracle, ctx):
    pm, _, _, g = case(oracle, "hex")
    ps, _ = settings_pair(oracle, reference_order=True, iterations=10)
    n = pm.n_cells

    def handle():
        st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
        st.set_fields(*(np.zeros(n) for _ in range(4)))
        return st

    plain, zero = handle(), handle()
    zero.couple_scalar(GAMMA, 0.0, PHI_REF, g, 2)
    phi = zero.get_scalar()
    assert np.array_equal(phi, np.zeros(n))
    for _ in range(3):
        plain.iterate(1)
        zero.iterate(1)
        for a, b in zip(plain.get_fields(), zero.get_fields()):
            assert np.array_equal(a, b)
        # the iteration's sweeps are solve_scalar on that iteration's flow, from the previous phi
        got = zero.get_scalar()
        assert np.array_equal(got, zero.solve_scalar(GAMMA, phi, 2)) and np.abs(got).max() > 0
        phi = got
    # coupled, then uncoupled: the same launches per iteration as a handle that never was, and the same fields
    was = handle()
    was.couple_scalar(GAMMA, BETA, PHI_REF, g, 1)
    was.uncouple_scalar()
    never = handle()
    counts = []
    for st in (was, never):
        before = ctx.launch_count()
        st.iterate(2)
        counts.append(ctx.launch_count() - before)
    assert counts[0] == counts[1] and counts[0] > 0, counts
    for a, b in zip(was.get_fields(), never.get_fields()):
        assert np.array_equal(a, b)


def test_errors(oracle, ctx):
    pm, _, _, g = case(oracle, "hex")
    ps, _ = settings_pair(oracle, reference_order=True, iterations=10)
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    n = pm.n_cells
    st.set_fields(*(np.zeros(n) for _ in range(4)))
    E_INVALID, E_UNSUPPORTED = orc_b200._lib.E_INVALID, orc_b200._lib.E_UNSUPPORTED

    def refused(code, fn, *args):
        with pytest.raises(orc_b200.OrcError) as e:
            fn(*args)
        assert e.value.code == code, e.value

    refused(E_INVALID, st.couple_scalar, -1e-3, BETA, PHI_REF, g)
    refused(E_INVALID, st.couple_scalar, float("nan"), BETA, PHI_REF, g)
    refused(E_INVALID, st.couple_scalar, GAMMA, float("nan"), PHI_REF, g)
    refused(E_INVALID, st.couple_scalar, GAMMA, BETA, PHI_REF, (0.0, float("nan"), 0.0))
    refused(E_INVALID, st.couple_scalar, GAMMA, BETA, PHI_REF, (0.0, float("inf"), 0.0))
    refused(E_INVALID, st.scalar_zone_flux, "WALL")   # not coupled: no gamma
    with pytest.raises(ValueError):
        st.set_scalar(np.zeros(n + 1))
    # the refused calls left the handle uncoupled: it iterates as a plain one
    ref = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    ref.set_fields(*(np.zeros(n) for _ in range(4)))
    st.iterate(1)
    ref.iterate(1)
    for a, b in zip(st.get_fields(), ref.get_fields()):
        assert np.array_equal(a, b)
    st.couple_scalar(GAMMA, BETA, PHI_REF, g)
    refused(E_INVALID, st.scalar_zone_flux, "NO_SUCH_ZONE")
    refused(E_INVALID, st.couple_scalar, GAMMA, float("nan"), PHI_REF, g)
    assert np.isfinite(st.scalar_zone_flux("WALL")).all()
    st.iterate(1)   # still coupled with the last accepted settings
    assert np.abs(st.get_scalar()).max() > 0
    # no FIXED zone: a mesh of its own
    bare = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(8, 6, 4)))
    syn.channel_bcs(bare)
    refused(E_INVALID, orc_b200.SteadySolver(bare, ps, RHO, MU, ctx).couple_scalar, GAMMA, BETA, PHI_REF, g)
    for kw in (dict(momentum=CD2), dict(velocity_interpolation=V_NONE)):   # the flow may refuse the settings before the coupling does
        bad, _ = settings_pair(oracle, reference_order=True, **kw)
        refused(E_UNSUPPORTED, lambda: orc_b200.SteadySolver(pm, bad, RHO, MU, ctx).couple_scalar(GAMMA, BETA, PHI_REF, g))


def test_reset_zeroes_phi_and_keeps_the_coupling(oracle, ctx):
    pm, _, _, g = case(oracle, "hex")
    ps, _ = settings_pair(oracle, reference_order=True, solver_type=1, iterations=20)
    n = pm.n_cells
    st = orc_b200.SteadySolver(pm, ps, RHO, MU, ctx)
    st.set_fields(*(np.zeros(n) for _ in range(4)))
    st.couple_scalar(GAMMA, BETA, PHI_REF, g, 1)
    st.iterate(2)
    first = (*st.get_fields(), st.get_scalar())
    assert np.abs(first[4]).max() > 0
    st.reset()
    assert np.array_equal(st.get_scalar(), np.zeros(n))
    st.iterate(2)
    for a, b in zip((*st.get_fields(), st.get_scalar()), first):
        assert np.array_equal(a, b)
    st.set_scalar(np.full(n, 0.75))
    assert np.array_equal(st.get_scalar(), np.full(n, 0.75))
