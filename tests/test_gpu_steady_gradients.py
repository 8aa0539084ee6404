"""Gradients of a steady handle's resident fields (orc_steady_gradients / SteadySolver.gradients, write_gradients) and the flow
initialisation on a partition mesh, on one GPU: against orc_gradients of the fetched fields and the whole-mesh initialisation."""
import numpy as np
import pytest

import orc_b200
from orc_b200 import synthetic as syn
from orc_b200 import discretization as disc
from orc_b200.settings import GradientReconstructionMethods as G, ReductionMode

pytestmark = pytest.mark.gpu
RHO, MU = 1000.0, 1e-3


def _mesh(kind):
    m = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(12, 8, 8) if kind == "hex" else syn.tet_box(4, 3, 3)))
    syn.channel_bcs(m)
    return m


@pytest.mark.parametrize("kind", ["hex", "tet"])
@pytest.mark.parametrize("scheme", [G.GreenGaussCellBased, G.LeastSquares])
def test_steady_gradients_equal_orc_gradients_of_the_fields(ctx, kind, scheme):
    m = _mesh(kind)
    st = orc_b200.SteadySolver(m, orc_b200.NumericalSettings(), RHO, MU, ctx)
    st.iterate(3)
    gp, gu = st.gradients(scheme)
    rp, ru = disc.calculate_gradients(m, *st.get_fields(), scheme, ctx)
    st.close()
    assert gp.shape == rp.shape and gu.shape == ru.shape
    assert np.array_equal(gp, rp) and np.array_equal(gu, ru)
    assert np.abs(gp).max() > 0 and np.abs(gu).max() > 0


def test_steady_gradients_refuse_what_orc_gradients_refuses(ctx):
    st = orc_b200.SteadySolver(_mesh("hex"), orc_b200.NumericalSettings(), RHO, MU, ctx)
    for scheme in (G.GreenGaussNodeBased, 7):
        with pytest.raises(orc_b200.OrcError) as e:
            st.gradients(scheme)
        assert e.value.code == orc_b200._lib.E_UNSUPPORTED
    st.close()


@pytest.mark.parametrize("scheme", [G.GreenGaussCellBased, G.LeastSquares])
def test_steady_write_gradients_equals_io_write_gradients(tmp_path, ctx, scheme):
    m = _mesh("hex")
    st = orc_b200.SteadySolver(m, orc_b200.NumericalSettings(), RHO, MU, ctx)
    st.iterate(3)
    st.write_gradients(str(tmp_path / "steady.csv"), 7, scheme)
    orc_b200.write_gradients(m, *st.get_fields(), str(tmp_path / "io.csv"), 7, scheme, ctx)
    st.close()
    assert (tmp_path / "steady.csv").read_bytes() == (tmp_path / "io.csv").read_bytes()


def _one_rank(m):
    """The whole mesh as the single partition of a one-rank run (no communicator needed)."""
    part = m.partition(0, 1)
    info = part.partition_info()
    assert info["n_lo"] == info["n_hi"] == 0 and info["n_own"] == m.n_cells
    return part


@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_initialisation_of_a_one_rank_partition_equals_the_whole_mesh(ctx, kind):
    m = _mesh(kind)
    part = _one_rank(m)
    for init, kw in ((orc_b200.initialize_flow, dict(iteration_count=6)), (orc_b200.initialize_flow_new, dict(iteration_count=0))):
        got = init(part, MU, RHO, ctx=ctx, reduction_mode=ReductionMode.Auto, **kw)
        ref = init(m, MU, RHO, ctx=ctx, reduction_mode=ReductionMode.Fast, **kw)
        for a, b in zip(got, ref):
            assert np.array_equal(a, b)
        with pytest.raises(orc_b200.OrcError) as e:
            init(part, MU, RHO, ctx=ctx, reduction_mode=ReductionMode.ReferenceOrder, **kw)
        assert e.value.code == orc_b200._lib.E_UNSUPPORTED


@pytest.mark.parametrize("nz,wraps", [(69, True), (68, False)])
def test_boundary_condition_count_of_a_partition_wraps_like_the_whole_mesh(ctx, nz, wraps):
    """A moving wall counts every face of the mesh in a u16: 22 x 42 x 69 hexes have 3 * 65536 faces, so the count wraps to 0 and
    the system is PressureOnly; 22 x 42 x 68 stays VelocityOnly. A partition must count the whole mesh's faces, not its own."""
    m = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(22, 42, nz)))
    assert (m.counts()["faces"] == 3 * 65536) == wraps
    m.set_zone("WALL", 3, 0.0, (1e-3, 0.0, 0.0))
    m.set_zone("INLET", 3, 0.0, (0.0, 0.0, 0.0))
    m.set_zone("OUTLET", 5, 1e-2, (0.0, 0.0, 0.0))   # PressureOnly: the Laplace field of the outlet pressure; VelocityOnly: rest
    expect = orc_b200.SystemConstraintType.PressureOnly if wraps else orc_b200.SystemConstraintType.VelocityOnly
    assert orc_b200.check_boundary_conditions(m) == expect
    part = _one_rank(m)
    got = orc_b200.initialize_flow_new(part, MU, RHO, 0, ctx=ctx)
    ref = orc_b200.initialize_flow_new(m, MU, RHO, 0, ctx=ctx, reduction_mode=ReductionMode.Fast)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)
    assert (np.abs(got[3]).max() > 0) == wraps


def test_steady_gradients_of_a_one_rank_partition(ctx):
    m = _mesh("hex")
    part = _one_rank(m)
    st = orc_b200.SteadySolver(part, orc_b200.NumericalSettings(), RHO, MU, ctx)
    st.iterate(3)
    gp, gu = st.gradients(G.LeastSquares)
    rp, ru = disc.calculate_gradients(m, *st.get_fields(), G.LeastSquares, ctx)
    st.close()
    assert np.array_equal(gp, rp) and np.array_equal(gu, ru)
