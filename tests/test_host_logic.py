"""CPU tests of the product's host side (no GPU): the C ABI library loads and exports every symbol the header declares,
the TGRID reader / geometry / pattern / scatter maps / level schedule of liborc_b200 agree bit for bit with the oracle,
and errors map to the documented status codes."""
import os
import re

import numpy as np
import pytest

import orc_b200
from orc_b200 import _lib
from orc_b200 import synthetic as syn
from cases import load_mesh_arrays, make_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MESHES = ["2D_3x6", "3D_1x3", "3x3_cube", "couette_flow_8x8x1", "channel_flow", "couette_flow_128x64x1"]


def test_library_exports_every_symbol_of_the_header():
    hdr = open(os.path.join(ROOT, "include", "orc_b200.h")).read()
    declared = set(re.findall(r"\b(orc_[a-z0-9_]+)\s*\(", hdr)) - {"orc_report_cb"}
    assert len(declared) > 35
    L = _lib.lib()
    missing = [n for n in sorted(declared) if not hasattr(L, n)]
    assert not missing, missing
    assert set(_lib.EXPORTS) <= declared
    assert b"sm_100a" in L.orc_version()


def test_settings_struct_layout_and_defaults():
    import ctypes as C
    s = _lib.Settings()
    _lib.lib().orc_settings_default(C.byref(s))
    d = orc_b200.NumericalSettings().to_c()
    for name, _ in _lib.Settings._fields_:
        assert getattr(s, name) == getattr(d, name), name
    assert (s.momentum, s.pressure_interpolation, s.velocity_interpolation, s.solver_type, s.iterations) == (1, 3, 2, 2, 50)  # src/lib.rs:58-86
    assert (s.pressure_relaxation, s.momentum_relaxation, s.relaxation, s.threshold) == (0.01, 0.5, 0.5, 1e-3)


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(orc_b200.OrcError) as e:
        orc_b200.Context(0)
    assert e.value.code == _lib.E_CUDA


def assert_same_mesh(pm, om):
    a, b = pm.export(), om.export()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    za, zb = pm.zones(), om.zones()
    assert za["names"] == zb["names"] and np.array_equal(za["ids"], zb["ids"]) and np.array_equal(za["types"], zb["types"])


@pytest.mark.parametrize("name", MESHES)
def test_geometry_of_reference_meshes_is_bit_exact(oracle, name):
    pm, om = make_pair(oracle, load_mesh_arrays(name))
    assert_same_mesh(pm, om)


@pytest.mark.parametrize("gen,args", [(syn.hex_box, (7, 5, 4)), (syn.hex_box, (9, 9, 1)), (syn.tet_box, (4, 3, 3)),
                                      (syn.wedge_box, (5, 4, 3)),     # triangular prisms: tri + quad faces, mixed TGRID sections
                                      (syn.poly_box, (6, 4, 3)),      # polyhedra with six-node polygon faces
                                      (syn.pyramid_box, (4, 3, 2))])  # pyramids: an apex node per hex, tri + quad faces
def test_synthetic_meshes_and_tgrid_reader_roundtrip(oracle, tmp_path, gen, args):
    arrays = gen(*args)
    pm, om = make_pair(oracle, arrays)
    assert_same_mesh(pm, om)
    e = pm.export()
    assert np.isclose(e["cell_volume"].sum(), 0.004 * 0.001 * 0.001, rtol=1e-6)
    out = e["face_centroid"] - e["cell_centroid"][e["face_c0"]]
    assert np.all(np.einsum("ij,ij->i", out, e["face_normal"]) > 0)      # normals point out of c0
    interior = e["face_c1"] >= 0
    assert np.all(e["face_c0"][interior] < e["face_c1"][interior])
    path = str(tmp_path / "m.msh")
    syn.write_tgrid(path, arrays)
    assert_same_mesh(orc_b200.read_mesh(path), om)                        # product reader == arrays path
    assert_same_mesh(orc_b200.read_mesh(path), oracle.Mesh.read(path))    # == the oracle's restatement of io.rs


def example_mesh_tgrid(m):
    """TGRID text of one of the reference's example meshes from its stored connectivity, laid out as tests/golden/make_golden.py
    parsed the original file: the mesh's own dimension ((2 2) and two coordinates per node for the 2D meshes), hex integers, face
    sections in file order, each after a `(0 "... NAME")` comment that names its zone."""
    dims = m["dims"]
    fo, fn, c0, c1, fz = m["face_node_offsets"], m["face_nodes"], m["c0"], m["c1"], m["face_zone"]
    zones = {int(z): (int(t), name) for z, t, name in zip(m["zone_ids"], m["zone_types"], m["zone_names"])}
    nn, nf, nc = m["xyz"].shape[0], c0.size, int(max(c0.max(), c1.max()))
    out = ['(0 "Dimensions")', f"(2 {dims})", '(0 "Node Section")', f"(10 (0 1 {nn:x} 0 {dims}))", f"(10 (1 1 {nn:x} 1 {dims})", "("]
    out += [" ".join(repr(float(x)) for x in row[:dims]) for row in m["xyz"]]
    out += ["))", f"(12 (0 1 {nc:x} 0 0))", f"(13 (0 1 {nf:x} 0 0))"]
    cuts = np.flatnonzero(np.diff(fz)) + 1
    for start, end in zip(np.r_[0, cuts], np.r_[cuts, nf]):
        z = int(fz[start])
        counts = np.diff(fo)[start:end]
        k = int(counts[0]) if np.all(counts == counts[0]) and counts[0] <= 4 else 0      # 0: mixed, the node count is the line length
        out += [f'(0 "Faces of zone {zones[z][1]}")', f"(13 ({z:x} {start + 1:x} {end:x} {zones[z][0]:x} {k:x})("]
        out += [" ".join(f"{int(v) + 1:x}" for v in fn[fo[q]:fo[q + 1]]) + f" {int(c0[q]):x} {int(c1[q]):x}" for q in range(start, end)]
        out += [")", ")"]
    return "\n".join(out) + "\n"


@pytest.mark.parametrize("name", MESHES)
def test_reader_on_the_reference_example_meshes(oracle, tmp_path, name):
    """The product's TGRID reader on the reference's example meshes, written back from their stored connectivity (the original
    files are not part of the repository): it must equal the oracle's restatement of io.rs::read_mesh on the same file, and the
    mesh built from the arrays parsed out of the original file."""
    arrays = load_mesh_arrays(name)
    path = str(tmp_path / f"{name}.msh")
    with open(path, "w") as f:
        f.write(example_mesh_tgrid(arrays))
    pm = orc_b200.read_mesh(path)
    assert pm.n_cells == int(max(arrays["c0"].max(), arrays["c1"].max()))
    assert_same_mesh(pm, oracle.Mesh.read(path))
    assert_same_mesh(pm, oracle.Mesh.from_arrays(*syn.mesh_args(arrays)))


@pytest.mark.parametrize("name", ["channel_flow", "couette_flow_8x8x1", "wedge_box", "poly_box"])
def test_pattern_equals_the_reference_matrix_pattern(oracle, name):
    pm, om = make_pair(oracle, {"wedge_box": lambda: syn.wedge_box(4, 3, 2), "poly_box": lambda: syn.poly_box(4, 3, 2)}[name]()
                       if name.endswith("_box") else load_mesh_arrays(name))
    rp, co = pm.pattern()
    orp, oco, ova = om.init_momentum_matrix().arrays()   # initialize_momentum_matrix carries the pattern (discretization.rs:450-472)
    assert np.array_equal(rp, orp) and np.array_equal(co, oco)
    drp, dco, _ = om.build_momentum_diffusion(1e-3)[0].arrays()
    assert np.array_equal(rp, drp) and np.array_equal(co, dco)


@pytest.mark.parametrize("arrays", [syn.hex_box(6, 5, 4), syn.tet_box(3, 3, 2), syn.wedge_box(4, 3, 3), syn.poly_box(6, 3, 3),
                                    syn.pyramid_box(3, 3, 2)], ids=["hex", "tet", "wedge", "polyhedra", "pyramid"])
def test_level_schedule_respects_the_recurrence(arrays):
    """level(i) = 1 + max level(j) over neighbours j < i: a cell only depends on strictly lower levels, cells with no lower
    neighbour sit on level 0, and a hex box numbered x-fastest has nx + ny + nz - 2 levels (SURVEY.md §7.2 K3)."""
    m = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    rp, co = m.pattern()
    lv = m.levels()
    for i in range(m.n_cells):
        lower = [j for j in co[rp[i]:rp[i + 1]] if j < i]
        assert lv[i] == (1 + max(lv[j] for j in lower) if lower else 0)
    assert m.counts()["levels"] == lv.max() + 1
    if arrays["n_cells"] == int(np.prod(arrays["shape"])) and arrays["face_node_offsets"][1] == 4:     # the plain hex box
        assert m.counts()["levels"] == sum(arrays["shape"]) - 2


def test_zone_assignment_by_name_and_errors(oracle, tmp_path):
    pm, _ = make_pair(oracle, load_mesh_arrays("channel_flow"))
    assert set(pm.zones()["names"]) == {"FLUID", "INLET", "OUTLET", "PERIODIC_-Z", "PERIODIC_+Z", "WALL"}
    z = pm.get_face_zone("INLET")                       # mesh.get_face_zone(name) (src/mesh.rs:189-195, src/tests.rs:60-76)
    z.zone_type = orc_b200.FaceConditionTypes.PressureInlet
    z.scalar_value = -0.01
    z.vector_value = (1.0, 2.0, 3.0)
    assert z.zone_type == 4 and z.scalar_value == -0.01 and z.vector_value == (1.0, 2.0, 3.0)
    with pytest.raises(orc_b200.OrcError) as e:
        pm.get_face_zone("NOPE")
    assert e.value.code == _lib.E_INVALID
    with pytest.raises(orc_b200.OrcError) as e:
        orc_b200.read_mesh(str(tmp_path / "missing.msh"))
    assert e.value.code == _lib.E_IO
    bad = tmp_path / "bad.msh"
    bad.write_text('(0 "x y")\n(2 3)\n(10 (0 1 2 0 3))\n(10 (1 1 2 1 3)\n(\n0 0 0\n1 0 0\n))\n(13 (2 1 1 3 3)(\n1 2 9 1 0\n)\n)\n')
    with pytest.raises(orc_b200.OrcError) as e:
        orc_b200.read_mesh(str(bad))
    assert e.value.code == _lib.E_IO


def test_check_boundary_conditions_is_host_logic_and_matches_the_oracle(oracle):
    """src/solver.rs:710-770 through the C ABI (no GPU involved) against the oracle's restatement."""
    import orc_b200
    from orc_b200 import synthetic as syn
    from cases import make_pair
    pm, om = make_pair(oracle, syn.hex_box(5, 4, 3))
    with pytest.raises(orc_b200.OrcError) as e:
        orc_b200.check_boundary_conditions(pm)
    assert e.value.code == orc_b200._lib.E_INVALID and "You must set boundary conditions" in e.value.message
    with pytest.raises(oracle.OraclePanic):
        om.check_boundary_conditions()
    for m in (pm, om):
        syn.channel_bcs(m)
    assert orc_b200.check_boundary_conditions(pm) == om.check_boundary_conditions() == 0      # PressureOnly
    for m in (pm, om):
        m.set_zone("WALL", 3, 0.0, (1e-3, 0.0, 0.0))
    assert orc_b200.check_boundary_conditions(pm) == om.check_boundary_conditions() == 2      # Hybrid
    for m in (pm, om):
        m.set_zone("OUTLET", 3, 0.0, (0.0, 0.0, 0.0))
    assert orc_b200.check_boundary_conditions(pm) == om.check_boundary_conditions() == 1      # VelocityOnly (one pressure BC left)


def test_solution_data_files_round_trip_and_format(tmp_path):
    """write_data / read_data (src/io.rs:519-620): `{:.e}` is Rust's shortest round-trip exponent format, the centroid is
    `{:.2e}` per component (src/lib.rs:551-556). Known strings of Rust's formatter + an exact round trip of the fields."""
    import orc_b200
    from orc_b200 import io as oio, synthetic as syn
    assert [oio._rust_exp(x) for x in (1.0, 0.5, 1234.5, -0.00042, 0.0, -0.0, 1e-300, 123456789.0, float("inf"))] == \
        ["1e0", "5e-1", "1.2345e3", "-4.2e-4", "0e0", "-0e0", "1e-300", "1.23456789e8", "inf"]
    assert oio._rust_exp(float("nan")) == "NaN"
    assert [oio._rust_exp(x, 2) for x in (0.002, 12345.678, 0.0, -0.000995)] == ["2.00e-3", "1.23e4", "0.00e0", "-9.95e-4"]
    mesh = orc_b200.Mesh.from_arrays(*syn.mesh_args(syn.hex_box(4, 3, 2)))
    rng = np.random.default_rng(0)
    u, v, w, p = (rng.standard_normal(mesh.n_cells) * 10.0 ** rng.integers(-12, 6, mesh.n_cells) for _ in range(4))
    path = tmp_path / "solution.csv"
    oio.write_data(mesh, u, v, w, p, str(path))
    lines = path.read_text().splitlines()
    assert len(lines) == mesh.n_cells and all(l.count("\t") == 2 and l.startswith("(") for l in lines)
    back = oio.read_data(str(path))
    for a, b in zip((u, v, w, p), back):
        assert np.array_equal(a, b)                       # shortest round-trip digits: nothing is lost
    oio.write_data(mesh, u, v, w, p, str(path), decimal_precision=3)
    assert path.read_text().splitlines()[0].split("\t")[2] == oio._rust_exp(p[0], 3)
    with pytest.raises(OSError, match="could not read data file"):
        oio.read_data(str(tmp_path / "missing.csv"))


@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_mesh_from_geometry_round_trip(kind):
    """orc_mesh_from_geometry (SURVEY.md §8b: the caller's flattened Mesh, geometry included): a mesh rebuilt from the exported
    SoA of another one is the same mesh — geometry bit for bit, the shared CSR pattern, the assembly level schedule, zones, and
    its partitions."""
    import orc_b200
    from orc_b200 import synthetic as syn
    arrays = syn.hex_box(5, 4, 6) if kind == "hex" else syn.tet_box(3, 2, 4)
    a = orc_b200.Mesh.from_arrays(*syn.mesh_args(arrays))
    syn.channel_bcs(a)
    ea = a.export()
    b = orc_b200.Mesh.from_geometry(arrays["dims"], ea, arrays["zone_ids"], arrays["zone_types"], arrays["zone_names"])
    syn.channel_bcs(b)
    eb = b.export()
    for k in ea:
        assert np.array_equal(ea[k], eb[k]), k
    ca, cb = a.counts(), b.counts()
    assert cb["nodes"] == 0 and {k: v for k, v in ca.items() if k != "nodes"} == {k: v for k, v in cb.items() if k != "nodes"}
    assert all(np.array_equal(x, y) for x, y in zip(a.pattern(), b.pattern()))
    assert np.array_equal(a.levels(), b.levels())
    pa, pb = a.partition(1, 2), b.partition(1, 2)
    assert pa.partition_info() == pb.partition_info()
    assert np.array_equal(pa.export()["cell_volume"], pb.export()["cell_volume"])
    # malformed input is refused, not trusted
    bad = dict(ea)
    bad["cell_face_indices"] = ea["cell_face_indices"][::-1].copy()
    with pytest.raises(orc_b200.OrcError):
        orc_b200.Mesh.from_geometry(arrays["dims"], bad, arrays["zone_ids"], arrays["zone_types"], arrays["zone_names"])


def test_reader_fast_path_and_fallback_agree_with_the_oracle(oracle, tmp_path):
    """Uniform face sections (face type 2 / 3 / 4 in the (13 header) are parsed by the host threads; anything irregular falls back to
    the line-by-line parser that follows io.rs:194-274. Variants of one file: as written (fast path), CRLF line endings, the "("
    of a section on its own line, a section declared as mixed (type 0: sequential parser), and a section with a blank line in its
    body (the reference stops reading that section there: both readers must agree, whatever the outcome)."""
    arrays = syn.hex_box(6, 5, 4)
    base = str(tmp_path / "base.msh")
    syn.write_tgrid(base, arrays)
    text = open(base).read()
    ref = oracle.Mesh.read(base)
    assert_same_mesh(orc_b200.read_mesh(base), ref)
    lines = text.split("\n")
    heads = [i for i, l in enumerate(lines) if l.startswith("(13 (") and not l.startswith("(13 (0 ")]
    assert len(heads) >= 3
    variants = {}
    variants["crlf"] = text.replace("\n", "\r\n")
    own = list(lines)
    own[heads[0]] = own[heads[0]][:-1]                      # "(13 (... 2 4)(" -> "(13 (... 2 4)" + a "(" line of its own
    own.insert(heads[0] + 1, "(")
    variants["paren_line"] = "\n".join(own)
    mixed = list(lines)
    mixed[heads[1]] = mixed[heads[1]].replace(" 4)(", " 0)(")
    variants["mixed_header"] = "\n".join(mixed)
    for name, body in variants.items():
        path = str(tmp_path / f"{name}.msh")
        with open(path, "w", newline="") as f:
            f.write(body)
        assert_same_mesh(orc_b200.read_mesh(path), oracle.Mesh.read(path))
        assert_same_mesh(orc_b200.read_mesh(path), ref)
    blank = list(lines)
    blank.insert(heads[2] + 3, "")
    path = str(tmp_path / "blank.msh")
    open(path, "w").write("\n".join(blank))
    outcomes = []
    for reader, err in ((orc_b200.read_mesh, orc_b200.OrcError), (oracle.Mesh.read, oracle.OraclePanic)):
        try:
            outcomes.append(("ok", reader(path).export()["face_area"].size if reader is orc_b200.read_mesh else reader(path).n_cells))
        except err as e:
            outcomes.append(("error", None))
    assert outcomes[0][0] == outcomes[1][0], outcomes


def _c_prototypes(text):
    """{name: (return type, [parameter types])} of the `orc_*` prototypes of a C header, types normalised to Rust FFI spelling."""
    import re
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    scalars = {"int32_t": "i32", "int64_t": "i64", "uint64_t": "u64", "double": "f64", "void": "c_void", "char": "c_char"}

    def ty(c):
        c = c.strip()
        c = re.sub(r"\b[A-Za-z_]\w*$", "", c).strip() if not c.endswith("*") and " " in c else c   # drop the parameter name
        stars = c.count("*")
        base = c.replace("*", " ").split()
        const = base[0] == "const"
        inner_const = len(base) > 2 and base[-1] == "const"            # `const char* const*`
        name = [b for b in base if b != "const"][0]
        r = scalars.get(name, name)
        for k in range(stars):
            r = ("*const " if (const if k == 0 else inner_const) else "*mut ") + r
        return r

    out = {}
    for m in re.finditer(r"^\s*((?:const\s+)?\w+\s*\*?)\s*(orc_\w+)\s*\(([^;{]*?)\)\s*;", text, flags=re.M | re.S):
        ret, name, params = m.group(1).strip(), m.group(2), " ".join(m.group(3).split())
        plist = [] if params in ("", "void") else [ty(q) for q in params.split(",")]
        out[name] = ("" if ret == "void" else ty(ret + " x" if not ret.endswith("*") else ret), plist)
    return out


def _rust_prototypes(text):
    import re
    text = re.sub(r"//[^\n]*", " ", text)
    out = {}
    for m in re.finditer(r"pub fn (orc_\w+)\s*\(([^)]*)\)\s*(?:->\s*([^;]+))?;", text, flags=re.S):
        params = [" ".join(q.split(":", 1)[1].split()) for q in m.group(2).split(",") if ":" in q]
        out[m.group(1)] = ((m.group(3) or "").strip(), params)
    return out


def test_rust_shim_declarations_match_the_header():
    """rust/orc-b200-sys cannot be compiled here (no cargo / rustc), so its `extern "C"` block is checked textually against
    include/orc_b200.h: every declared function exists in the header and in the built library, with the same parameter and return
    types in the same order, and the two #[repr(C)] structs list the header's fields in the header's order."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "orc_b200.h")).read()
    rust = open(os.path.join(root, "rust", "orc-b200-sys", "src", "lib.rs")).read()
    cp, rp = _c_prototypes(header), _rust_prototypes(rust)
    assert len(rp) >= 10 and "orc_solve_steady" in rp
    L = _lib.lib()
    for name, (ret, params) in rp.items():
        assert name in cp, f"{name} is declared in the Rust shim but not in include/orc_b200.h"
        assert hasattr(L, name), f"{name} is not exported by liborc_b200.so"
        assert (ret, params) == cp[name], (name, (ret, params), cp[name])

    def c_fields(struct):
        body = re.search(r"typedef struct " + struct + r"\s*\{(.*?)\}\s*" + struct + r"\s*;", header, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", " ", body, flags=re.S)
        conv = {"int32_t": "i32", "uint64_t": "u64", "double": "f64", "int64_t": "i64"}
        return [(n.strip(), conv[f.split()[0]]) for f in body.split(";") if f.strip() for n in f.split(None, 1)[1].split(",")]

    def rust_fields(struct):
        body = re.search(r"pub struct " + struct + r"\s*\{(.*?)\}", rust, flags=re.S).group(1)
        return [(n, t) for n, t in re.findall(r"pub (\w+):\s*(\w+)", body)]

    for struct in ("orc_settings", "orc_report"):
        assert rust_fields(struct) == c_fields(struct), struct


@pytest.mark.parametrize("kind,seed", [("hex", 1), ("tet", 2), ("wedge", 3), ("polyhedra", 4), ("hex", 5), ("pyramid", 6)])
def test_faces_listed_from_the_other_side(oracle, kind, seed):
    """TGRID does not promise c0 < c1 nor that a boundary face names its cell first: the reference drops a missing c0 and NEGATES the
    normal (src/io.rs:333-339), and `get_outward_face_normal` (src/mesh.rs:216-222) sorts out the rest. Boxes of every cell type with
    the OUTLET faces given as (0, cell) and a random third of the interior faces as (higher, lower), node loops reversed accordingly:
    the product's host pass equals the oracle's bit for bit, describes the same geometry as the untouched box, and the pattern /
    schedule are unchanged."""
    a = {"hex": lambda: syn.hex_box(5, 4, 3), "tet": lambda: syn.tet_box(3, 3, 2), "wedge": lambda: syn.wedge_box(4, 3, 2),
         "polyhedra": lambda: syn.poly_box(6, 3, 2), "pyramid": lambda: syn.pyramid_box(3, 2, 2)}[kind]()
    fo, fn = a["face_node_offsets"], a["face_nodes"].copy()
    c0, c1 = a["c0"].copy(), a["c1"].copy()
    rng = np.random.default_rng(seed)
    flipped = 0
    for q in range(c0.size):
        if a["face_zone"][q] == 4 or (c1[q] != 0 and rng.random() < 0.33):
            c0[q], c1[q] = c1[q], c0[q]
            loop = fn[fo[q]:fo[q + 1]].copy()
            fn[fo[q]:fo[q + 1]] = np.r_[loop[0], loop[:0:-1]]
            flipped += 1
    assert flipped > 10
    b = dict(a)
    b.update(c0=c0, c1=c1, face_nodes=fn)
    pm, om = make_pair(oracle, b)
    assert_same_mesh(pm, om)
    ref = orc_b200.Mesh.from_arrays(*syn.mesh_args(a))
    e, r = pm.export(), ref.export()
    assert np.allclose(e["cell_volume"], r["cell_volume"], rtol=1e-12) and np.allclose(e["face_area"], r["face_area"], rtol=1e-12)   # reversed loops: other summation order
    out = e["face_centroid"] - e["cell_centroid"][e["face_c0"]]
    assert np.all(np.einsum("ij,ij->i", out, e["face_normal"]) > 0)      # after the reference's fix-up every normal points out of the first cell
    assert all(np.array_equal(x, y) for x, y in zip(pm.pattern(), ref.pattern())) and np.array_equal(pm.levels(), ref.levels())


def test_rust_exponent_format_properties():
    """`{:e}` of the data files (src/io.rs:585-589) on arbitrary doubles: the text reads back to the same bits (the restart of
    src/tests.rs:84-86 is lossless), has Rust's shape — one leading digit, no trailing zeros, a bare exponent — and `{:.Ne}` equals
    the correctly rounded decimal expansion of the exact binary value."""
    import re
    import struct
    from decimal import ROUND_HALF_EVEN, Decimal
    from hypothesis import given, settings, strategies as st
    from orc_b200 import io as oio
    shape = re.compile(r"^-?\d(\.\d*[1-9])?e-?(0|[1-9]\d*)$")

    @settings(max_examples=400, deadline=None, derandomize=True)
    @given(st.floats(allow_nan=False, allow_infinity=False))
    def shortest(x):
        s = oio._rust_exp(x)
        assert shape.match(s), s
        assert struct.pack("<d", float(s)) == struct.pack("<d", x)

    @settings(max_examples=400, deadline=None, derandomize=True)
    @given(st.floats(allow_nan=False, allow_infinity=False, allow_subnormal=False), st.integers(min_value=0, max_value=9))
    def fixed(x, n):
        s = oio._rust_exp(x, n)
        mant, e10 = s.split("e")
        assert re.match(r"^-?\d" + (r"\.\d{%d}" % n if n else "") + "$", mant) and re.match(r"^-?(0|[1-9]\d*)$", e10), s
        if x != 0.0:
            exact = Decimal(x)
            e = exact.adjusted()
            q = (exact.scaleb(-e)).quantize(Decimal(1).scaleb(-n), rounding=ROUND_HALF_EVEN)
            if abs(q) >= 10:            # 9.99..5 rounded up to 10.0: one more power of ten
                q, e = (q / 10).quantize(Decimal(1).scaleb(-n), rounding=ROUND_HALF_EVEN), e + 1
            assert Decimal(mant) == q and int(e10) == e, (s, q, e)

    shortest()
    fixed()
