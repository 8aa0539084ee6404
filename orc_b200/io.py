"""Mirror of the reference's io::read_mesh (src/io.rs:32-515): TGRID/Fluent ASCII .msh reader + geometry."""
import ctypes as C

from . import _lib
from .mesh import Mesh


def read_mesh(mesh_path):
    out = C.c_void_p()
    _lib.check(_lib.lib().orc_mesh_read(str(mesh_path).encode(), C.byref(out)))
    return Mesh(out)


# ---- solution data files (src/io.rs:519-620): the reference's only persistence, a text checkpoint ------------------------------
def _rust_exp(x, precision=None):
    """Rust's `{:e}` / `{:.Ne}` for an f64: shortest round-trip digits (or N decimals, correctly rounded), exponent without sign
    padding: 1e0, -4.2e-4, 1.2345e3, 0e0, NaN, inf."""
    x = float(x)
    if x != x:
        return "NaN"
    if x in (float("inf"), float("-inf")):
        return "inf" if x > 0 else "-inf"
    if precision is None:   # repr() holds the shortest round-trip digits; only their arrangement differs from Rust's
        s = repr(x)
        neg = s[0] == "-"
        if neg:
            s = s[1:]
        if "e" in s:
            mant, e = s.split("e")
            e10 = int(e)
            digits = mant.replace(".", "")
        else:
            ip, _, fp = s.partition(".")
            ip = ip.lstrip("0")
            if ip:
                digits, e10 = ip + fp, len(ip) - 1
            else:
                digits = fp.lstrip("0")
                if not digits:
                    return "-0e0" if neg else "0e0"
                e10 = -(len(fp) - len(digits) + 1)
        digits = digits.rstrip("0") or "0"
        out = digits[0] + ("." + digits[1:] if len(digits) > 1 else "") + "e" + str(e10)
        return "-" + out if neg else out
    mant, e10 = format(x, f".{precision}e").split("e")
    return f"{mant}e{int(e10)}"


def _vector_display(x, y, z):   # impl Display for Vector (src/lib.rs:551-556)
    return f"({_rust_exp(x, 2)}, {_rust_exp(y, 2)}, {_rust_exp(z, 2)})"


def _owned_centroids(mesh):
    """Cell centroids of the cells a caller holds fields for: the owned cells of a partition mesh (its local cells are
    [lower halo | owned | upper halo]), all cells otherwise."""
    cc = mesh.export()["cell_centroid"]
    try:
        info = mesh.partition_info()
    except _lib.OrcError:
        return cc
    return cc[info["n_lo"]:info["n_lo"] + info["n_own"]]


def write_data(mesh, u, v, w, p, output_file_name, decimal_precision=None):
    """write_data (src/io.rs:572-591) / write_data_with_precision (:593-619) when `decimal_precision` is given: one line per cell,
    `centroid \\t (u, v, w) \\t p`. On a partition mesh the fields are the owned cells' and so are the lines: the rank files,
    concatenated in rank order, are the whole mesh's file."""
    import numpy as np
    cc = _owned_centroids(mesh).tolist()
    n = len(cc)
    cols = [np.asarray(a, dtype=np.float64).tolist() for a in (u, v, w, p)]
    if any(len(c) != n for c in cols):
        raise ValueError(f"u, v, w, p must hold {n} values, one per (owned) cell")
    e, prec = _rust_exp, decimal_precision
    if decimal_precision is None:
        print(f"Writing data to {output_file_name}...")
    with open(output_file_name, "w") as f:
        for lo in range(0, n, 65536):          # plain Python floats and one write per block: the loop is the cost at 10^6+ cells
            hi = min(lo + 65536, n)
            f.write("".join(f"({e(c[0], 2)}, {e(c[1], 2)}, {e(c[2], 2)})\t({e(a, prec)}, {e(b, prec)}, {e(g, prec)})\t{e(d, prec)}\n"
                            for c, a, b, g, d in zip(cc[lo:hi], cols[0][lo:hi], cols[1][lo:hi], cols[2][lo:hi], cols[3][lo:hi])))
    if decimal_precision is None:
        print("Done!")


def format_gradient_line(centroid, velocity_gradient9, pressure_gradient3, decimal_precision):
    """One line of write_gradients (src/io.rs:636-659). The reference strips the trailing ", " of each list and DISCARDS the
    result (`strip_suffix(..).unwrap();` as a statement), so the separators stay: `(a, b, ..., i, )`."""
    vg = "".join(f"{_rust_exp(x, decimal_precision)}, " for x in velocity_gradient9)
    pg = "".join(f"{_rust_exp(x, decimal_precision)}, " for x in pressure_gradient3)
    return f"{_vector_display(*centroid)}\t({vg})\t({pg})"


def write_gradients(mesh, u, v, w, p, output_file_name, decimal_precision, gradient_scheme, ctx=None):
    """write_gradients (src/io.rs:623-662), same argument order: per cell `centroid \t (grad u, row major) \t (grad p)`; the
    gradients come from the device (orc_gradients), Green-Gauss cell based or least squares."""
    from .discretization import calculate_gradients
    gp, gu = calculate_gradients(mesh, u, v, w, p, gradient_scheme, ctx)
    _write_gradient_lines(output_file_name, mesh.export()["cell_centroid"], gp, gu, decimal_precision)


def _write_gradient_lines(output_file_name, centroids, gp, gu, decimal_precision):
    n = len(centroids)
    cc, gul, gpl = centroids.tolist(), gu.reshape(n, 9).tolist(), gp.tolist()
    print(f"Writing data to {output_file_name}...")
    with open(output_file_name, "w") as f:
        for lo in range(0, n, 65536):
            hi = min(lo + 65536, n)
            f.write("".join(format_gradient_line(c, a, b, decimal_precision) + "\n" for c, a, b in zip(cc[lo:hi], gul[lo:hi], gpl[lo:hi])))


def read_data(data_file_path):
    """read_data (src/io.rs:519-570) -> (u, v, w, p); raises OSError("could not read data file") like the reference's Err."""
    import numpy as np
    u, v, w, p = [], [], [], []
    try:
        f = open(data_file_path)
    except OSError:
        raise OSError("could not read data file")
    with f:
        print(f"Reading solution data from {data_file_path}...")
        for line in f:
            chunks = line.rstrip("\n").split("\t", 2)           # splitn(3, '\t'): column 0 (the centroid) is ignored
            if len(chunks) > 1:
                if not (chunks[1].startswith("(") and chunks[1].endswith(")")):
                    raise ValueError("called `Option::unwrap()` on a `None` value")   # Vector::parse (src/lib.rs:319-333)
                x, y, z = (float(s) for s in chunks[1][1:-1].split(", ", 2))
                u.append(x); v.append(y); w.append(z)
            if len(chunks) > 2:
                p.append(float(chunks[2]))
        print("Done!")
    return tuple(np.array(a, dtype=np.float64) for a in (u, v, w, p))
