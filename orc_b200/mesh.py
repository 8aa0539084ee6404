"""Mirror of the reference's mesh data model (src/mesh.rs): Mesh, FaceZone, FaceConditionTypes."""
import ctypes as C
import enum

import numpy as np

from . import _lib


class FaceConditionTypes(enum.IntEnum):  # TGRID ids, src/mesh.rs:26-66
    Interior = 2
    Wall = 3
    PressureInlet = 4
    PressureOutlet = 5
    Symmetry = 7
    PeriodicShadow = 8
    PressureFarField = 9
    VelocityInlet = 10
    Periodic = 12
    PorousJump = 14
    MassFlowInlet = 20
    Interface = 24
    Parent = 31
    Outflow = 36
    Axis = 37


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class ScalarCondition(enum.IntEnum):
    """Condition of a boundary zone for the passive scalar (include/orc_b200.h ORC_SBC_*; not part of the reference)."""
    ZeroGradient = 0
    Fixed = 1


class FaceZoneView:
    """`mesh.get_face_zone(name)` of the reference (src/mesh.rs:189-195) returns a &mut FaceZone; assignments to
    zone_type / scalar_value / vector_value go through orc_mesh_set_zone."""

    def __init__(self, mesh, name):
        object.__setattr__(self, "_mesh", mesh)
        object.__setattr__(self, "name", name)

    def _get(self):
        z = self._mesh.zones()
        k = z["names"].index(self.name)
        return int(z["types"][k]), float(z["scalar"][k]), tuple(float(x) for x in z["vector"][k])

    @property
    def zone_type(self):
        return FaceConditionTypes(self._get()[0])

    @property
    def scalar_value(self):
        return self._get()[1]

    @property
    def vector_value(self):
        return self._get()[2]

    def __setattr__(self, key, value):
        t, s, v = self._get()
        if key == "zone_type":
            t = int(value)
        elif key == "scalar_value":
            s = float(value)
        elif key == "vector_value":
            v = tuple(float(x) for x in value)
        else:
            raise AttributeError(key)
        self._mesh.set_zone(self.name, t, s, v)


class Mesh:
    """Host mesh handle (orc_mesh). Geometry, the shared CSR pattern, the face->nnz scatter map and the assembly level
    schedule are built on the host when the mesh is created; the device mirror is created lazily by the first compute call."""

    def __init__(self, handle):
        self._h = handle
        self._ctxs = []   # contexts that hold this mesh's device mirror: they must outlive the handle (orc_mesh_free syncs their stream)

    def _bind(self, ctx):
        if all(c is not ctx for c in self._ctxs):
            self._ctxs.append(ctx)
        return self

    @classmethod
    def from_arrays(cls, dims, xyz, face_node_offsets, face_nodes, c0, c1, face_zone, zone_ids, zone_types, zone_names):
        out = C.c_void_p()
        xyz = _f64(xyz)
        fo, fn, a0, a1, fz = _i64(face_node_offsets), _i64(face_nodes), _i64(c0), _i64(c1), _i64(face_zone)
        zi, zt = _i64(zone_ids), _i64(zone_types)
        names = (C.c_char_p * len(zone_names))(*[n.encode() for n in zone_names])
        _lib.check(_lib.lib().orc_mesh_from_arrays(C.c_int32(dims), C.c_int64(xyz.size // 3), _p(xyz), C.c_int64(a0.size), _p(fo), _p(fn),
                                                   _p(a0), _p(a1), _p(fz), C.c_int64(zi.size), _p(zi), _p(zt), names, C.byref(out)))
        return cls(out)

    @classmethod
    def from_geometry(cls, dims, geometry, zone_ids, zone_types, zone_names):
        """A mesh from the reference's own flattened Mesh: `geometry` is the dict that `export()` returns (face_c0, face_c1,
        face_zone, face_area, face_normal, face_centroid, cell_volume, cell_centroid, cell_face_offsets, cell_face_indices).
        Nothing is recomputed (include/orc_b200.h: orc_mesh_from_geometry)."""
        g = geometry
        out = C.c_void_p()
        c0, c1, fz = _i64(g["face_c0"]), _i64(g["face_c1"]), _i64(g["face_zone"])
        fa, fn, fc = _f64(g["face_area"]), _f64(g["face_normal"]), _f64(g["face_centroid"])
        cv, cc = _f64(g["cell_volume"]), _f64(g["cell_centroid"])
        co, ci = _i64(g["cell_face_offsets"]), _i64(g["cell_face_indices"])
        zi, zt = _i64(zone_ids), _i64(zone_types)
        names = (C.c_char_p * len(zone_names))(*[n.encode() for n in zone_names])
        _lib.check(_lib.lib().orc_mesh_from_geometry(C.c_int32(dims), C.c_int64(cv.size), C.c_int64(c0.size), _p(c0), _p(c1), _p(fz), _p(fa),
                                                     _p(fn), _p(fc), _p(cv), _p(cc), _p(co), _p(ci), C.c_int64(zi.size), _p(zi), _p(zt),
                                                     names, C.byref(out)))
        return cls(out)

    @property
    def handle(self):
        return self._h

    def __del__(self):
        try:
            if self._h:
                _lib.lib().orc_mesh_free(self._h)
                self._h = None
        except Exception:
            pass

    def counts(self):
        d = np.zeros(8, np.int64)
        _lib.check(_lib.lib().orc_mesh_counts(self._h, _p(d)))
        return dict(cells=int(d[0]), faces=int(d[1]), nodes=int(d[2]), zones=int(d[3]), cell_faces=int(d[4]), dims=int(d[5]),
                    nnz=int(d[6]), levels=int(d[7]))

    @property
    def n_cells(self):
        return self.counts()["cells"]

    def export(self):
        c = self.counts()
        nf, nc = c["faces"], c["cells"]
        out = dict(face_c0=np.zeros(nf, np.int64), face_c1=np.zeros(nf, np.int64), face_zone=np.zeros(nf, np.int64), face_area=np.zeros(nf),
                   face_normal=np.zeros((nf, 3)), face_centroid=np.zeros((nf, 3)), cell_volume=np.zeros(nc), cell_centroid=np.zeros((nc, 3)),
                   cell_face_offsets=np.zeros(nc + 1, np.int64), cell_face_indices=np.zeros(c["cell_faces"], np.int64))
        _lib.check(_lib.lib().orc_mesh_export(self._h, *[_p(out[k]) for k in (
            "face_c0", "face_c1", "face_zone", "face_area", "face_normal", "face_centroid", "cell_volume", "cell_centroid",
            "cell_face_offsets", "cell_face_indices")]))
        return out

    def geometry_on_device(self, ctx=None):
        """The geometry pass of read_mesh (src/io.rs:289-438) recomputed on the device from the node coordinates: a dict like
        export()'s geometry entries plus "device_ms". Bit-identical to the host pass."""
        from .context import default_context
        ctx = ctx or default_context()
        c = self.counts()
        nf, nc = c["faces"], c["cells"]
        out = dict(face_area=np.zeros(nf), face_normal=np.zeros((nf, 3)), face_centroid=np.zeros((nf, 3)), cell_volume=np.zeros(nc),
                   cell_centroid=np.zeros((nc, 3)))
        ms = C.c_double()
        _lib.check(_lib.lib().orc_mesh_geometry_device(ctx.handle, self._h, _p(out["face_area"]), _p(out["face_normal"]), _p(out["face_centroid"]),
                                                       _p(out["cell_volume"]), _p(out["cell_centroid"]), C.byref(ms)))
        out["device_ms"] = ms.value
        return out

    def zones(self):
        nz = self.counts()["zones"]
        ids, types, sc, vec = np.zeros(nz, np.int64), np.zeros(nz, np.int64), np.zeros(nz), np.zeros((nz, 3))
        names = C.create_string_buffer(64 * max(nz, 1))
        _lib.check(_lib.lib().orc_mesh_zones(self._h, _p(ids), _p(types), _p(sc), _p(vec), names))
        nm = [names.raw[64 * k:64 * (k + 1)].split(b"\0")[0].decode() for k in range(nz)]
        return dict(ids=ids, types=types, scalar=sc, vector=vec, names=nm)

    def set_zone(self, name, zone_type, scalar=0.0, vector=(0.0, 0.0, 0.0)):
        _lib.check(_lib.lib().orc_mesh_set_zone(self._h, name.encode(), C.c_int64(int(zone_type)), C.c_double(scalar),
                                                C.c_double(vector[0]), C.c_double(vector[1]), C.c_double(vector[2])))

    def set_zone_scalar(self, name, kind, value=0.0):
        """The passive scalar condition of zone `name` (every zone starts as ZeroGradient): ScalarCondition.Fixed holds phi = value
        on the zone's faces. Partitions taken afterwards inherit it."""
        _lib.check(_lib.lib().orc_mesh_set_zone_scalar(self._h, name.encode(), C.c_int32(int(kind)), C.c_double(value)))

    def get_face_zone(self, name):  # src/mesh.rs:189-195
        if name not in self.zones()["names"]:
            raise _lib.OrcError(_lib.E_INVALID, f"face zone '{name}' should exist in mesh")
        return FaceZoneView(self, name)

    def pattern(self):
        c = self.counts()
        rp, co = np.zeros(c["cells"] + 1, np.int64), np.zeros(c["nnz"], np.int64)
        _lib.check(_lib.lib().orc_mesh_pattern(self._h, _p(rp), _p(co)))
        return rp, co

    def levels(self):
        lv = np.zeros(self.n_cells, np.int64)
        _lib.check(_lib.lib().orc_mesh_levels(self._h, _p(lv)))
        return lv


    # ---- multi-GPU: row-range partition (include/orc_b200.h: orc_mesh_partition*) ----
    def partition(self, rank, nranks):
        """This rank's share of the mesh: [lower halo | owned | upper halo] cells + the halo-exchange plan. BCs set on this
        (global) mesh so far are inherited; later changes must be applied to the partition as well."""
        out = C.c_void_p()
        _lib.check(_lib.lib().orc_mesh_partition(self._h, C.c_int32(rank), C.c_int32(nranks), C.byref(out)))
        return Mesh(out)

    def partition_window(self, rank, nranks, cuts, id_offset, n_global):
        """Like partition(), but `self` is only a window of the global mesh (see orc_mesh_partition_window)."""
        out = C.c_void_p()
        cu = _i64(cuts)
        assert cu.size == nranks + 1
        _lib.check(_lib.lib().orc_mesh_partition_window(self._h, C.c_int32(rank), C.c_int32(nranks), _p(cu), C.c_int64(id_offset),
                                                        C.c_int64(n_global), C.byref(out)))
        return Mesh(out)

    def partition_info(self):
        d = np.zeros(8, np.int64)
        _lib.check(_lib.lib().orc_mesh_partition_info(self._h, _p(d)))
        return dict(g0=int(d[0]), g1=int(d[1]), n_lo=int(d[2]), n_own=int(d[3]), n_hi=int(d[4]), neighbours=int(d[5]), n_send=int(d[6]),
                    n_global=int(d[7]))

    def partition_maps(self):
        i = self.partition_info()
        nloc, nn = i["n_lo"] + i["n_own"] + i["n_hi"], i["neighbours"]
        l2g = np.zeros(nloc, np.int64)
        nbr, sp, rb, rc = np.zeros(nn, np.int32), np.zeros(nn + 1, np.int32), np.zeros(nn, np.int32), np.zeros(nn, np.int32)
        si = np.zeros(max(i["n_send"], 1), np.int32)
        _lib.check(_lib.lib().orc_mesh_partition_maps(self._h, _p(l2g), _p(nbr), _p(sp), _p(si), _p(rb), _p(rc)))
        return dict(local_to_global=l2g, nbr_rank=nbr, send_ptr=sp, send_idx=si[:i["n_send"]], recv_begin=rb, recv_count=rc)
