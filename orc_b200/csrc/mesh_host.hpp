// mesh_host.hpp — host-side mesh model of liborc_b200: the reference's AoS Mesh (src/mesh.rs:12-187)
// flattened to SoA arrays sized for multi-million-cell meshes, plus everything the device path
// precomputes once per mesh: the shared CSR pattern, the (cell, face) -> nnz scatter map that replaces
// the reference's get_entry_mut binary searches (src/discretization.rs:312-350), and the level
// schedule that makes the momentum-assembly recurrence (SURVEY.md Q2) parallel without changing it.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

namespace orc {

struct MeshError : std::runtime_error {
    int code;
    MeshError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct HostZone {  // src/mesh.rs:12-17
    int64_t id = 0;
    int32_t type = 3;
    double scalar = 0.;
    double vec[3] = {0., 0., 0.};
    std::string name;
    // passive scalar condition of the zone (orc_mesh_set_zone_scalar; not part of the reference's FaceZone)
    int32_t scalar_bc_kind = 0;     // ORC_SBC_ZERO_GRADIENT / ORC_SBC_FIXED
    double scalar_bc_value = 0.;
};

struct HostMesh {
    int32_t dims = 3;
    int64_t n_nodes = 0, n_faces = 0, n_cells = 0;
    std::vector<double> xyz;               // 3 * n_nodes
    std::vector<int64_t> face_node_ptr;    // n_faces + 1
    std::vector<int32_t> face_nodes;
    std::vector<int32_t> face_c0, face_c1; // cell_indices[0], cell_indices[1] (-1: boundary) AFTER io.rs:332-337
    std::vector<int32_t> face_zone;        // index into `zones`
    std::vector<uint8_t> face_flipped;     // 1: the file had no cell 0 on this face, the normal was flipped (io.rs:332-337)
    std::vector<double> face_area, face_normal, face_centroid;  // F, 3F (AoS xyz), 3F
    std::vector<double> cell_volume, cell_centroid;             // N, 3N
    std::vector<int32_t> cf_ptr, cf_face;  // cell -> faces, ascending face index (io.rs:404-411)
    std::vector<HostZone> zones;           // ascending zone id
    uint64_t zone_epoch = 1;               // bumped by set_zone: device zone table is refreshed lazily
    int64_t own_lo = 0, own_hi = -1;       // owned cell range of a partition mesh (own_hi < 0: the whole mesh is owned)

    // ---- derived once per mesh ----
    std::vector<int32_t> cf_nb;    // per (cell, face-slot): neighbour cell or -1
    std::vector<int32_t> cf_slot;  // per (cell, face-slot): nnz index of (cell, nb) in the shared pattern, or -1
    std::vector<int32_t> rowptr, col, diag_idx;  // shared pattern: diag + face neighbours, columns sorted
    std::vector<int32_t> level_of_cell, level_ptr, level_order;  // cells grouped by assembly level
    int64_t nnz() const { return (int64_t)col.size(); }

    int find_zone(const std::string& name) const;  // mesh.rs:189-195, -1 if absent
};

// src/io.rs:32-287 (TGRID ASCII sections) + :289-438 (geometry)
HostMesh* read_tgrid(const std::string& path);
HostMesh* mesh_from_arrays(int32_t dims, int64_t n_nodes, const double* xyz, int64_t n_faces, const int64_t* face_node_offsets,
                           const int64_t* face_nodes, const int64_t* c0, const int64_t* c1, const int64_t* face_zone,
                           int64_t n_zones, const int64_t* zone_ids, const int64_t* zone_types, const char* const* zone_names);

// the reference's own Mesh, flattened by the caller (geometry included; no nodes): SURVEY.md §8b orc_mesh_view
HostMesh* mesh_from_geometry(int32_t dims, int64_t n_cells, int64_t n_faces, const int64_t* face_c0, const int64_t* face_c1,
                             const int64_t* face_zone, const double* face_area, const double* face_normal3, const double* face_centroid3,
                             const double* cell_volume, const double* cell_centroid3, const int64_t* cell_face_offsets,
                             const int64_t* cell_face_indices, int64_t n_zones, const int64_t* zone_ids, const int64_t* zone_types,
                             const char* const* zone_names);

}  // namespace orc

namespace orc {
// Row-range partition of a mesh (SURVEY.md §8e): rank r owns the global cells [g0, g1); its local mesh holds
// [lower halo | owned | upper halo] in ascending GLOBAL id (so column order, hence summation order, is unchanged),
// every face of an owned cell, and the geometry of all local cells copied from the global mesh (bit-identical).
// Halo cells carry no face list and no matrix row. The level schedule only follows OWNED lower neighbours: lower-halo
// neighbours are "partition-lagged" (C4) — they are read in the state of the last halo exchange.
struct PartPlan {
    int32_t rank = 0, nranks = 1;
    int64_t g0 = 0, g1 = 0;            // owned global range
    int64_t n_global = 0;
    int64_t n_lo = 0, n_own = 0, n_hi = 0;
    std::vector<int64_t> local_to_global;          // n_lo + n_own + n_hi
    // per neighbour rank q (ascending): cells I send (local ids of owned cells, ascending global id) and the contiguous
    // slice of my halo [recv_begin, recv_begin + recv_count) (local ids) that q fills, in ascending global id
    std::vector<int32_t> nbr_rank;
    std::vector<int32_t> send_ptr, send_idx;       // CSR over neighbours
    std::vector<int32_t> recv_begin, recv_count;
};
// `cuts` (nranks + 1 ascending cell indices of `g`, clamped to [0, n_cells]) says who owns what: rank q owns [cuts[q], cuts[q+1]).
// `g` may be the whole mesh or only a window of it that contains this rank's cells and their face neighbours (a slab of a
// structured box): `id_offset` is the global id of g's cell 0 and `n_global` the global cell count.
HostMesh* extract_partition(const HostMesh& g, int32_t rank, int32_t nranks, const std::vector<int64_t>& cuts, int64_t id_offset,
                            int64_t n_global, PartPlan& plan);
inline std::vector<int64_t> even_cuts(int64_t n, int32_t nranks) {
    // even cut points (coarse rows i/2 stay aligned, SURVEY.md §8e)
    std::vector<int64_t> c(nranks + 1);
    for (int32_t r = 0; r <= nranks; ++r) c[r] = (r == nranks) ? n : ((n * r / nranks) & ~int64_t(1));
    return c;
}
}  // namespace orc
