// Host-side packing of a triangle mesh into shared-memory sized vertex patches.
//
// The context packs on the device (ms_pack_device.cuh), byte for byte this layout; pack_patches stays as the
// reference the emulator and the tests compare against (its MS_PACK_THREADS knob concerns only this host version).
//
// This replaces, for the device path, what geometry/triangle_rows.py:10-35 and
// Mesh.triangle_row_cache (geometry/mesh.py:597-624) do for the reference: it
// turns the (nf,3) int32 triangle rows into the layout the kernels stream.
//
// A patch owns a contiguous range of vertex rows and lists every facet touching
// an owned vertex (ring facets are listed by each patch that touches them).
// Facets of a patch are scheduled in ROUNDS: within one round no two facets write
// the same owned vertex, so a CTA can accumulate corner contributions into shared
// memory with plain read-modify-writes, without atomics, in an order fixed at pack
// time -> run-to-run reproducible results.
#pragma once

#include <stdint.h>

#include <vector>

namespace ms {

struct PatchHeader {  // 32 bytes
  int32_t v_lo;       // first owned vertex row
  int32_t n_owned;    // owned vertices [v_lo, v_lo + n_owned)
  int32_t halo_off;   // first entry of this patch in halo_ids
  int32_t n_halo;     // local index n_owned + j  ->  vertex row halo_ids[halo_off + j]
  int64_t slot_off;   // first record slot of this patch
  int32_t reserved;
  int32_t n_rounds;   // round r holds the `threads` slots [slot_off + r*threads, slot_off + (r+1)*threads);
                      // slots without a facet carry flags == 0
};
static_assert(sizeof(PatchHeader) == 32, "PatchHeader layout");

// One record slot.  flags bit0: valid (0 marks an empty slot); bit1: primary (this patch owns
// the facet's first vertex, so per-facet scalars are summed here exactly once); bit2: facet
// belongs to the body.  (a,b,c) may be a cyclic rotation of the facet's vertex order.
struct FacetRec {
  uint16_t a, b, c;  // patch-local vertex indices (owned first, then halo)
  uint16_t flags;
};
static_assert(sizeof(FacetRec) == 8, "FacetRec layout");

enum : uint16_t { REC_VALID = 1, REC_PRIMARY = 2, REC_BODY = 4 };

struct PackParams {
  int32_t threads = 96;      // record slots per round (= lanes of one consumer group)
  int32_t max_owned = 512;   // owned vertices per patch
  int32_t max_local = 896;   // owned + halo vertices per patch (shared-memory budget)
  int32_t max_slots = 1536;  // record slots per patch (rounds x threads; shared-memory budget)
  int32_t repair_sweeps = 1; // lane-placement repair passes (0 = greedy only)
  int32_t fill_pct = 87;     // target share of valid slots: lower = more free lanes = fewer bank clashes
};

struct PackedMesh {
  int32_t nv = 0, nf = 0;
  int32_t n_owned_vertices = 0;  // rows [0, n_owned_vertices) belong to patches
  PackParams params;
  std::vector<PatchHeader> patches;
  std::vector<int32_t> halo_ids;
  std::vector<FacetRec> recs;
  std::vector<int32_t> slot_facet;  // facet row of each slot
  int32_t max_owned = 0, max_local = 0, max_rounds = 0, max_slots = 0;
  int64_t n_round_slots = 0;  // sum over patches of n_rounds * threads (== recs.size())
  int64_t n_lane_conflicts = 0;  // corner placements that share a bank residue inside a half-warp
  int64_t n_hw_groups = 0;  // (round, half-warp, corner position) gather groups holding a facet
  int64_t n_hw_excess = 0;  // extra shared-memory wavefronts over those groups (0 = conflict free)
  int64_t n_listed = 0;   // facet listings over all patches (>= valid facets)
  int64_t n_valid = 0;    // facets with all indices in range
};

// body_mask: nf bytes (nonzero = facet in the body) or nullptr (no facet flagged).
// Facets with an index outside [0,nv) are skipped, like surface_energy.f90:57-59; so are facets that name
// one vertex twice: they have zero area and volume and their curvature / gradient contributions vanish
// identically (every term carries a factor e_k = 0 or fK_i - fK_i = 0), in the reference as well.
// Returns 0, or a negative error code (-1 bad arguments, -2 a single vertex needs
// more than max_local local vertices, -3 a single vertex needs more than max_slots slots).
// n_owned_vertices (multi-GPU partitions): only vertex rows [0, n_owned_vertices) are owned
// by patches; rows beyond are ghost vertices of neighbouring partitions, referenced as halo
// only.  Facets without an owned vertex are not listed.  -1 = all vertices are owned.
int pack_patches(int32_t nv, int32_t nf, const int32_t* tri, const uint8_t* body_mask,
                 const PackParams& params, PackedMesh& out, int32_t n_owned_vertices = -1);

// Vertex -> corner incidence in CSR form, facet-major order, for the generic
// (stateless) kernels.  corner id = 3*facet + column.
void build_corner_csr(int32_t nv, int32_t nf, const int32_t* tri, std::vector<int32_t>& ptr,
                      std::vector<int32_t>& idx);

}  // namespace ms
