// Refinement (the `r` command: 1 -> 4 midpoint subdivision) on plain global arrays, shared by the device kernels and
// the test-only host emulator; and the Morton key of the internal vertex order, shared with morton_permutation.
//
// Reference: geometry/refine.py (refine_triangles), the host twin.  One level, in the CALLER's vertex numbering:
//   1. every half-edge h = 3 f + k (tri[f][k] -> tri[f][k+1], the twin's edge k of facet f) gets the key
//      min*nv + max of its end points (EqMesh::key_id maps a row id to the caller's id); (key, h) pairs are sorted;
//   2. the e-th distinct key in ascending order is edge e: its midpoint is vertex nv + e, as np.unique numbers them;
//   3. old vertex v keeps its caller id; the midpoint of edge a-b is 0.5 * (pos[a] + pos[b]) (no fused multiply-add),
//      fixed when both ends are, and a boundary vertex when both ends are and the edge has a single half-edge;
//   4. facet f = (v0, v1, v2) becomes rows f, nf + f, 2 nf + f, 3 nf + f:
//      (v0, m01, m20), (v1, m12, m01), (v2, m20, m12), (m01, m12, m20).
#pragma once

#include "ms_equiangulate.cuh"

namespace ms {

// One level of refinement: the mesh, its sorted half-edge keys (m.keys / m.order) and the edges they define.
struct RfMesh {
  EqMesh m;                 // rows, positions, fixed mask (may be null), caller numbering, sorted keys and half-edges
  const uint8_t* boundary;  // nv boundary flags or nullptr
  const int32_t* head;      // n_edges + 1: sorted position where the run of edge e starts; head[n_edges] = 3 nf
  const int32_t* edge;      // 3 nf: edge of half-edge h
  int32_t n_edges;
};

// The refined mesh in the caller's numbering: nv + n_edges vertex rows, 4 nf facet rows.
struct RfOut {
  double* pos;
  uint8_t* fixed;     // written when m.fixed is set
  uint8_t* boundary;  // written when RfMesh::boundary is set
  int32_t* tri;
};

MS_HD int32_t rf_caller(const EqMesh& m, int32_t v) { return m.key_id ? m.key_id[v] : v; }

// sorted position i opens the run of a new key
MS_HD bool rf_head(const uint64_t* keys, int64_t i) { return i == 0 || keys[i] != keys[i - 1]; }

// Vertex row v of the mesh, copied to its caller id.
MS_HD void rf_vertex(const RfMesh& r, const RfOut& o, int32_t v) {
  const size_t j = size_t(rf_caller(r.m, v));
  for (int k = 0; k < 3; ++k) o.pos[3 * j + k] = r.m.pos[3 * size_t(v) + k];
  if (r.m.fixed) o.fixed[j] = r.m.fixed[v];
  if (r.boundary) o.boundary[j] = r.boundary[v];
}

// The midpoint of edge e: vertex nv + e.  Its ends are read from the first half-edge of the run.
MS_HD void rf_midpoint(const RfMesh& r, const RfOut& o, int32_t e) {
  const int32_t s = r.head[e];
  const int64_t h = r.m.order[s];
  const int a = eq_tail(r.m, h), b = eq_head(r.m, h);
  const size_t j = size_t(r.m.nv) + size_t(e);
  for (int k = 0; k < 3; ++k)
    o.pos[3 * j + k] = eq_mul(0.5, eq_add(r.m.pos[3 * size_t(a) + k], r.m.pos[3 * size_t(b) + k]));
  if (r.m.fixed) o.fixed[j] = uint8_t(r.m.fixed[a] && r.m.fixed[b]);
  if (r.boundary) o.boundary[j] = uint8_t(r.head[e + 1] - s == 1 && r.boundary[a] && r.boundary[b]);
}

// The four children of facet f.
MS_HD void rf_children(const RfMesh& r, const RfOut& o, int32_t f) {
  const size_t nf = size_t(r.m.nf), f3 = 3 * size_t(f);
  const int32_t v0 = rf_caller(r.m, r.m.tri[f3]), v1 = rf_caller(r.m, r.m.tri[f3 + 1]),
                v2 = rf_caller(r.m, r.m.tri[f3 + 2]);
  const int32_t m01 = r.m.nv + r.edge[f3], m12 = r.m.nv + r.edge[f3 + 1], m20 = r.m.nv + r.edge[f3 + 2];
  const int32_t rows[4][3] = {{v0, m01, m20}, {v1, m12, m01}, {v2, m20, m12}, {m01, m12, m20}};
  for (size_t q = 0; q < 4; ++q)
    for (int k = 0; k < 3; ++k) o.tri[3 * (q * nf + size_t(f)) + k] = rows[q][k];
}

// --- Morton (Z-curve) order of positions: the bounding box, then 21 bits per axis interleaved ---
struct MortonBox {
  double lo[3], hi[3];
};

MS_HD MortonBox morton_box_empty() { return MortonBox{{1e300, 1e300, 1e300}, {-1e300, -1e300, -1e300}}; }

// Adds a point; NaN coordinates are skipped.  Any grouping of the additions gives the same box (up to the sign of a
// zero bound, which changes no key).
MS_HD void morton_box_add(MortonBox& b, const double* p) {
  for (int k = 0; k < 3; ++k) {
    if (p[k] < b.lo[k]) b.lo[k] = p[k];
    if (p[k] > b.hi[k]) b.hi[k] = p[k];
  }
}

MS_HD void morton_box_merge(MortonBox& b, const MortonBox& o) {
  for (int k = 0; k < 3; ++k) {
    if (o.lo[k] < b.lo[k]) b.lo[k] = o.lo[k];
    if (o.hi[k] > b.hi[k]) b.hi[k] = o.hi[k];
  }
}

MS_HD uint64_t morton_spread(uint64_t x) {
  x &= 0x1FFFFFull;
  x = (x | (x << 32)) & 0x1F00000000FFFFull;
  x = (x | (x << 16)) & 0x1F0000FF0000FFull;
  x = (x | (x << 8)) & 0x100F00F00F00F00Full;
  x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
  x = (x | (x << 2)) & 0x1249249249249249ull;
  return x;
}

MS_HD uint64_t morton_key(const MortonBox& b, const double* p) {
  uint64_t q[3];
  for (int k = 0; k < 3; ++k) {
    const double span = eq_sub(b.hi[k], b.lo[k]);
    double t = span > 0 ? eq_mul(eq_sub(p[k], b.lo[k]) / span, 2097151.0) : 0.0;
    if (!(t >= 0)) t = 0;  // also catches NaN
    if (t > 2097151.0) t = 2097151.0;
    q[k] = uint64_t(t);
  }
  return morton_spread(q[0]) | (morton_spread(q[1]) << 1) | (morton_spread(q[2]) << 2);
}

}  // namespace ms
