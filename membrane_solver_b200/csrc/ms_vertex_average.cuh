// Evolver-style vertex averaging (the `V` command) on plain global arrays, shared by the device kernel
// and the test-only host emulator.
//
// Reference: runtime/vertex_average.py:28-120, restated for arrays by geometry/vertex_average.py
// (vertex_average_arrays).  Every edge {v,u} gets the weight w = sum of the areas of the facets that list it
// (areas of the positions before the call); a movable vertex with at least two usable edges moves to
//
//     x_v + 1/4 * sum_u w^2 (x_u - x_v) / sum_u w^2        (Jacobi: every vertex reads the old positions).
//
// Each vertex finds its edges in its own corner list: the two edges of corner (f,k) are (v, tri[f][k+1]) and
// (v, tri[f][k+2]), and both facets of an interior edge are incident to v.  Neighbours are merged by an O(d^2)
// scan of the corner list, so the valence is not capped.  The weights are summed in corner (= facet) order and
// nothing is accumulated across threads: the result is bitwise repeatable.
#pragma once

#include "ms_math.cuh"

namespace ms {

struct VaMesh {
  int32_t nv;
  const int32_t* tri;      // (nf,3)
  const double* pos;       // (nv,3) positions before the call
  const int32_t* csr_ptr;  // vertex -> corners (corner id = 3 f + k), facet-major order; invalid facets absent
  const int32_t* csr_idx;
  const int32_t* group;    // nv pin groups (-1: none) or nullptr
  const uint8_t* fixed;    // nv or nullptr
};

MS_HD d3 va_row(const double* p, int i) { return make_d3(p[3 * size_t(i)], p[3 * size_t(i) + 1], p[3 * size_t(i) + 2]); }

// neighbour across edge s (0: next corner, 1: previous corner) of corner j of the CSR
MS_HD int va_neighbour(const VaMesh& m, int j, int s) {
  const int c = m.csr_idx[j];
  const int f = c / 3, k = c - 3 * f;
  return m.tri[3 * size_t(f) + size_t((k + 1 + s) % 3)];
}

// A_f = |(x1 - x0) x (x2 - x0)| / 2
MS_HD double va_facet_area(const VaMesh& m, int f) {
  const d3 a = va_row(m.pos, m.tri[3 * size_t(f)]), b = va_row(m.pos, m.tri[3 * size_t(f) + 1]),
           c = va_row(m.pos, m.tri[3 * size_t(f) + 2]);
  const d3 n = cross(b - a, c - a);
  return 0.5 * sqrt(n.x * n.x + n.y * n.y + n.z * n.z);
}

// New position of vertex v.
MS_HD d3 va_vertex(const VaMesh& m, int v) {
  const d3 xv = va_row(m.pos, v);
  if (m.fixed && m.fixed[v]) return xv;
  const int j0 = m.csr_ptr[v], j1 = m.csr_ptr[v + 1];
  const int gv = m.group ? m.group[v] : -1;
  int degree = 0, used = 0;
  double total = 0.0;
  d3 xsum = make_d3(0.0, 0.0, 0.0);
  for (int j = j0; j < j1; ++j)
    for (int s = 0; s < 2; ++s) {
      const int u = va_neighbour(m, j, s);
      bool seen = false;  // an earlier edge slot of v names u: that slot already counted the edge
      for (int i = j0; i <= j && !seen; ++i)
        for (int t = 0; t < 2 && !(i == j && t == s) && !seen; ++t) seen = va_neighbour(m, i, t) == u;
      if (seen) continue;
      if (u == v) {  // self-edge of a repeated-index facet: counted from both ends, zero area, never usable
        degree += 2;
        continue;
      }
      ++degree;
      double w = 0.0;  // every facet slot that lists {v,u} adds its facet's area once
      for (int i = j; i < j1; ++i) {
        const int hits = (va_neighbour(m, i, 0) == u) + (va_neighbour(m, i, 1) == u);
        if (hits) {
          const double a = va_facet_area(m, m.csr_idx[i] / 3);
          w += a;
          if (hits == 2) w += a;
        }
      }
      if (!(w > 0.0)) continue;
      if (gv >= 0 && m.group[u] != gv) continue;  // a grouped end only uses neighbours of its own group
      ++used;
      const double w2 = w * w;
      total += w2;
      const d3 xu = va_row(m.pos, u);
      xsum = xsum + make_d3(w2 * (xu.x - xv.x), w2 * (xu.y - xv.y), w2 * (xu.z - xv.z));
    }
  if (used > 1 && total >= 1.0e-15 && degree > 1)
    return make_d3(xv.x + 0.25 * xsum.x / total, xv.y + 0.25 * xsum.y / total, xv.z + 0.25 * xsum.z / total);
  return xv;
}

}  // namespace ms
