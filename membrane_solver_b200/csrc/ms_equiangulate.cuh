// Equiangulation (the `u` command: Delaunay edge flips) on plain global arrays, shared by the device kernels and
// the test-only host emulator.
//
// Reference: geometry/equiangulate.py (equiangulate_triangles), the host twin; its criterion restates
// runtime/equiangulation.py:151-233.  One sweep:
//   1. every half-edge h = 3 f + k (tri[f][k] -> tri[f][k+1]) gets the key min*nv + max of its end points in the
//      CALLER's vertex numbering; (key, h) pairs are sorted stably, so equal keys are ordered by h;
//   2. a key that occurs exactly twice with opposite directions is an interior edge (a, b, f1, f2, c, d); it is a
//      candidate when eq_should_flip holds (tangent-plane angle test, fixed ends, c != d, the new diagonal is not an
//      edge yet, both new triangles valid);
//   3. candidates are taken in ascending key; one is skipped when an earlier flip of the sweep touched one of its
//      facets or claimed its new diagonal.  That is the lexicographically first maximal independent set of the
//      conflict graph (shared facet, or same new diagonal), computed in rounds by eq_round;
//   4. the selected flips rewrite tri[f1] = (a, d, c) and tri[f2] = (b, c, d).
//
// The geometry repeats the twin's NumPy arithmetic operation for operation: no fused multiply-add, np.cross's
// products-then-difference, np.linalg.norm's sequential sum of squares and einsum's (x0 y0 + x2 y2) + x1 y1 for
// three-vectors.  The one operation that is not bitwise the twin's is arccos (the platform's acos against NumPy's),
// so a decision can differ only where an angle sum lies within a few ulp of pi + margin.
#pragma once

#include "ms_math.cuh"

namespace ms {

constexpr double kEqMargin = 1.0e-3;          // DELAUNAY_MARGIN of geometry/equiangulate.py
constexpr double kEqPi = 3.141592653589793;   // np.pi
enum : uint8_t { EQ_UNDECIDED = 0, EQ_SELECTED = 1, EQ_REJECTED = 2 };

// rounded products / sums that the compiler may not contract into an fma (the twin rounds every operation)
#ifdef __CUDA_ARCH__
MS_HD double eq_mul(double a, double b) { return __dmul_rn(a, b); }
MS_HD double eq_add(double a, double b) { return __dadd_rn(a, b); }
MS_HD double eq_sub(double a, double b) { return __dsub_rn(a, b); }
#else
MS_HD double eq_mul(double a, double b) { return a * b; }
MS_HD double eq_add(double a, double b) { return a + b; }
MS_HD double eq_sub(double a, double b) { return a - b; }
#endif

struct EqMesh {
  int32_t nv, nf;
  const int32_t* tri;        // (nf,3) rows; vertex ids index pos / fixed
  const double* pos;         // (nv,3)
  const uint8_t* fixed;      // nv or nullptr
  const int32_t* key_id;     // vertex id -> the caller's id used in keys (nullptr: the same)
  const uint64_t* keys;      // the 3 nf sorted half-edge keys
  const int32_t* order;      // half-edge of each sorted key
};

MS_HD int eq_tail(const EqMesh& m, int64_t h) { return m.tri[h]; }
MS_HD int eq_head(const EqMesh& m, int64_t h) { return m.tri[h - h % 3 + (h % 3 + 1) % 3]; }
MS_HD int eq_apex(const EqMesh& m, int64_t h) { return m.tri[h - h % 3 + (h % 3 + 2) % 3]; }

MS_HD uint64_t eq_key(const EqMesh& m, int u, int v) {
  const int64_t a = m.key_id ? m.key_id[u] : u, b = m.key_id ? m.key_id[v] : v;
  return uint64_t(a < b ? a : b) * uint64_t(m.nv) + uint64_t(a < b ? b : a);
}

// sorted position i opens a run of exactly two equal keys whose half-edges run in opposite directions
MS_HD bool eq_interior(const EqMesh& m, int64_t i, int64_t& h1, int64_t& h2) {
  const int64_t n = 3 * int64_t(m.nf);
  const uint64_t k = m.keys[i];
  if ((i > 0 && m.keys[i - 1] == k) || i + 1 >= n || m.keys[i + 1] != k || (i + 2 < n && m.keys[i + 2] == k)) return false;
  h1 = m.order[i];
  h2 = m.order[i + 1];
  return eq_tail(m, h1) == eq_head(m, h2) && eq_head(m, h1) == eq_tail(m, h2);
}

MS_HD bool eq_key_exists(const EqMesh& m, uint64_t k) {
  int64_t lo = 0, hi = 3 * int64_t(m.nf);
  while (lo < hi) {
    const int64_t mid = lo + (hi - lo) / 2;
    if (m.keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  return lo < 3 * int64_t(m.nf) && m.keys[lo] == k;
}

MS_HD d3 eq_row(const double* p, int i) { return make_d3(p[3 * size_t(i)], p[3 * size_t(i) + 1], p[3 * size_t(i) + 2]); }
MS_HD d3 eq_diff(d3 a, d3 b) { return make_d3(eq_sub(a.x, b.x), eq_sub(a.y, b.y), eq_sub(a.z, b.z)); }
MS_HD d3 eq_cross(d3 a, d3 b) {  // np.cross
  return make_d3(eq_sub(eq_mul(a.y, b.z), eq_mul(a.z, b.y)), eq_sub(eq_mul(a.z, b.x), eq_mul(a.x, b.z)),
                 eq_sub(eq_mul(a.x, b.y), eq_mul(a.y, b.x)));
}
MS_HD double eq_norm(d3 a) { return sqrt(eq_add(eq_add(eq_mul(a.x, a.x), eq_mul(a.y, a.y)), eq_mul(a.z, a.z))); }
MS_HD double eq_dot(d3 a, d3 b) { return eq_add(eq_add(eq_mul(a.x, b.x), eq_mul(a.z, b.z)), eq_mul(a.y, b.y)); }  // einsum
MS_HD d3 eq_div(d3 a, double s) { return make_d3(a.x / s, a.y / s, a.z / s); }

// the angle at q between the directions to x and y (2-D), and whether both legs are long enough
MS_HD double eq_angle(double qx, double qy, double xx, double xy, double yx, double yy, bool& good) {
  const double ax = eq_sub(xx, qx), ay = eq_sub(xy, qy), bx = eq_sub(yx, qx), by = eq_sub(yy, qy);
  const double na = sqrt(eq_add(eq_mul(ax, ax), eq_mul(ay, ay))), nb = sqrt(eq_add(eq_mul(bx, bx), eq_mul(by, by)));
  good = na >= 1e-12 && nb >= 1e-12;
  double c = eq_add(eq_mul(ax, bx), eq_mul(ay, by)) / (good ? eq_mul(na, nb) : 1.0);
  c = c < -1.0 ? -1.0 : (c > 1.0 ? 1.0 : c);  // np.clip keeps a NaN
  return acos(c);
}

// _should_flip: the angles opposite to edge a-b, at c and d, add up to more than pi + margin in the tangent plane
MS_HD bool eq_delaunay_violated(const EqMesh& m, int a, int b, int c, int d) {
  const d3 p1 = eq_row(m.pos, a), p2 = eq_row(m.pos, b), p3 = eq_row(m.pos, c), p4 = eq_row(m.pos, d);
  const d3 n1 = eq_cross(eq_diff(p2, p1), eq_diff(p3, p1)), n2 = eq_cross(eq_diff(p4, p1), eq_diff(p2, p1));
  d3 n = make_d3(eq_add(n1.x, n2.x), eq_add(n1.y, n2.y), eq_add(n1.z, n2.z));
  double nn = eq_norm(n);
  if (nn < 1e-12) { n = n1; nn = eq_norm(n1); }
  if (nn < 1e-12) { n = n2; nn = eq_norm(n2); }
  bool valid = nn >= 1e-12;
  n = eq_div(n, valid ? nn : 1.0);
  const d3 e = eq_diff(p2, p1);
  const double en = eq_norm(e);
  valid = valid && en >= 1e-12;
  const d3 u = eq_div(e, en >= 1e-12 ? en : 1.0);
  d3 v = eq_cross(n, u);
  const double vn = eq_norm(v);
  valid = valid && vn >= 1e-12;
  v = eq_div(v, vn >= 1e-12 ? vn : 1.0);
  const d3 r2 = eq_diff(p2, p1), r3 = eq_diff(p3, p1), r4 = eq_diff(p4, p1);
  const double q2x = eq_dot(r2, u), q2y = eq_dot(r2, v), q3x = eq_dot(r3, u), q3y = eq_dot(r3, v),
               q4x = eq_dot(r4, u), q4y = eq_dot(r4, v);
  bool g1 = false, g2 = false;
  const double t1 = eq_angle(q3x, q3y, 0.0, 0.0, q2x, q2y, g1), t2 = eq_angle(q4x, q4y, 0.0, 0.0, q2x, q2y, g2);
  return valid && g1 && g2 && eq_add(t1, t2) > kEqPi + kEqMargin;
}

// _unit_normals of one row
MS_HD d3 eq_unit_normal(const EqMesh& m, int i, int j, int k, double& mag) {
  const d3 p = eq_row(m.pos, i);
  const d3 n = eq_cross(eq_diff(eq_row(m.pos, j), p), eq_diff(eq_row(m.pos, k), p));
  mag = eq_norm(n);
  return eq_div(n, mag > 0 ? mag : 1.0);
}

// The whole candidate test of the interior edge (h1, h2): a -> b in f1 with apex c, b -> a in f2 with apex d.
MS_HD bool eq_should_flip(const EqMesh& m, int64_t h1, int64_t h2) {
  const int a = eq_tail(m, h1), b = eq_head(m, h1), c = eq_apex(m, h1), d = eq_apex(m, h2);
  if (c == d) return false;
  if (m.fixed && m.fixed[a] && m.fixed[b]) return false;
  if (!eq_delaunay_violated(m, a, b, c, d)) return false;
  if (eq_key_exists(m, eq_key(m, c, d))) return false;  // the new diagonal would become an edge of four facets
  const int32_t* t1 = m.tri + (h1 - h1 % 3);
  const int32_t* t2 = m.tri + (h2 - h2 % 3);
  double m1o, m2o, m1n, m2n;
  const d3 n1o = eq_unit_normal(m, t1[0], t1[1], t1[2], m1o), n2o = eq_unit_normal(m, t2[0], t2[1], t2[2], m2o);
  const d3 n1n = eq_unit_normal(m, a, d, c, m1n), n2n = eq_unit_normal(m, b, c, d, m2n);
  return m1o > 0 && m2o > 0 && m1n > 1e-300 && m2n > 1e-300 && eq_dot(n1n, n1o) >= -0.5 && eq_dot(n2n, n2o) >= -0.5;
}

// Candidates of one sweep, indexed in ascending edge key (= priority: lower index is scanned first).
struct EqCands {
  int32_t n;
  const int32_t* h1;         // half-edge a -> b (in f1) of each candidate
  const int32_t* h2;         // half-edge b -> a (in f2)
  const int32_t* slot_cand;  // 3 nf: candidate owning half-edge h, -1 = none
  const uint64_t* nkey;      // new-diagonal keys sorted stably (candidates with one new diagonal are adjacent)
  const int32_t* nkey_cand;  // candidate of each sorted new key
  const int32_t* nkey_pos;   // candidate -> its position in nkey
};

// One selection round for candidate i, reading the states of the previous round.  An undecided candidate is
// rejected when an earlier conflicting candidate is selected and selected when every earlier conflicting one is
// rejected; decided candidates keep their state.  By induction on i this is the sequential scan's answer, and the
// lowest undecided candidate is always decided.
MS_HD uint8_t eq_round(const EqCands& s, const uint8_t* state, int i) {
  if (state[i] != EQ_UNDECIDED) return state[i];
  bool all_rejected = true;
  const int32_t hs[2] = {s.h1[i], s.h2[i]};
  for (int q = 0; q < 2; ++q) {  // candidates sharing f1 or f2 own one of its other two half-edges
    const int32_t base = hs[q] - hs[q] % 3;
    for (int k = 0; k < 3; ++k) {
      const int32_t h = base + k;
      if (h == hs[0] || h == hs[1]) continue;
      const int32_t j = s.slot_cand[h];
      if (j < 0 || j >= i) continue;
      if (state[j] == EQ_SELECTED) return EQ_REJECTED;
      if (state[j] != EQ_REJECTED) all_rejected = false;
    }
  }
  const int32_t p = s.nkey_pos[i];
  for (int32_t r = p - 1; r >= 0 && s.nkey[r] == s.nkey[p]; --r) {  // earlier claims of the same new diagonal
    const uint8_t st = state[s.nkey_cand[r]];
    if (st == EQ_SELECTED) return EQ_REJECTED;
    if (st != EQ_REJECTED) all_rejected = false;
  }
  return all_rejected ? EQ_SELECTED : EQ_UNDECIDED;
}

// The flip of a selected candidate: reads and writes only its own two rows (selected candidates share none).
MS_HD void eq_apply(int32_t* tri, int32_t h1, int32_t h2) {
  const EqMesh m{0, 0, tri, nullptr, nullptr, nullptr, nullptr, nullptr};
  const int a = eq_tail(m, h1), b = eq_head(m, h1), c = eq_apex(m, h1), d = eq_apex(m, h2);
  int32_t* r1 = tri + (h1 - h1 % 3);
  int32_t* r2 = tri + (h2 - h2 % 3);
  r1[0] = a; r1[1] = d; r1[2] = c;
  r2[0] = b; r2[1] = c; r2[2] = d;
}

}  // namespace ms
