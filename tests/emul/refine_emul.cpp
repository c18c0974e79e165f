// TEST-ONLY host emulator of the refinement kernels.
//
// Runs the SAME per-vertex, per-midpoint and per-facet bodies (ms_refine.cuh) as ms_ctx_refine, serially on the
// host, so that the no-GPU test tier checks the device code against the host twin geometry/refine.py.  The key sort
// is std::stable_sort, which orders like the device's stable radix sort; the edge numbering is a running count of
// run heads, as the device's inclusive scan.  Nothing under membrane_solver_b200/ loads it.
#include <algorithm>
#include <numeric>
#include <vector>

#include "../../membrane_solver_b200/csrc/ms_refine.cuh"

using namespace ms;

extern "C" {

// `levels` >= 1 levels of refinement of (nv, nf, tri, pos); fixed / boundary (nv) and key_id (nv: vertex id -> the
// caller's id, as the device's internal-to-caller permutation) may be null.  The result is in the caller's numbering:
// *nv_out rows of pos_out / fixed_out / boundary_out and 4^levels nf rows of tri_out; the caller sizes them (an upper
// bound of the vertex count is nv + 3 nf (4^levels - 1) / 3).  Returns -1 on bad arguments.
int emul_refine(int32_t nv, int32_t nf, const int32_t* tri, const double* pos, const uint8_t* fixed,
                const uint8_t* boundary, const int32_t* key_id, int32_t levels, double* pos_out, int32_t* tri_out,
                uint8_t* fixed_out, uint8_t* boundary_out, int32_t* nv_out) {
  if (nv < 0 || nf < 0 || levels < 1) return -1;
  for (int64_t h = 0; h < 3 * int64_t(nf); ++h)
    if (tri[h] < 0 || tri[h] >= nv) return -1;
  std::vector<double> cpos(pos, pos + 3 * size_t(nv));
  std::vector<int32_t> ctri(tri, tri + 3 * size_t(nf));
  std::vector<uint8_t> cfixed, cbnd;
  if (fixed) cfixed.assign(fixed, fixed + nv);
  if (boundary) cbnd.assign(boundary, boundary + nv);
  const int32_t* kid = key_id;
  for (int32_t l = 0; l < levels; ++l) {
    EqMesh m{nv, nf, ctri.data(), cpos.data(), fixed ? cfixed.data() : nullptr, kid, nullptr, nullptr};
    const size_t nh = 3 * size_t(nf);
    std::vector<uint64_t> key(nh), skey(nh);
    std::vector<int32_t> order(nh), edge(nh), head;
    for (size_t h = 0; h < nh; ++h) key[h] = eq_key(m, eq_tail(m, int64_t(h)), eq_head(m, int64_t(h)));
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return key[size_t(x)] < key[size_t(y)]; });
    for (size_t i = 0; i < nh; ++i) skey[i] = key[size_t(order[i])];
    int32_t ne = 0;
    for (size_t i = 0; i < nh; ++i) {
      if (rf_head(skey.data(), int64_t(i))) {
        head.push_back(int32_t(i));
        ++ne;
      }
      edge[size_t(order[i])] = ne - 1;
    }
    head.push_back(int32_t(nh));
    m.keys = skey.data();
    m.order = order.data();
    const RfMesh r{m, boundary ? cbnd.data() : nullptr, head.data(), edge.data(), ne};
    const size_t nv2 = size_t(nv) + size_t(ne);
    std::vector<double> npos(3 * nv2);
    std::vector<int32_t> ntri(12 * size_t(nf));
    std::vector<uint8_t> nfixed(fixed ? nv2 : 0), nbnd(boundary ? nv2 : 0);
    const RfOut o{npos.data(), nfixed.data(), nbnd.data(), ntri.data()};
    for (int64_t i = 0; i < int64_t(nv2); ++i) {
      if (i < nv) rf_vertex(r, o, int32_t(i));
      else rf_midpoint(r, o, int32_t(i - nv));
    }
    for (int32_t f = 0; f < nf; ++f) rf_children(r, o, f);
    cpos.swap(npos);
    ctri.swap(ntri);
    cfixed.swap(nfixed);
    cbnd.swap(nbnd);
    nv = int32_t(nv2);
    nf *= 4;
    kid = nullptr;  // later levels are in the caller's numbering already
  }
  std::copy(cpos.begin(), cpos.end(), pos_out);
  std::copy(ctri.begin(), ctri.end(), tri_out);
  if (fixed) std::copy(cfixed.begin(), cfixed.end(), fixed_out);
  if (boundary) std::copy(cbnd.begin(), cbnd.end(), boundary_out);
  *nv_out = nv;
  return 0;
}

}  // extern "C"
