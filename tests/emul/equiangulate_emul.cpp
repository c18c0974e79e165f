// TEST-ONLY host emulator of the equiangulation kernels.
//
// Runs the SAME candidate predicate and the SAME round-based selection (ms_equiangulate.cuh) as the device sweep,
// serially on the host, so that the no-GPU test tier checks the device code against the host twin
// geometry/equiangulate.py.  The sorts are std::stable_sort, which orders like the device's stable radix sort.
// Nothing under membrane_solver_b200/ loads it.
#include <algorithm>
#include <numeric>
#include <vector>

#include "../../membrane_solver_b200/csrc/ms_equiangulate.cuh"

using namespace ms;

extern "C" {

// Sweeps over tri_inout (nf,3) until one makes no flip or max_iterations have run.  fixed (nv) and key_id (nv:
// vertex id -> the id its keys use, as the device's internal-to-caller permutation) may be null.  rounds_out
// (capacity max_iterations) receives the selection rounds of every sweep run.  Returns -1 on bad arguments.
int emul_equiangulate(int32_t nv, int32_t nf, int32_t* tri_inout, const double* pos, const uint8_t* fixed,
                      const int32_t* key_id, int32_t max_iterations, int64_t* n_flips, int32_t* n_sweeps,
                      int32_t* rounds_out) {
  if (nv < 0 || nf < 0 || max_iterations < 0) return -1;
  for (int64_t h = 0; h < 3 * int64_t(nf); ++h)
    if (tri_inout[h] < 0 || tri_inout[h] >= nv) return -1;
  const int64_t nh = 3 * int64_t(nf);
  EqMesh m{nv, nf, tri_inout, pos, fixed, key_id, nullptr, nullptr};
  const size_t n3 = static_cast<size_t>(nh);
  std::vector<uint64_t> key(n3), skey(n3);
  std::vector<int32_t> order(n3), slot_cand(n3);
  *n_flips = 0;
  *n_sweeps = 0;
  for (int32_t sweep = 0; sweep < max_iterations; ++sweep) {
    for (int64_t h = 0; h < nh; ++h) key[size_t(h)] = eq_key(m, eq_tail(m, h), eq_head(m, h));
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return key[size_t(x)] < key[size_t(y)]; });
    for (int64_t i = 0; i < nh; ++i) skey[size_t(i)] = key[size_t(order[size_t(i)])];
    m.keys = skey.data();
    m.order = order.data();
    std::vector<int32_t> h1, h2;
    for (int64_t i = 0; i < nh; ++i) {
      int64_t a = 0, b = 0;
      if (eq_interior(m, i, a, b) && eq_should_flip(m, a, b)) {
        h1.push_back(int32_t(a));
        h2.push_back(int32_t(b));
      }
    }
    const int32_t nc = int32_t(h1.size());
    rounds_out[sweep] = 0;
    if (nc == 0) break;
    std::fill(slot_cand.begin(), slot_cand.end(), -1);
    const size_t ncs = static_cast<size_t>(nc);
    std::vector<uint64_t> nkey(ncs), nkey_sorted(ncs);
    std::vector<int32_t> nkey_cand(ncs), nkey_pos(ncs);
    for (int32_t i = 0; i < nc; ++i) {
      slot_cand[size_t(h1[size_t(i)])] = slot_cand[size_t(h2[size_t(i)])] = i;
      nkey[size_t(i)] = eq_key(m, eq_apex(m, h1[size_t(i)]), eq_apex(m, h2[size_t(i)]));
    }
    std::iota(nkey_cand.begin(), nkey_cand.end(), 0);
    std::stable_sort(nkey_cand.begin(), nkey_cand.end(),
                     [&](int32_t x, int32_t y) { return nkey[size_t(x)] < nkey[size_t(y)]; });
    for (int32_t p = 0; p < nc; ++p) {
      nkey_sorted[size_t(p)] = nkey[size_t(nkey_cand[size_t(p)])];
      nkey_pos[size_t(nkey_cand[size_t(p)])] = p;
    }
    const EqCands s{nc, h1.data(), h2.data(), slot_cand.data(), nkey_sorted.data(), nkey_cand.data(), nkey_pos.data()};
    std::vector<uint8_t> cur(ncs, EQ_UNDECIDED), next(ncs);
    int32_t rounds = 0, undecided = nc;
    while (undecided > 0) {  // Jacobi rounds, as the device runs them
      undecided = 0;
      for (int32_t i = 0; i < nc; ++i) {
        next[size_t(i)] = eq_round(s, cur.data(), i);
        undecided += next[size_t(i)] == EQ_UNDECIDED;
      }
      cur.swap(next);
      ++rounds;
    }
    rounds_out[sweep] = rounds;
    int64_t flips = 0;
    for (int32_t i = 0; i < nc; ++i)
      if (cur[size_t(i)] == EQ_SELECTED) {
        eq_apply(tri_inout, h1[size_t(i)], h2[size_t(i)]);
        ++flips;
      }
    *n_flips += flips;
    ++*n_sweeps;
  }
  return 0;
}

}  // extern "C"
