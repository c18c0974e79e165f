// TEST-ONLY host emulator of the vertex-averaging kernel.
//
// Runs the SAME per-vertex body (ms_vertex_average.cuh) over the SAME corner CSR (ms_pack.cpp) as
// k_vertex_average, serially on the host, so that the no-GPU test tier checks the device code against the host
// twin and the reference's golden vectors.  Nothing under membrane_solver_b200/ loads it.
#include <cstring>
#include <vector>

#include "../../membrane_solver_b200/csrc/ms_pack.h"
#include "../../membrane_solver_b200/csrc/ms_vertex_average.cuh"

using namespace ms;

extern "C" {

// `rounds` Jacobi rounds of the per-vertex body.  fixed / group may be null.  pos_inout (nv,3) is replaced by the
// result.  Returns -1 on rounds < 0.
int emul_vertex_average(int32_t nv, int32_t nf, const int32_t* tri, const uint8_t* fixed, const int32_t* group,
                        int32_t rounds, double* pos_inout) {
  if (rounds < 0) return -1;
  std::vector<int32_t> csr_ptr, csr_idx;
  build_corner_csr(nv, nf, tri, csr_ptr, csr_idx);
  std::vector<double> cur(pos_inout, pos_inout + 3 * size_t(nv)), next(3 * size_t(nv));
  VaMesh m{nv, tri, nullptr, csr_ptr.data(), csr_idx.data(), group, fixed};
  for (int32_t r = 0; r < rounds; ++r) {
    m.pos = cur.data();
    for (int v = 0; v < nv; ++v) {
      const d3 x = va_vertex(m, v);
      next[3 * size_t(v)] = x.x; next[3 * size_t(v) + 1] = x.y; next[3 * size_t(v) + 2] = x.z;
    }
    cur.swap(next);
  }
  std::memcpy(pos_inout, cur.data(), cur.size() * sizeof(double));
  return 0;
}

}  // extern "C"
