// TEST-ONLY host emulator of the device patch packer.
//
// Runs the SAME per-chunk, per-row and per-half-warp bodies (ms_pack_device.cuh) as the context's device packing,
// serially on the host: a warp of one lane (every lane loop runs serially, the argmin reduction is the identity),
// the corner sort by std::stable_sort (ordered like the device's stable radix sort).  It also exports the host
// packer ms::pack_patches and ms::build_corner_csr in the same array form, so that the no-GPU test tier compares the
// two byte for byte.  Nothing under membrane_solver_b200/ loads it.
#include <algorithm>
#include <cstring>
#include <numeric>
#include <vector>

#include "../../membrane_solver_b200/csrc/ms_pack_device.cuh"

using namespace ms;

namespace {

struct Serial {
  int lane() const { return 0; }
  int size() const { return 1; }
  void sync() const {}
  uint32_t ballot(bool p) const { return p ? 1u : 0u; }
  uint32_t lt_mask() const { return 0u; }
  int bcast(int x) const { return x; }
  uint64_t min64(uint64_t x) const { return x; }
};

void corner_csr_emul(int32_t nv, int32_t nf, const int32_t* tri, std::vector<int32_t>& ptr, std::vector<int32_t>& idx) {
  const int64_t n = 3 * int64_t(nf);
  std::vector<int32_t> key(size_t(n), 0);
  for (int64_t c = 0; c < n; ++c) key[size_t(c)] = pk_corner_key(tri, nv, c);
  idx.resize(size_t(n));
  std::iota(idx.begin(), idx.end(), 0);
  std::stable_sort(idx.begin(), idx.end(), [&](int32_t a, int32_t b) { return key[size_t(a)] < key[size_t(b)]; });
  ptr.assign(size_t(nv) + 1, 0);
  for (int32_t v = 0; v <= nv; ++v)  // first sorted position with a key >= v
    ptr[size_t(v)] = int32_t(std::lower_bound(idx.begin(), idx.end(), v,
                                              [&](int32_t c, int32_t x) { return key[size_t(c)] < x; }) - idx.begin());
  idx.resize(size_t(ptr[size_t(nv)]));
}

int pack_emul(int32_t nv, int32_t nf, const int32_t* tri, const uint8_t* body, const PackParams& prm, PackedMesh& out,
              int32_t n_owned) {
  if (n_owned < 0 || n_owned > nv) n_owned = nv;
  if (nv < 0 || nf < 0 || (nf > 0 && !tri) || prm.threads <= 0 || prm.max_owned <= 0 || prm.max_local <= 0 ||
      prm.max_local > 65535 || prm.max_slots < prm.threads || prm.fill_pct < 10 || prm.fill_pct > 100)
    return -1;
  out = PackedMesh();
  out.nv = nv;
  out.nf = nf;
  out.params = prm;
  out.n_owned_vertices = n_owned;
  std::vector<int32_t> ptr, idx;
  corner_csr_emul(nv, nf, tri, ptr, idx);
  for (int32_t f = 0; f < nf; ++f) out.n_valid += pk_valid(tri + 3 * size_t(f), nv) ? 1 : 0;
  const int64_t chunk = pk_chunk_rows(prm);
  const int64_t n_chunks = (int64_t(n_owned) + chunk - 1) / chunk;
  std::vector<int64_t> bounds(3 * size_t(n_chunks), 0);
  for (int32_t v = 0; v < n_owned; ++v) {
    const int64_t c = v / chunk;
    const int32_t c1 = int32_t(std::min<int64_t>((c + 1) * chunk, n_owned));
    int64_t window, deg;
    pk_row_bounds(prm, ptr.data(), v, c1, &window, &deg);
    bounds[3 * c] = std::max(bounds[3 * c], window);
    bounds[3 * c + 1] = std::max(bounds[3 * c + 1], deg);
    if (v == c * chunk) bounds[3 * c + 2] = int64_t(ptr[size_t(c1)]) - ptr[size_t(v)];
  }
  std::vector<PkChunk> ck(static_cast<size_t>(n_chunks));
  const PkPlan plan = pk_plan(prm, n_owned, bounds.data(), ck.data(), n_chunks);
  std::vector<int64_t> scratch(size_t(plan.scratch_words / 2) + 1);
  std::vector<PatchHeader> hdr(size_t(plan.hdr));
  std::vector<int32_t> halo(size_t(plan.halo)), ent_fac(size_t(plan.ent));
  std::vector<FacetRec> ent_rec(size_t(plan.ent));
  std::vector<int64_t> ent_slot(size_t(plan.ent));
  const PkStage st{hdr.data(), halo.data(), ent_rec.data(), ent_fac.data(), ent_slot.data()};
  const PkMesh m{nv, nf, n_owned, tri, body, ptr.data(), idx.data(), prm};
  for (int64_t c = 0; c < n_chunks; ++c) {
    Serial w;
    pk_chunk(w, m, reinterpret_cast<int32_t*>(scratch.data()), st, ck[size_t(c)], int32_t(c * chunk),
             int32_t(std::min<int64_t>((c + 1) * chunk, n_owned)));
  }
  for (const PkChunk& k : ck)
    if (k.rc) return k.rc;
  // concatenation in chunk order
  for (const PkChunk& k : ck) {
    const int32_t halo_base = int32_t(out.halo_ids.size());
    const int64_t slot_base = int64_t(out.recs.size());
    for (int32_t j = 0; j < k.n_patches; ++j) {
      PatchHeader h = hdr[size_t(k.hdr_off + j)];
      h.halo_off += halo_base;
      h.slot_off += slot_base;
      out.patches.push_back(h);
    }
    out.halo_ids.insert(out.halo_ids.end(), halo.begin() + k.halo_off, halo.begin() + k.halo_off + k.n_halo);
    FacetRec empty;
    std::memset(&empty, 0, sizeof(empty));
    out.recs.resize(size_t(slot_base + k.n_slots), empty);
    out.slot_facet.resize(size_t(slot_base + k.n_slots), -1);
    for (int64_t e = k.ent_off; e < k.ent_off + k.n_listed; ++e) {
      out.recs[size_t(slot_base + ent_slot[size_t(e)])] = ent_rec[size_t(e)];
      out.slot_facet[size_t(slot_base + ent_slot[size_t(e)])] = ent_fac[size_t(e)];
    }
    out.max_owned = std::max(out.max_owned, k.max_owned);
    out.max_local = std::max(out.max_local, k.max_local);
    out.max_rounds = std::max(out.max_rounds, k.max_rounds);
    out.max_slots = std::max(out.max_slots, k.max_slots);
    out.n_round_slots += k.n_round_slots;
    out.n_listed += k.n_listed;
    out.n_lane_conflicts += k.n_lane_conflicts;
  }
  const int32_t T = prm.threads;
  for (const PatchHeader& h : out.patches)
    for (int32_t r = 0; r < h.n_rounds; ++r)
      for (int hw = 0; hw < pk_n_hw(T); ++hw)
        pk_hw_excess(out.recs.data() + size_t(h.slot_off) + size_t(r) * T + size_t(hw) * 16, std::min(16, T - hw * 16),
                     &out.n_hw_groups, &out.n_hw_excess);
  return 0;
}

PackedMesh g_out[2];  // [0] the emulated device packer, [1] the host packer

}  // namespace

extern "C" {

// Corner CSR of (nv, nf, tri): device (1: the sort of ms_pack_device.cuh) or host (0: ms::build_corner_csr).  ptr
// gets nv + 1 offsets, idx up to 3 nf corner ids.  Returns the number of corners listed.
int64_t emul_corner_csr(int device, int32_t nv, int32_t nf, const int32_t* tri, int32_t* ptr, int32_t* idx) {
  std::vector<int32_t> p, x;
  if (device) corner_csr_emul(nv, nf, tri, p, x);
  else build_corner_csr(nv, nf, tri, p, x);
  std::copy(p.begin(), p.end(), ptr);
  std::copy(x.begin(), x.end(), idx);
  return int64_t(x.size());
}

// Packs with the emulated device packer (device = 1) or the host packer (device = 0); keeps the result for
// emul_pack_fetch.  stats (13): n_patches, n_halo, n_slots, max_owned, max_local, max_rounds, max_slots,
// n_round_slots, n_listed, n_valid, n_lane_conflicts, n_hw_groups, n_hw_excess.  Returns the packer's code.
int emul_pack(int device, int32_t nv, int32_t nf, const int32_t* tri, const uint8_t* body, int32_t threads,
              int32_t max_owned, int32_t max_local, int32_t max_slots, int32_t fill_pct, int32_t repair_sweeps,
              int32_t n_owned, int64_t* stats) {
  PackParams prm;
  prm.threads = threads;
  prm.max_owned = max_owned;
  prm.max_local = max_local;
  prm.max_slots = max_slots;
  prm.fill_pct = fill_pct;
  prm.repair_sweeps = repair_sweeps;
  PackedMesh& o = g_out[device ? 0 : 1];
  o = PackedMesh();
  const int rc = device ? pack_emul(nv, nf, tri, body, prm, o, n_owned) : pack_patches(nv, nf, tri, body, prm, o, n_owned);
  const int64_t s[13] = {int64_t(o.patches.size()), int64_t(o.halo_ids.size()), int64_t(o.recs.size()), o.max_owned,
                         o.max_local, o.max_rounds, o.max_slots, o.n_round_slots, o.n_listed, o.n_valid,
                         o.n_lane_conflicts, o.n_hw_groups, o.n_hw_excess};
  std::copy(s, s + 13, stats);
  return rc;
}

// Copies the last emul_pack result of that packer: headers (32 B each), halo ids, records (8 B each), slot facets.
int emul_pack_fetch(int device, void* headers, int32_t* halo_ids, void* recs, int32_t* slot_facet) {
  const PackedMesh& o = g_out[device ? 0 : 1];
  std::memcpy(headers, o.patches.data(), o.patches.size() * sizeof(PatchHeader));
  std::copy(o.halo_ids.begin(), o.halo_ids.end(), halo_ids);
  std::memcpy(recs, o.recs.data(), o.recs.size() * sizeof(FacetRec));
  std::copy(o.slot_facet.begin(), o.slot_facet.end(), slot_facet);
  return 0;
}

}  // extern "C"
