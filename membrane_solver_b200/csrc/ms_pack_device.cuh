// Patch packing on the device: the host packer ms::pack_patches (ms_pack.cpp) restated so that one warp packs one
// chunk of 32 * max_owned vertex rows, shared by the device kernels and the test-only host emulator.  The output is
// byte for byte the host packer's (headers, halo ids, records, slot facets, statistics and return codes).
//
// What the restatement rests on (each checked against ms_pack.cpp):
//   - incidence: the host's vertex -> facet lists are the corner CSR (corner ids 3 f + k ordered by vertex, then by
//     corner id) with the facets that name a vertex twice skipped;
//   - chunks are packed independently and concatenated in chunk order; the first failing chunk decides the code;
//   - collect: facet f enters a patch at its smallest owned corner, so the list is ordered by (that corner, f), and
//     "no owned corner below v" replaces the host's facet stamps; halo slots are numbered in order of first
//     appearance over that list (corners k = 0, 1, 2), which a small hash table of the patch keeps;
//   - find_slot is the lexicographic argmin of (cost, round fill, r, hw, rot) over the feasible candidates: the
//     host's early exits only prune candidates that cannot win, so the lanes evaluate candidates and reduce;
//   - insertion, the repair sweeps, lane numbering, dropping empty rounds and the emission keep the host's order
//     (lane 0, or lanes over independent items);
//   - the trimming arithmetic is the host's IEEE double expressions, never contracted.
// The warp policy W provides lane(), size(), sync(), ballot(p), lt_mask(), bcast(x) (lane 0's x) and min64(x); the
// emulator's policy is a single lane, so every lane loop runs serially and the reductions are the identity.
#pragma once

#include "ms_math.cuh"
#include "ms_pack.h"

namespace ms {

constexpr uint64_t kPkNone = ~uint64_t(0);  // find_slot: no feasible candidate
constexpr int32_t kPkInternal = -101;       // a scratch or staging bound did not hold (cannot happen)

#ifdef __CUDA_ARCH__
MS_HD double pk_mul(double a, double b) { return __dmul_rn(a, b); }
MS_HD double pk_div(double a, double b) { return __ddiv_rn(a, b); }
#else
MS_HD double pk_mul(double a, double b) { return a * b; }
MS_HD double pk_div(double a, double b) { return a / b; }
#endif

struct PkMesh {
  int32_t nv, nf, n_owned;
  const int32_t* tri;
  const uint8_t* body;     // nf bytes or nullptr
  const int32_t* csr_ptr;  // corner CSR: nv + 1 offsets
  const int32_t* csr_idx;  // corner ids 3 f + k
  PackParams prm;
};

// One chunk: its scratch and staging (set by the caller) and what it produced (set by pk_chunk).  The staging bounds
// are exact: a chunk of len rows has at most len patches, and its patches list at most D facets, D = the corners
// at its rows, with at most 2 D halo entries (a listed facet has an owned corner).
struct PkChunk {
  int64_t scratch;    // first int32 of the chunk's scratch
  int32_t fac_cap;    // facets of one patch, at most
  int32_t round_cap;  // rounds of one patch, at most
  int64_t hdr_off, halo_off, ent_off;  // staging offsets
  int64_t hdr_cap, halo_cap, ent_cap;
  int32_t rc, n_patches;
  int64_t n_halo, n_slots;
  int32_t max_owned, max_local, max_rounds, max_slots;
  int64_t n_round_slots, n_listed, n_lane_conflicts;
};

// Staging of all chunks: headers with chunk-relative halo_off / slot_off, halo ids, and one entry per listed facet
// (its record, facet and chunk-relative slot); every other slot is empty (a zero record, facet -1).
struct PkStage {
  PatchHeader* hdr;
  int32_t* halo;
  FacetRec* ent_rec;
  int32_t* ent_fac;
  int64_t* ent_slot;
};

MS_HD int pk_popc(uint32_t x) {
#ifdef __CUDA_ARCH__
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}

MS_HD int64_t pk_chunk_rows(const PackParams& p) { return int64_t(32) * int64_t(p.max_owned); }
MS_HD int pk_n_hw(int32_t T) { return (T + 15) / 16; }
MS_HD int32_t pk_hash_cap(const PackParams& p) {
  int32_t h = 64;
  while (h < 2 * (p.max_local + 1)) h *= 2;
  return h;
}
MS_HD int32_t pk_words(int32_t round_cap) { return (round_cap + 63) / 64 + 1; }
MS_HD bool pk_listed(const int32_t* t, int32_t nv) {
  return t[0] >= 0 && t[0] < nv && t[1] >= 0 && t[1] < nv && t[2] >= 0 && t[2] < nv && t[0] != t[1] && t[1] != t[2] &&
         t[0] != t[2];
}
MS_HD bool pk_valid(const int32_t* t, int32_t nv) {
  return t[0] >= 0 && t[0] < nv && t[1] >= 0 && t[1] < nv && t[2] >= 0 && t[2] < nv;
}
// corner CSR sort key of corner c: its vertex, or nv for the corners of facets with an index out of range
MS_HD int32_t pk_corner_key(const int32_t* tri, int32_t nv, int64_t c) {
  return pk_valid(tri + 3 * (c / 3), nv) ? tri[c] : nv;
}

// Rounds of one patch of at most fac facets whose owned vertices have at most deg incident corners: the host starts
// with max(ceil(fac / (T fill)), min(7, fac)) rounds and adds one only when every round is full (<= fac / T of them)
// or writes an owned corner of the facet (<= 3 deg of them).
MS_HD int32_t pk_round_cap(const PackParams& p, int64_t fac, int64_t deg) {
  const int64_t T = p.threads;
  int64_t a = (fac * 100 + T * p.fill_pct - 1) / (T * p.fill_pct);
  if (a < 7) a = 7;
  const int64_t b = fac / T + 3 * deg + 1;
  return int32_t((a > b ? a : b) + 1);
}

// The scratch of one chunk, carved from int32 words.
struct PkScratch {
  int32_t *facets, *floc, *place, *halo, *hkey, *hval, *round_fill, *hw_fill, *members, *remap;
  uint64_t* used;
  uint8_t* cnt;
  int32_t words, hcap;
};

MS_HD int64_t pk_scratch_words(const PackParams& p, int32_t fac_cap, int32_t round_cap) {
  const int64_t F = fac_cap, R = round_cap, nhw = pk_n_hw(p.threads);
  int64_t w = 8 * F + (p.max_local + 1) + 2 * int64_t(pk_hash_cap(p));
  w += (w & 1);
  w += 2 * int64_t(p.max_owned) * pk_words(round_cap);
  w += R * (2 + nhw * (1 + 16 + 12));
  return w + 2;
}

MS_HD PkScratch pk_scratch_at(int32_t* base, const PackParams& p, int32_t fac_cap, int32_t round_cap) {
  PkScratch s;
  const int64_t F = fac_cap, R = round_cap, nhw = pk_n_hw(p.threads);
  s.hcap = pk_hash_cap(p);
  s.words = pk_words(round_cap);
  int32_t* q = base;
  s.facets = q; q += F;
  s.floc = q; q += 3 * F;
  s.place = q; q += 4 * F;  // (round, half-warp, rotation, lane)
  s.halo = q; q += p.max_local + 1;
  s.hkey = q; q += s.hcap;
  s.hval = q; q += s.hcap;
  q += (q - base) & 1;
  s.used = reinterpret_cast<uint64_t*>(q); q += 2 * int64_t(p.max_owned) * s.words;
  s.round_fill = q; q += R;
  s.remap = q; q += R;
  s.hw_fill = q; q += R * nhw;
  s.members = q; q += R * nhw * 16;
  s.cnt = reinterpret_cast<uint8_t*>(q);
  return s;
}

MS_HD uint32_t pk_hash(int32_t u) { return uint32_t(u) * 2654435761u; }

// local halo index of vertex u in the last collect
MS_HD int32_t pk_halo_find(const PkScratch& s, int32_t u) {
  for (uint32_t h = pk_hash(u) & uint32_t(s.hcap - 1);; h = (h + 1) & uint32_t(s.hcap - 1))
    if (s.hkey[h] == u) return s.hval[h];
}

// Facets and halo of the patch owning [v_lo, v_lo + n): returns the local vertex count, or max_local + 1 once it is
// known to exceed max_local.  *nfac / *nhalo receive the list lengths.
template <class W>
MS_HD int64_t pk_collect(W& w, const PkMesh& m, const PkScratch& s, int32_t v_lo, int32_t n, int32_t* nfac_out,
                         int32_t* nhalo_out) {
  const int32_t v_hi = v_lo + n;
  for (int32_t i = w.lane(); i < s.hcap; i += w.size()) s.hkey[i] = -1;
  w.sync();
  const int64_t e0 = m.csr_ptr[v_lo], e1 = m.csr_ptr[v_hi];
  int32_t nfac = 0, nhalo = 0;
  const int32_t halo_max = m.prm.max_local - n;  // more than this many halo vertices: too large
  bool over = halo_max < 0;
  for (int64_t base = e0; base < e1; base += w.size()) {
    const int64_t e = base + w.lane();
    bool take = false;
    int32_t f = 0, u[3] = {0, 0, 0};
    if (e < e1) {
      const int32_t c = m.csr_idx[e];
      f = c / 3;
      const int32_t* t = m.tri + 3 * int64_t(f);
      u[0] = t[0]; u[1] = t[1]; u[2] = t[2];
      const int32_t v = u[c - 3 * f];
      take = pk_listed(u, m.nv);
      for (int k = 0; k < 3; ++k) take = take && !(u[k] >= v_lo && u[k] < v);
    }
    const uint32_t mask = w.ballot(take);
    if (take) s.facets[nfac + pk_popc(mask & w.lt_mask())] = f;
    w.sync();
    // halo vertices in order of first appearance: lane 0 walks the facets taken in this batch
    if (!over && w.lane() == 0) {
      for (int32_t j = nfac; j < nfac + int32_t(pk_popc(mask)) && !over; ++j) {
        const int32_t* t = m.tri + 3 * int64_t(s.facets[j]);
        for (int k = 0; k < 3 && !over; ++k) {
          const int32_t x = t[k];
          if (x >= v_lo && x < v_hi) continue;
          uint32_t h = pk_hash(x) & uint32_t(s.hcap - 1);
          while (s.hkey[h] >= 0 && s.hkey[h] != x) h = (h + 1) & uint32_t(s.hcap - 1);
          if (s.hkey[h] == x) continue;
          if (nhalo == halo_max) { over = true; break; }
          s.hkey[h] = x;
          s.hval[h] = nhalo;
          s.halo[nhalo++] = x;
        }
      }
    }
    nfac += int32_t(pk_popc(mask));
    over = w.bcast(int(over)) != 0;
    w.sync();
  }
  nhalo = w.bcast(nhalo);
  *nfac_out = nfac;
  *nhalo_out = nhalo;
  return over ? int64_t(m.prm.max_local) + 1 : int64_t(n) + nhalo;
}

// --- the per-patch placement state (see pack_range in ms_pack.cpp) ---
struct PkPatch {
  PkScratch s;
  int32_t n, nfac, n_hw, T, words;
};

MS_HD uint8_t* pk_cnt(const PkPatch& p, int32_t r, int hw) { return p.s.cnt + (size_t(r) * p.n_hw + hw) * 48; }
MS_HD int32_t* pk_members(const PkPatch& p, int32_t r, int hw) { return p.s.members + (size_t(r) * p.n_hw + hw) * 16; }

MS_HD bool pk_round_free(const PkPatch& p, int32_t i, int32_t r) {
  for (int k = 0; k < 3; ++k) {
    const int32_t l = p.s.floc[3 * i + k];
    if (l < p.n && ((p.s.used[size_t(l) * p.words + size_t(r >> 6)] >> (r & 63)) & 1u)) return false;
  }
  return true;
}

MS_HD void pk_mark_round(const PkPatch& p, int32_t i, int32_t r, bool on) {
  for (int k = 0; k < 3; ++k) {
    const int32_t l = p.s.floc[3 * i + k];
    if (l >= p.n) continue;
    uint64_t& x = p.s.used[size_t(l) * p.words + size_t(r >> 6)];
    if (on) x |= uint64_t(1) << (r & 63); else x &= ~(uint64_t(1) << (r & 63));
  }
}

MS_HD int pk_cost_at(const PkPatch& p, int32_t i, int32_t r, int hw, int rot) {
  const uint8_t* c = pk_cnt(p, r, hw);
  int cost = 0;
  for (int k = 0; k < 3; ++k) cost += c[k * 16 + (p.s.floc[3 * i + (k + rot) % 3] & 15)] ? 1 : 0;
  return cost;
}

MS_HD void pk_insert(const PkPatch& p, int32_t i, int32_t r, int hw, int rot) {
  uint8_t* c = pk_cnt(p, r, hw);
  for (int k = 0; k < 3; ++k) ++c[k * 16 + (p.s.floc[3 * i + (k + rot) % 3] & 15)];
  int32_t* mm = pk_members(p, r, hw);
  for (int l = 0; l < 16; ++l)
    if (mm[l] < 0) { mm[l] = i; break; }
  ++p.s.hw_fill[size_t(r) * p.n_hw + hw];
  ++p.s.round_fill[r];
  p.s.place[4 * i] = r; p.s.place[4 * i + 1] = hw; p.s.place[4 * i + 2] = rot;
  pk_mark_round(p, i, r, true);
}

MS_HD void pk_remove(const PkPatch& p, int32_t i) {
  const int32_t r = p.s.place[4 * i], hw = p.s.place[4 * i + 1], rot = p.s.place[4 * i + 2];
  uint8_t* c = pk_cnt(p, r, hw);
  for (int k = 0; k < 3; ++k) --c[k * 16 + (p.s.floc[3 * i + (k + rot) % 3] & 15)];
  int32_t* mm = pk_members(p, r, hw);
  for (int l = 0; l < 16; ++l)
    if (mm[l] == i) { mm[l] = -1; break; }
  --p.s.hw_fill[size_t(r) * p.n_hw + hw];
  --p.s.round_fill[r];
  pk_mark_round(p, i, r, false);
}

MS_HD bool pk_is_bad(const PkPatch& p, int32_t i) {
  const int32_t r = p.s.place[4 * i], hw = p.s.place[4 * i + 1], rot = p.s.place[4 * i + 2];
  const uint8_t* c = pk_cnt(p, r, hw);
  for (int k = 0; k < 3; ++k)
    if (c[k * 16 + (p.s.floc[3 * i + (k + rot) % 3] & 15)] > 1) return true;
  return false;
}

// Candidate c = (r * n_hw + hw) * 3 + rot for facet i: key (cost, fill, c), or kPkNone when infeasible.
MS_HD uint64_t pk_candidate(const PkPatch& p, int32_t i, int64_t c) {
  const int rot = int(c % 3);
  const int hw = int((c / 3) % p.n_hw);
  const int32_t r = int32_t(c / (3 * p.n_hw));
  const int32_t fill = p.s.round_fill[r];
  if (fill >= p.T) return kPkNone;
  const int cap = 16 < p.T - hw * 16 ? 16 : p.T - hw * 16;
  if (p.s.hw_fill[size_t(r) * p.n_hw + hw] >= cap) return kPkNone;
  if (!pk_round_free(p, i, r)) return kPkNone;
  return (uint64_t(pk_cost_at(p, i, r, hw, rot)) << 60) | (uint64_t(fill) << 48) | uint64_t(c);
}

// The host's find_slot: the smallest key over all candidates of facet i (every lane returns it).
template <class W>
MS_HD uint64_t pk_find_slot(W& w, const PkPatch& p, int32_t i, int32_t n_rounds) {
  const int64_t nc = int64_t(n_rounds) * p.n_hw * 3;
  uint64_t best = kPkNone;
  for (int64_t c = w.lane(); c < nc; c += w.size()) {
    const uint64_t k = pk_candidate(p, i, c);
    if (k < best) best = k;
  }
  return w.min64(best);
}

MS_HD void pk_decode(const PkPatch& p, uint64_t key, int32_t& r, int& hw, int& rot) {
  const int64_t c = int64_t(key & ((uint64_t(1) << 48) - 1));
  rot = int(c % 3);
  hw = int((c / 3) % p.n_hw);
  r = int32_t(c / (3 * p.n_hw));
}

// The host's swap repair of facet i (already removed from `old`): exchange with a facet of another half-warp of the
// same round.  Returns whether it swapped; otherwise i is back at its old place.
MS_HD bool pk_swap_repair(const PkPatch& p, int32_t i, int32_t old_r, int old_hw, int old_rot) {
  for (int hw2 = 0; hw2 < p.n_hw; ++hw2) {
    if (hw2 == old_hw) continue;
    for (int l = 0; l < 16; ++l) {
      const int32_t j = pk_members(p, old_r, hw2)[l];
      if (j < 0) continue;
      const int32_t pr = p.s.place[4 * j], phw = p.s.place[4 * j + 1], prot = p.s.place[4 * j + 2];
      pk_remove(p, j);
      int rot_i = -1, rot_j = -1;
      for (int q = 0; q < 3 && rot_i < 0; ++q)
        if (pk_cost_at(p, i, old_r, hw2, q) == 0) rot_i = q;
      for (int q = 0; q < 3 && rot_i >= 0 && rot_j < 0; ++q)
        if (pk_cost_at(p, j, old_r, old_hw, q) == 0) rot_j = q;
      if (rot_i >= 0 && rot_j >= 0) {
        pk_insert(p, i, old_r, hw2, rot_i);
        pk_insert(p, j, old_r, old_hw, rot_j);
        return true;
      }
      pk_insert(p, j, pr, phw, prot);
    }
  }
  pk_insert(p, i, old_r, old_hw, old_rot);
  return false;
}

// empty rounds [r0, r1)
template <class W>
MS_HD void pk_clear_rounds(W& w, const PkPatch& p, int32_t r0, int32_t r1) {
  for (int64_t x = r0 + w.lane(); x < r1; x += w.size()) p.s.round_fill[x] = 0;
  for (int64_t x = int64_t(r0) * p.n_hw + w.lane(); x < int64_t(r1) * p.n_hw; x += w.size()) p.s.hw_fill[x] = 0;
  for (int64_t x = int64_t(r0) * p.n_hw * 16 + w.lane(); x < int64_t(r1) * p.n_hw * 16; x += w.size()) p.s.members[x] = -1;
  for (int64_t x = int64_t(r0) * p.n_hw * 48 + w.lane(); x < int64_t(r1) * p.n_hw * 48; x += w.size()) p.s.cnt[x] = 0;
}

// Packs the vertex rows [v_begin, v_end) of chunk ck (pack_range of ms_pack.cpp).  Every lane of w runs it.
template <class W>
MS_HD void pk_chunk(W& w, const PkMesh& m, int32_t* scratch_base, const PkStage& st, PkChunk& ck, int32_t v_begin,
                    int32_t v_end) {
  const PackParams& prm = m.prm;
  const int32_t T = prm.threads;
  PkPatch p;
  p.s = pk_scratch_at(scratch_base + ck.scratch, prm, ck.fac_cap, ck.round_cap);
  p.T = T;
  p.n_hw = pk_n_hw(T);
  p.words = p.s.words;
  const int32_t R = ck.round_cap;
  int32_t n_patches = 0, max_owned = 0, max_local = 0, max_rounds = 0, max_slots = 0;
  int64_t n_halo_total = 0, n_slots_total = 0, n_round_slots = 0, n_listed = 0, n_conf = 0;
  int32_t rc = 0;
  int32_t forced_n = 0;
  for (int32_t v_lo = v_begin; v_lo < v_end;) {
    int32_t n = forced_n > 0 ? forced_n : prm.max_owned;
    if (n > v_end - v_lo) n = v_end - v_lo;
    int32_t nfac = 0, nhalo = 0;
    int64_t n_local = pk_collect(w, m, p.s, v_lo, n, &nfac, &nhalo);
    while (n_local > prm.max_local && n > 1) {
      n = n / 2 > 1 ? n / 2 : 1;
      n_local = pk_collect(w, m, p.s, v_lo, n, &nfac, &nhalo);
    }
    if (n_local > prm.max_local) { rc = -2; break; }
    if (forced_n == 0 && n == prm.max_owned && n > 64) {
      const double per_round = pk_div(pk_mul(double(T), double(prm.fill_pct)), 100.0);
      const int64_t whole = int64_t(pk_div(double(nfac), per_round));
      const int64_t target = int64_t(pk_mul(double(whole), per_round));
      for (int it = 0; it < 4 && whole >= 4 && int64_t(nfac) > target; ++it) {
        const int32_t t = int32_t(pk_div(pk_mul(double(n), double(target)), double(nfac))) - (it > 0 ? 2 : 0);
        n = t > 64 ? t : 64;
        n_local = pk_collect(w, m, p.s, v_lo, n, &nfac, &nhalo);
      }
    }
    if (nfac > ck.fac_cap) { rc = kPkInternal; break; }
    p.n = n;
    p.nfac = nfac;
    const int32_t v_hi = v_lo + n;
    // --- schedule the facets into rounds and lanes ---
    const int64_t tf = int64_t(T) * prm.fill_pct;
    int32_t n_rounds = int32_t((int64_t(nfac) * 100 + tf - 1) / tf);
    if (n_rounds < (nfac < 7 ? nfac : 7)) n_rounds = nfac < 7 ? nfac : 7;
    if (n_rounds > R) { rc = kPkInternal; break; }
    for (int64_t x = w.lane(); x < int64_t(n) * p.words; x += w.size()) p.s.used[x] = 0;
    pk_clear_rounds(w, p, 0, n_rounds);
    for (int32_t i = w.lane(); i < nfac; i += w.size()) {
      const int32_t* t = m.tri + 3 * int64_t(p.s.facets[i]);
      for (int k = 0; k < 3; ++k) {
        const int32_t u = t[k];
        p.s.floc[3 * i + k] = (u >= v_lo && u < v_hi) ? u - v_lo : n + pk_halo_find(p.s, u);
      }
    }
    w.sync();
    bool internal = false;
    for (int32_t i = 0; i < nfac; ++i) {
      uint64_t key = pk_find_slot(w, p, i, n_rounds);
      if (key == kPkNone) {  // grow a round: its arrays are clear already
        if (n_rounds == R) { internal = true; break; }
        pk_clear_rounds(w, p, n_rounds, n_rounds + 1);
        w.sync();
        ++n_rounds;
        key = pk_find_slot(w, p, i, n_rounds);
      }
      w.sync();
      if (w.lane() == 0) {
        int32_t r; int hw, rot;
        pk_decode(p, key, r, hw, rot);
        pk_insert(p, i, r, hw, rot);
      }
      w.sync();
    }
    if (internal) { rc = kPkInternal; break; }
    // repair: relocate facets that still clash
    for (int sweep = 0; sweep < prm.repair_sweeps; ++sweep) {
      int64_t fixed = 0;
      for (int32_t i = 0; i < nfac; ++i) {
        if (!pk_is_bad(p, i)) continue;
        const int32_t old_r = p.s.place[4 * i], old_hw = p.s.place[4 * i + 1], old_rot = p.s.place[4 * i + 2];
        w.sync();
        if (w.lane() == 0) pk_remove(p, i);
        w.sync();
        const uint64_t key = pk_find_slot(w, p, i, n_rounds);
        w.sync();
        bool ok = false;
        if (w.lane() == 0) {
          if (key != kPkNone && (key >> 60) == 0) {
            int32_t r; int hw, rot;
            pk_decode(p, key, r, hw, rot);
            pk_insert(p, i, r, hw, rot);
            ok = true;
          } else {
            ok = pk_swap_repair(p, i, old_r, old_hw, old_rot);
          }
        }
        fixed += w.bcast(int(ok));
        w.sync();
      }
      if (fixed == 0) break;
    }
    // lanes: position inside the half-warp's member list
    for (int64_t g = w.lane(); g < int64_t(n_rounds) * p.n_hw; g += w.size()) {
      const int32_t* mm = p.s.members + g * 16;
      int lane = 0;
      for (int l = 0; l < 16; ++l)
        if (mm[l] >= 0) p.s.place[4 * mm[l] + 3] = lane++;
    }
    int64_t clashes = 0;
    for (int32_t b = 0; b < nfac; b += w.size()) {
      const int32_t i = b + w.lane();
      clashes += pk_popc(w.ballot(i < nfac && pk_is_bad(p, i)));
    }
    // drop rounds that stayed empty
    int32_t kept = 0;
    if (w.lane() == 0)
      for (int32_t r = 0; r < n_rounds; ++r) p.s.remap[r] = p.s.round_fill[r] > 0 ? kept++ : -1;
    kept = w.bcast(kept);
    w.sync();
    const int64_t n_slots = int64_t(kept) * T;
    if (n_slots > prm.max_slots && n > 1) {  // over the slot capacity: halve
      forced_n = n / 2 > 1 ? n / 2 : 1;
      continue;
    }
    if (n_slots > prm.max_slots) { rc = -3; break; }
    if (n_patches >= ck.hdr_cap || n_halo_total + nhalo > ck.halo_cap || n_listed + nfac > ck.ent_cap) {
      rc = kPkInternal;
      break;
    }
    // --- emit header, halo list and the records ---
    if (w.lane() == 0) {
      PatchHeader h;
      h.v_lo = v_lo;
      h.n_owned = n;
      h.halo_off = int32_t(n_halo_total);
      h.n_halo = nhalo;
      h.slot_off = n_slots_total;
      h.reserved = 0;
      h.n_rounds = kept;
      st.hdr[ck.hdr_off + n_patches] = h;
    }
    for (int32_t j = w.lane(); j < nhalo; j += w.size()) st.halo[ck.halo_off + n_halo_total + j] = p.s.halo[j];
    for (int32_t i = w.lane(); i < nfac; i += w.size()) {
      const int32_t f = p.s.facets[i];
      const int32_t* t = m.tri + 3 * int64_t(f);
      uint16_t flags = REC_VALID;
      if (t[0] >= v_lo && t[0] < v_hi) flags |= REC_PRIMARY;
      if (m.body && m.body[f]) flags |= REC_BODY;
      const int32_t* pl = p.s.place + 4 * i;
      const int rot = pl[2];
      FacetRec rec;
      rec.a = uint16_t(p.s.floc[3 * i + rot % 3]);
      rec.b = uint16_t(p.s.floc[3 * i + (1 + rot) % 3]);
      rec.c = uint16_t(p.s.floc[3 * i + (2 + rot) % 3]);
      rec.flags = flags;
      const int64_t e = ck.ent_off + n_listed + i;
      st.ent_rec[e] = rec;
      st.ent_fac[e] = f;
      st.ent_slot[e] = n_slots_total + int64_t(p.s.remap[pl[0]]) * T + int64_t(pl[1]) * 16 + pl[3];
    }
    w.sync();
    forced_n = 0;
    ++n_patches;
    n_halo_total += nhalo;
    n_slots_total += n_slots;
    n_conf += clashes;
    if (n > max_owned) max_owned = n;
    if (int32_t(n_local) > max_local) max_local = int32_t(n_local);
    if (kept > max_rounds) max_rounds = kept;
    if (int32_t(n_slots) > max_slots) max_slots = int32_t(n_slots);
    n_round_slots += n_slots;
    n_listed += nfac;
    v_lo += n;
  }
  if (w.lane() == 0) {
    ck.rc = rc;
    ck.n_patches = n_patches;
    ck.n_halo = n_halo_total;
    ck.n_slots = n_slots_total;
    ck.max_owned = max_owned;
    ck.max_local = max_local;
    ck.max_rounds = max_rounds;
    ck.max_slots = max_slots;
    ck.n_round_slots = n_round_slots;
    ck.n_listed = n_listed;
    ck.n_lane_conflicts = n_conf;
  }
}

// Per-chunk bounds from the corner CSR, one vertex row v of chunk `chunk` [c0, c1): facets of a patch starting at v
// (at most max_owned rows) and corners at v.
MS_HD void pk_row_bounds(const PackParams& p, const int32_t* csr_ptr, int32_t v, int32_t c1, int64_t* window,
                         int64_t* deg) {
  const int32_t hi = int64_t(v) + p.max_owned < c1 ? v + p.max_owned : c1;
  *window = int64_t(csr_ptr[hi]) - csr_ptr[v];
  *deg = int64_t(csr_ptr[v + 1]) - csr_ptr[v];
}

// Scratch and staging of every chunk from its bounds (3 per chunk: the largest facet window of a patch, the largest
// vertex degree and the corners at its rows); returns the int32 scratch words and staging entries of all chunks.
struct PkPlan {
  int64_t scratch_words, hdr, halo, ent;
};

inline PkPlan pk_plan(const PackParams& p, int32_t n_owned, const int64_t* bounds, PkChunk* ck, int64_t n_chunks) {
  PkPlan t{0, 0, 0, 0};
  const int64_t chunk = pk_chunk_rows(p);
  for (int64_t c = 0; c < n_chunks; ++c) {
    PkChunk& k = ck[c];
    const int64_t len = (c + 1) * chunk < n_owned ? chunk : n_owned - c * chunk;
    k = PkChunk{};
    k.fac_cap = int32_t(bounds[3 * c] > 1 ? bounds[3 * c] : 1);
    k.round_cap = pk_round_cap(p, k.fac_cap, bounds[3 * c + 1]);
    k.scratch = t.scratch_words;
    const int64_t words = pk_scratch_words(p, k.fac_cap, k.round_cap);
    t.scratch_words += words + (words & 1);  // every chunk starts 8-byte aligned
    k.hdr_off = t.hdr;
    k.hdr_cap = len;
    t.hdr += len;
    k.halo_off = t.halo;
    k.halo_cap = 2 * bounds[3 * c + 2];
    t.halo += k.halo_cap;
    k.ent_off = t.ent;
    k.ent_cap = bounds[3 * c + 2];
    t.ent += k.ent_cap;
  }
  return t;
}

// The exact bank statistic of one (round, half-warp) of records rr with `cap` lanes: adds its gather groups and
// extra wavefronts (see pack_patches).
MS_HD void pk_hw_excess(const FacetRec* rr, int cap, int64_t* groups, int64_t* excess) {
  bool any = false;
  for (int l = 0; l < cap; ++l) any |= (rr[l].flags & REC_VALID) != 0;
  if (!any) return;
  for (int k = 0; k < 3; ++k) {
    int32_t seen[16][16];
    int cnt[16];
    for (int q = 0; q < 16; ++q) cnt[q] = 0;
    for (int l = 0; l < cap; ++l) {
      if (!(rr[l].flags & REC_VALID)) continue;
      const int32_t idx = k == 0 ? rr[l].a : (k == 1 ? rr[l].b : rr[l].c);
      const int res = idx & 15;
      bool dup = false;
      for (int j = 0; j < cnt[res]; ++j) dup |= seen[res][j] == idx;
      if (!dup) seen[res][cnt[res]++] = idx;
    }
    int mx = 1;
    for (int q = 0; q < 16; ++q) mx = mx > cnt[q] ? mx : cnt[q];
    *groups += 1;
    *excess += mx - 1;
  }
}

}  // namespace ms
