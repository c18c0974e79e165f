// sm_100a kernels of the energy+gradient path.
//
// Patch kernels (pass A / pass B): PERSISTENT CTAs, one per SM, each walking its share of
// the vertex patches.  A CTA is warp-specialised:
//
//   * one PRODUCER warp stages patch j+1 into the second shared-memory buffer with
//     asynchronous copies (cp.async / LDGSTS) while patch j is being computed: records,
//     halo ids and owned rows first, the halo rows (which need the ids) second.  Global rows
//     are (nv,3) / (nv,5) arrays-of-structures; they land in shared memory as structure of
//     arrays, so every component of a local vertex is one address register + an immediate.
//   * the CONSUMER threads form G groups of `threads` lanes.  The patch's facet records are
//     scheduled in ROUNDS (ms_pack.cpp): within a round no two facets write the same owned
//     vertex and the lanes of a half-warp gather from distinct bank pairs.  Group g takes
//     every G-th round: it computes its facets entirely in registers, then waits for a
//     token (named barrier), adds the corner contributions to the shared accumulators with
//     plain read-modify-writes, and passes the token on.  Accumulation therefore happens in
//     round order -- fixed at pack time, no atomics, run-to-run reproducible -- while the
//     other groups are computing.  After the last round come the patch's EPILOGUE turns
//     (vertex stage + seeds in pass A; gradient rows + KKT dot products in pass B), taken by
//     the groups in the same rotation; accumulators are double buffered so that the next
//     patch's rounds overlap them.
//
// Reference functions replaced: see the header of ms_math.cuh.
#include "ms_kernels.cuh"

#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "ms_bt.cuh"
#include "ms_patch_body.cuh"

namespace ms {

namespace {

static_assert(kSeedStride == kSeedStrideBody, "seed row layout");
static_assert(int(SC_E_BENDING_TILT) == int(PS_E_BENDING_TILT) && int(SC_G_G) == int(PS_G_G) &&
                  int(SC_GC_GC) == int(PS_GC_GC) && kPartialStride == PS_COUNT, "partial layout");

// Deterministic block sum of N values per thread over the first n_threads threads (a multiple
// of 32) synchronised through named barrier `bar`; result valid in thread 0.
template <int N>
__device__ __forceinline__ void block_sum(double (&v)[N], double* red, int n_threads, int bar) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_warps = n_threads >> 5;
#pragma unroll
  for (int k = 0; k < N; ++k) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
  }
  asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(n_threads) : "memory");  // red may still be read
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) red[warp * N + k] = v[k];
  }
  asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(n_threads) : "memory");
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) {
      double x = (lane < n_warps) ? red[lane * N + k] : 0.0;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
      v[k] = x;
    }
  }
}

// Bound of every wait for a peer's flag (clock64 cycles, about 10 s at 1.97 GHz): a rank that left the lock-step
// sequence is reported through the error word instead of hanging the box; generous, because a peer's first launch of a
// kernel includes its lazy load.
constexpr long long kWaitCycles = 20000000000LL;

// ---- asynchronous copies (LDGSTS): global -> shared without a register round trip ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return unsigned(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src));
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
// One contiguous global range -> shared memory (16-byte aligned on both sides, size a multiple of 16) by the copy
// engine; completion is counted in bytes on the mbarrier (mbar_expect_tx).
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// all groups of this thread but the most recent one are complete
__device__ __forceinline__ void cp_async_wait_but_one() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
// the mbarrier receives one arrival (counted in its init value) when every copy this thread has issued so far has
// landed: the issuing warp does not wait for its own copies
__device__ __forceinline__ void cp_async_arrive_on(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- mbarriers (producer <-> consumers) and named barriers (token ring) ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(smem_u32(bar)) : "memory");
}
// arrival that also announces `bytes` of bulk copies to come (they complete the phase together with the arrivals)
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try(unsigned addr, unsigned parity) {
  unsigned ok = 0;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the hardware parks the warp until the phase completes (or the hint expires),
// so a waiting warp issues nothing.  A bare try_wait / nanosleep loop re-issues every few tens of nanoseconds -- ncu
// counted a quarter of all warp instructions of a pass as SYNCS / BRA / NANOSLEEP / YIELD of waiting warps, taken from
// the issue slots of the working ones.
__device__ __forceinline__ bool mbar_try_suspend(unsigned addr, unsigned parity) {
  unsigned ok = 0;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(addr), "r"(parity), "r"(1000000u)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  const unsigned addr = smem_u32(bar);
  while (!mbar_try_suspend(addr, parity)) {
  }
}
// service warps (producer, epilogue): same wait; kept as a separate name for the call sites
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, unsigned parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void named_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// ---------------------------------------------------------------------------
// Shared-memory plan.  Capacities are compile-time so that strides fold into immediates;
// the run-time pack parameters must stay within them (checked by the C-ABI layer).
// ---------------------------------------------------------------------------
constexpr int kACap = kPatchOwnedCap + kDumpRows;  // accumulator stride (owned rows + dump rows)
static_assert(kPatchOwnedCap % 16 == 0 && kPatchLocalCap % 16 == 0 && kPatchSlotCap % 32 == 0, "capacities");
using DevStrides = StaticStrides<kPatchLocalCap, kACap>;

struct PatchHdrS {  // header of the staged patch, written by the producer
  int32_t v_lo, n_owned, n_halo, n_rounds;
  int32_t n_slots, halo_off;
  int64_t slot_off;
};

// Area-weighted unit normal of owned vertex i of a patch, read from GLOBAL memory (the epilogue
// warps never touch the staging buffers).  Same record order as vertex_normal_scan.
__device__ d3 vertex_normal_global(const PatchLaunch& a, const PatchHdrS& hs, int i) {
  const FacetRec* recs = a.recs + hs.slot_off;
  const int32_t* ids = a.halo_ids + hs.halo_off;
  d3 n = make_d3(0, 0, 0);
  for (int k = 0; k < hs.n_slots; ++k) {
    const FacetRec rec = recs[k];
    if (!(rec.flags & REC_VALID)) continue;
    if (rec.a != i && rec.b != i && rec.c != i) continue;
    const int ra = rec.a < hs.n_owned ? hs.v_lo + rec.a : ids[rec.a - hs.n_owned];
    const int rb = rec.b < hs.n_owned ? hs.v_lo + rec.b : ids[rec.b - hs.n_owned];
    const int rc = rec.c < hs.n_owned ? hs.v_lo + rec.c : ids[rec.c - hs.n_owned];
    const d3 v0 = ld3(a.pos, ra), v1 = ld3(a.pos, rb), v2 = ld3(a.pos, rc);
    n = n + cross(v1 - v0, v2 - v0);
  }
  const double m = sqrt(dot(n, n));
  if (m > 1.0e-15) n = (1.0 / m) * n;
  return n;
}

template <int PASS>
struct Plan {
  // positions (and seeds) as rows, two spare rows each: a patch whose first owned row is odd starts its bulk copy
  // one row earlier (16-byte alignment) and its consumers address the rows from base + one row
  static constexpr int kInRows = kPatchLocalCap + 2;
  static constexpr int kInDoubles = (PASS == 0 ? 3 : 3 + kSeedStride) * kInRows;  // pos (+ seeds)
  static constexpr int kAccRows = PASS == 0 ? 5 : 6;
  // byte offsets inside one input buffer
  static constexpr size_t oPos = 0;
  static constexpr size_t oSeed = size_t(3) * kInRows * 8;
  static constexpr size_t oRecs = size_t(kInDoubles) * 8;
  static constexpr size_t oIds = oRecs + size_t(kPatchSlotCap) * sizeof(FacetRec);
  static constexpr size_t oHdr = oIds + size_t(kPatchLocalCap) * 4;
  static constexpr size_t kInBytes = oHdr + 32;
  // whole window: in[2] | acc[2] | mbarriers | reduction scratch | optional arrays
  static constexpr size_t oAcc = 2 * kInBytes;
  static constexpr size_t kAccBytes = size_t(kAccRows) * kACap * 8;
  static constexpr size_t oBars = oAcc + 2 * kAccBytes;
  static constexpr size_t oMail = oBars + 64;   // PatchHdrS[2]: header handed to the epilogue warps
  static constexpr size_t oRed = oMail + 64;
  static constexpr size_t oOpt = oRed + size_t(kMaxConsumerWarps + 1) * PS_COUNT * 8;
};
// optional arrays (after the fixed part): bfl[2][L] i32, t2[2][L] f64, accAb[2][ACap] f64
__host__ __device__ inline size_t opt_bytes(bool boundary, bool tilt, bool tilt_acc) {
  size_t n = 0;
  if (boundary) n += 2 * size_t(kPatchLocalCap) * 4;
  if (tilt) n += 2 * size_t(kPatchLocalCap) * 8;
  if (tilt_acc) n += 2 * size_t(kACap) * 8;
  return n;
}

__device__ __forceinline__ FacetRec load_rec(const FacetRec* p) {
  const uint2 w = *reinterpret_cast<const uint2*>(p);
  FacetRec r;
  r.a = uint16_t(w.x & 0xffffu);
  r.b = uint16_t(w.x >> 16);
  r.c = uint16_t(w.y & 0xffffu);
  r.flags = uint16_t(w.y >> 16);
  return r;
}

// ---------------------------------------------------------------------------
// The persistent patch kernel.  PASS 0 = pass A (curvature accumulation, per-facet scalars,
// vertex stage -> seeds; alone it is the energy-only evaluation of the line search);
// PASS 1 = pass B (shape gradient of surface + bending (+ tilt magnitude) and dV/dx).
// FAST fixes the configuration of the headline workload at compile time: closed mesh,
// uniform gamma / kappa / c0, surface + Helfrich bending (analytic) + volume, no tilt.
// ---------------------------------------------------------------------------
constexpr uint32_t kFastModules = MS_MOD_SURFACE | MS_MOD_BENDING | MS_MOD_VOLUME;

// ---- self-check build (-DMS_SELF_CHECK; libms_b200_checked.so): compute-sanitizer is closed on the GPU pool, so the
// hand-over protocol checks itself.  Every read-modify-write of an owned accumulator row takes a per-row lock word
// with atomicCAS and releases it afterwards: the packer promises that no two facets of a round write the same owned
// row, and the token ring that no two groups accumulate at the same time, so the CAS can never fail; the epilogue
// must find every lock free.  Local indices are bounds-checked.  Violations are counted in PatchLaunch::self_check
// (0: rows locked twice, 1: index out of range, 2: lock held at the epilogue).
#ifdef MS_SELF_CHECK
__shared__ int s_row_lock[2][kPatchOwnedCap + 16];
__device__ __forceinline__ void self_check_fail(const PatchLaunch& a, int which) {
  if (a.self_check) atomicAdd(a.self_check + which, 1);
}
__device__ __forceinline__ void self_check_lock(const PatchLaunch& a, int b, FacetRec rec, int n_owned, int n_local, bool lock) {
  const int idx[3] = {rec.a, rec.b, rec.c};
  for (int k = 0; k < 3; ++k) {
    if (idx[k] >= n_local) self_check_fail(a, 1);
    if (idx[k] >= n_owned) continue;
    if (lock) {
      if (atomicCAS(&s_row_lock[b][idx[k]], 0, 1) != 0) self_check_fail(a, 0);
    } else {
      __threadfence_block();
      atomicExch(&s_row_lock[b][idx[k]], 0);
    }
  }
}
#endif

// KKT coefficient of the single volume constraint (runtime/constraint_manager.py:294-301) or of the volume
// penalty (geometry/body.py:223-238): projected gradient = g + coef * gC.
__device__ __forceinline__ void kkt_coefficient(double* scalars, int mode, int has_gc, double k_vol, double v_target) {
  double coef = 0.0;
  if (has_gc) {
    if (mode == 0) {
      const double den = scalars[SC_GC_GC];
      coef = den > 1.0e-18 ? -(scalars[SC_G_GC] / den) : 0.0;
    } else if (mode == 1) {
      coef = k_vol * (scalars[SC_VOLUME] - v_target);
    }
  }
  scalars[SC_COEF] = coef;
  scalars[SC_LAMBDA] = (mode == 0) ? -coef : coef;
}

// Fixed-order sum of the per-CTA rows by ONE CTA (the last one of the evaluation): thread (row, k) sums slot k of
// rows row, row + kFinRows, ...; twelve threads then add the kFinRows row sums in index order.
constexpr int kFinRows = 32;
__device__ __forceinline__ void finalize_scalars(const PatchFinalize& f, double (*part)[kPartialStride], int tid) {
  if (tid < kFinRows * kPartialStride) {
    const int k = tid % kPartialStride, row = tid / kPartialStride;
    const bool from_b = (f.b_mask >> k) & 1u;
    const double* src = from_b ? f.partials_b : f.partials_a;
    const int count = from_b ? f.rows_b : f.rows_a;
    double v = 0.0;
    for (int p = row; p < count; p += kFinRows) v += __ldcg(src + size_t(p) * kPartialStride + k);
    part[row][k] = v;
  }
  __syncthreads();
  if (tid < kPartialStride) {
    double t = 0.0;
    for (int r = 0; r < kFinRows; ++r) t += part[r][tid];
    f.scalars[tid] = (tid == PS_VOLUME6) ? t / 6.0 : t;
  }
  __syncthreads();
  // energy-only evaluations (mode -2) leave the coefficient of the pending projection alone
  if (tid == 0 && f.constraint_mode != -2) kkt_coefficient(f.scalars, f.constraint_mode, f.has_gc, f.k_vol, f.v_target);
}

// Warp roles inside the 512-thread CTA: warps [0, NC/32) are consumers, warp NC/32 runs the
// patch epilogues, the last warp is the producer.
template <int PASS, int KIND, int NC>
__global__ void __launch_bounds__(NC + 64, 1) k_patch(PatchLaunch a, bool bending_b, bool scalars_here_arg) {
  extern __shared__ __align__(128) unsigned char smem[];
  using P = Plan<PASS>;
  const DevStrides ST{};
  const int tid = threadIdx.x;
  const int T = a.threads;
  int G = NC / T;
  if (G > kMaxGroups) G = kMaxGroups;
  const int n_active = G * T;  // consumer threads that take turns
  const int n_epi_warps = (NC + 32 - n_active) / 32;  // every warp between consumers and producer
  const int n_my = a.patch_count > int(blockIdx.x) ? (a.patch_count - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x) : 0;

  // KIND 0: everything decided at run time.  KIND 1 (headline): surface + Helfrich bending (analytic) +
  // volume, closed mesh, uniform parameters.  KIND 2: surface and/or volume only, uniform gamma (boundary
  // flags are irrelevant without bending).
  constexpr bool FAST = KIND == 1 || KIND == 2;  // KIND 3: run-time parameters but no tilt module
  const uint32_t modules = KIND == 1 ? kFastModules
                           : KIND == 2 ? (a.modules & (MS_MOD_SURFACE | MS_MOD_VOLUME)) : a.modules;
  const uint32_t flags = FAST ? 0u : a.flags;
  const bool do_tilt = KIND == 0 && (modules & MS_MOD_TILT) && a.tilts != nullptr;
  const bool has_boundary = !FAST && a.is_boundary != nullptr;
  const bool do_bending = (KIND == 1 || KIND == 3) ? true
                          : KIND == 2 ? false
                          : (PASS == 0 ? (modules & (MS_MOD_BENDING | MS_MOD_BENDING_TILT)) != 0 : bending_b);
  const bool do_volume = KIND == 1 ? true : (modules & MS_MOD_VOLUME) != 0;
  const bool scalars_here = (KIND == 1 || KIND == 3) ? false : scalars_here_arg;
  const bool want_epi = PASS == 1 || do_bending;  // pass A without bending accumulates nothing

  // mbarriers: full[2] producer -> all; empty[2] consumers (+ epilogue in pass A) -> producer;
  // acc_done[2] last round's group -> epilogue; acc_free[2] epilogue -> consumers
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + P::oBars);
  uint64_t* bar_full = bars;
  uint64_t* bar_empty = bars + 2;
  uint64_t* bar_done = bars + 4;
  uint64_t* bar_free = bars + 6;
  double* red = reinterpret_cast<double*>(smem + P::oRed);
  unsigned char* opt = smem + P::oOpt;
  int32_t* bfl_base = nullptr;
  double* t2_base = nullptr;
  double* ab_base = nullptr;
  if (has_boundary) { bfl_base = reinterpret_cast<int32_t*>(opt); opt += 2 * size_t(kPatchLocalCap) * 4; }
  if (do_tilt) { t2_base = reinterpret_cast<double*>(opt); opt += 2 * size_t(kPatchLocalCap) * 8; }
  if (do_tilt && PASS == 1) { ab_base = reinterpret_cast<double*>(opt); }

  PatchHdrS* mail = reinterpret_cast<PatchHdrS*>(smem + P::oMail);
  if (tid == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_full[b], 33);  // 32 asynchronous copy completions + the header write of lane 0
      mbar_init(&bar_empty[b], unsigned(n_active / 32));
      mbar_init(&bar_done[b], unsigned(T));
      mbar_init(&bar_free[b], 32u * unsigned(n_epi_warps));
    }
  }
  if (a.pull.own_flag && blockIdx.x == 0 && tid == 0) {  // in-kernel exchange: "my owned rows are written"
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(a.pull.own_flag) = a.pull.epoch;
    __threadfence_system();
  }
  if (a.wait_flags && tid < 64 && ((a.wait_mask >> tid) & 1ull)) {  // push transport: ghost rows in place?
    const volatile unsigned long long* f = a.wait_flags + tid;
    const long long t0 = clock64();
    while (*f < a.wait_epoch) {
      if (clock64() - t0 > kWaitCycles) {
        atomicExch(a.wait_error, 1);
        break;
      }
      __nanosleep(100);
    }
    __threadfence_system();
  }
  {  // zero both accumulator buffers (and the tilt area accumulators)
    double* acc0 = reinterpret_cast<double*>(smem + P::oAcc);
    for (int j = tid; j < 2 * P::kAccRows * kACap; j += NC + 64) acc0[j] = 0.0;
    if (ab_base)
      for (int j = tid; j < 2 * kACap; j += NC + 64) ab_base[j] = 0.0;
#ifdef MS_SELF_CHECK
    for (int j = tid; j < 2 * (kPatchOwnedCap + 16); j += NC + 64) (&s_row_lock[0][0])[j] = 0;
#endif
  }
  __syncthreads();

  if (tid >= NC + 32) {
    // =========================== producer warp ===========================
    const int lane = tid - (NC + 32);
#ifdef MS_DEBUG_VARIANTS
    const bool dbg_copy = !(a.debug & 8);   // 8: stage header, records and ids only (consumer-bound timing)
#else
    constexpr bool dbg_copy = true;
#endif
    // Software pipeline over the patches of this CTA.  The header of patch j+1 is loaded (registers) and its halo
    // ids are copied (into the id area of the OTHER input buffer, which its consumers never read) while patch j is
    // staged, so that the owned rows and the halo rows of a patch -- the latter need the ids -- are issued back to
    // back: one memory round trip per patch instead of three (header, level 1, level 2).  Completion is signalled
    // by the copies themselves (cp.async.mbarrier.arrive.noinc): the warp never waits for its bulk data, only for
    // the small id copy of the next patch, and has both buffers' copies in flight.
    auto patch_id = [&](int j) {
      const int pidx = a.patch_begin + int(blockIdx.x) + j * int(gridDim.x);
      return a.patch_list ? a.patch_list[pidx] : pidx;
    };
    auto stage_ids = [&](const PatchHeader& h, int b) {
      int32_t* ids = reinterpret_cast<int32_t*>(smem + size_t(b) * P::kInBytes + P::oIds);
      const int32_t* hsrc = a.halo_ids + h.halo_off;
      for (int k = lane; k < h.n_halo; k += 32) cp_async4(ids + k, hsrc + k);
    };
    auto load_header = [&](int j, PatchHeader& h, int& n_slots) {
      const int pid = patch_id(j);
      h = a.patches[pid];
      n_slots = int(a.patches[pid + 1].slot_off - h.slot_off);  // sentinel header at the end
    };
    PatchHeader h_cur{}, h_n1{}, h_n2{};
    int slots_cur = 0, slots_n1 = 0, slots_n2 = 0;
    bool ghosts_in_place = false;
    if (n_my > 0) {
      load_header(0, h_cur, slots_cur);
      if (n_my > 1) load_header(1, h_n1, slots_n1);
      stage_ids(h_cur, 0);
      cp_async_wait_all();
      __syncwarp();
    }
    for (int j = 0; j < n_my; ++j) {
      const int b = j & 1;
      const PatchHeader h = h_cur;
      const int n_slots = slots_cur;
      if (j + 2 < n_my) load_header(j + 2, h_n2, slots_n2);  // in flight while this patch is being issued
      if (j >= 2) mbar_wait_relaxed(&bar_empty[b], unsigned(((j >> 1) - 1) & 1));
      if (a.pull.n_ghost > 0 && !ghosts_in_place && int(blockIdx.x) + j * int(gridDim.x) >= a.pull.first_boundary) {
        // first patch of this CTA that reads ghost rows: every CTA must have copied its slice of them
        const volatile unsigned int* cnt = a.pull.arrived;
        const long long t0 = clock64();
        while (int(*cnt - a.pull.arrived_target) < 0) {
          if (clock64() - t0 > kWaitCycles) {
            atomicExch(a.pull.error, 1);
            break;
          }
          __nanosleep(100);
        }
        __threadfence();
        ghosts_in_place = true;
      }
      // ids of the NEXT patch into the other buffer's id area (free: the data of patch j-1 there may still be in
      // use, its ids are not).  Committed before this patch's bulk copies, so that wait_group 1 below waits for the
      // ids only.
      if (j + 1 < n_my) stage_ids(h_n1, b ^ 1);
      cp_async_commit();
      unsigned char* in = smem + size_t(b) * P::kInBytes;
      FacetRec* recs = reinterpret_cast<FacetRec*>(in + P::oRecs);
      const int32_t* ids = reinterpret_cast<const int32_t*>(in + P::oIds);  // arrived during the previous iteration
      const int Pn = h.n_owned;
      const bool with_seeds = PASS == 1 && do_bending;
      // Owned rows: ONE bulk copy per array.  The copy engine wants 16-byte aligned addresses and sizes; a row is 24
      // (40) bytes, so the copy starts at the even row v_lo - shift and covers an even number of rows; the consumers
      // address local vertex i at row shift + i of the buffer.  A last odd row travels with the halo rows.
      const int shift = h.v_lo & 1;
      const int n_bulk = dbg_copy ? ((shift + Pn) & ~1) : 0;
      double* pos = reinterpret_cast<double*>(in + P::oPos) + 3 * shift;
      double* seed = reinterpret_cast<double*>(in + P::oSeed) + kSeedStride * shift;
      if (lane == 0) {
        PatchHdrS* hs = reinterpret_cast<PatchHdrS*>(in + P::oHdr);
        hs->v_lo = h.v_lo; hs->n_owned = h.n_owned; hs->n_halo = h.n_halo; hs->n_rounds = h.n_rounds;
        hs->n_slots = n_slots; hs->halo_off = h.halo_off; hs->slot_off = h.slot_off;
        const unsigned rec_bytes = unsigned(n_slots) * unsigned(sizeof(FacetRec));   // n_slots is a multiple of 32
        const unsigned tx = rec_bytes + unsigned(n_bulk) * (with_seeds ? 64u : 24u);
        // release (the header is visible to whoever sees the phase complete) + the bytes the copy engine will deliver
        mbar_arrive_expect_tx(&bar_full[b], tx);
        if (rec_bytes) bulk_copy(recs, a.recs + h.slot_off, rec_bytes, &bar_full[b]);
        if (n_bulk) {
          const size_t g0 = size_t(h.v_lo - shift);
          bulk_copy(in + P::oPos, a.pos + g0 * 3, unsigned(n_bulk) * 24u, &bar_full[b]);
          if (with_seeds) bulk_copy(in + P::oSeed, a.seeds + g0 * kSeedStride, unsigned(n_bulk) * 40u, &bar_full[b]);
        }
      }
      auto stage_row = [&](int i, size_t row) {  // one vertex row with 8-byte asynchronous copies
        if (a.pull.n_ghost > 0 && int(row) >= a.pull.first_ghost_row) {
          // a ghost row copied by another CTA of THIS launch: LDGSTS.ca could hit an L1 line that an earlier patch
          // brought in for the neighbouring owned rows (rows n_owned - 1 and n_owned share lines), so read around L1
          const double* prow = a.pos + row * 3;
          pos[3 * i] = __ldcg(prow); pos[3 * i + 1] = __ldcg(prow + 1); pos[3 * i + 2] = __ldcg(prow + 2);
          if (with_seeds) {
            const double* srow = a.seeds + row * kSeedStride;
#pragma unroll
            for (int c = 0; c < kSeedStride; ++c) seed[kSeedStride * i + c] = __ldcg(srow + c);
          }
          return;
        }
        const double* prow = a.pos + row * 3;
        cp_async8(pos + 3 * i, prow);
        cp_async8(pos + 3 * i + 1, prow + 1);
        cp_async8(pos + 3 * i + 2, prow + 2);
        if (with_seeds) {
          const double* srow = a.seeds + row * kSeedStride;
#pragma unroll
          for (int c = 0; c < kSeedStride; ++c) cp_async8(seed + kSeedStride * i + c, srow + c);
        }
      };
      // halo rows (gathered by id) and the owned rows the bulk copy did not cover
      for (int k = lane; dbg_copy && k < h.n_halo; k += 32) stage_row(Pn + k, size_t(ids[k]));
      for (int i = n_bulk - shift + lane; dbg_copy && i < Pn; i += 32) stage_row(i, size_t(h.v_lo) + i);
      if (has_boundary || do_tilt) {  // flags (int32) and |t|^2 ride the same asynchronous copies
        int32_t* bf = has_boundary ? bfl_base + size_t(b) * kPatchLocalCap : nullptr;
        double* t2 = do_tilt ? t2_base + size_t(b) * kPatchLocalCap : nullptr;
        for (int i = lane; i < Pn; i += 32) {
          if (bf) cp_async4(bf + i, a.boundary32 + h.v_lo + i);
          if (t2) cp_async8(t2 + i, a.tilt_sq + h.v_lo + i);
        }
        for (int k = lane; k < h.n_halo; k += 32) {
          const size_t row = size_t(ids[k]);
          if (bf) cp_async4(bf + Pn + k, a.boundary32 + row);
          if (t2) cp_async8(t2 + Pn + k, a.tilt_sq + row);
        }
      }
      if (a.pull.n_ghost > 0) __threadfence_block();  // ghost rows were stored with plain stores (stage_row)
      cp_async_arrive_on(&bar_full[b]);   // one arrival per lane, when this lane's row copies have landed
      cp_async_commit();
      cp_async_wait_but_one();  // the ids of patch j+1 have landed; the bulk copies of patch j stay in flight
      __syncwarp();
      h_cur = h_n1; slots_cur = slots_n1;
      h_n1 = h_n2; slots_n1 = slots_n2;
    }
    cp_async_wait_all();
    return;
  }

  double sums[PS_COUNT];
#pragma unroll
  for (int k = 0; k < PS_COUNT; ++k) sums[k] = 0.0;

  if (tid >= n_active) {
    // =========================== epilogue warps ===========================
    // After the last round of a patch has been accumulated: vertex stage + seeds (pass A) or
    // gradient rows + KKT dot products (pass B) of the owned vertices; the accumulator is zeroed
    // on the way and handed back to the consumers.
    const int lane = tid - n_active;   // 0 .. 32*n_epi_warps-1: one owned vertex per lane and sweep
    const int epi_threads = 32 * n_epi_warps;
    const bool willmore = (flags & MS_FLAG_WILLMORE) != 0;
    if (a.pull.n_ghost > 0) {
      // In-kernel halo exchange (HaloPull): these warps have nothing to do until the first patch is accumulated.
      // Wait for the owners' flags, copy this CTA's slice of the ghost rows out of the owners' arrays, report.
      const HaloPull& hp = a.pull;
      for (int s = lane; s < hp.n_slots; s += epi_threads) {
        if (!hp.peer_flag[s] || !hp.peer_base[s]) continue;  // only the owners of this rank's ghosts
        const volatile unsigned long long* f = hp.peer_flag[s] + hp.flag_index;
        const long long t0 = clock64();
        while (*f < hp.epoch) {
          if (clock64() - t0 > kWaitCycles) {
            atomicExch(hp.error, 1);
            break;
          }
          __nanosleep(200);
        }
      }
      named_sync(14, epi_threads);
      __threadfence_system();
      const int total = hp.n_ghost * hp.width;
      for (int i = int(blockIdx.x) * epi_threads + lane; i < total; i += int(gridDim.x) * epi_threads) {
        const int g = i / hp.width, k = i - g * hp.width;
        hp.dst[i] = __ldcv(hp.peer_base[hp.owner[g]] + size_t(hp.row[g]) * hp.width + k);
      }
      __threadfence();
      named_sync(14, epi_threads);
      if (lane == 0) atomicAdd(hp.arrived, 1u);
    }
    for (int j = 0; want_epi && j < n_my; ++j) {
      const int b = j & 1;
      mbar_wait_relaxed(&bar_done[b], unsigned((j >> 1) & 1));   // every round accumulated, header mailed
      const PatchHdrS hs = mail[b];
      double* acc = reinterpret_cast<double*>(smem + P::oAcc + size_t(b) * P::kAccBytes);
      const int Pn = hs.n_owned;
      LocalA la;
      if (PASS == 0) {
        la.pos = nullptr;
        la.bfl = nullptr;  // boundary flags of the owned rows come from global memory below
        la.t2 = nullptr;
        la.acc = acc;
        la.P = Pn;
      }
      double* accAb = ab_base ? ab_base + size_t(b) * kACap : nullptr;
      for (int i = lane; i < Pn; i += epi_threads) {
        const size_t row = size_t(hs.v_lo) + i;
#ifdef MS_SELF_CHECK
        if (s_row_lock[b][i] != 0) self_check_fail(a, 2);
#endif
#ifdef MS_DEBUG_VARIANTS
        if (a.debug & 16) {  // 16: the epilogue only clears the accumulators
          for (int c = 0; c < P::kAccRows; ++c) acc[c * kACap + i] = 0.0;
          continue;
        }
#endif
        if (PASS == 0) {
          const double kap = (!FAST && a.kappa) ? a.kappa[row] : a.kappa_u;
          const double c0 = (!FAST && a.c0) ? a.c0[row] : a.c0_u;
          auto normal_of = [&](int v) { return vertex_normal_global(a, hs, v); };
          const bool on_boundary = has_boundary && a.is_boundary[row] != 0;
          const VertexSeed sd = vertex_body_a(ST, i, la, on_boundary, normal_of, kap, c0, willmore);
          sums[PS_E_BENDING] += sd.E;
          if (a.seeds) {
            double* o = a.seeds + row * kSeedStride;
            o[0] = sd.fK.x; o[1] = sd.fK.y; o[2] = sd.fK.z; o[3] = sd.fAe; o[4] = sd.fAv;
          }
          if (!FAST) {
            if (a.k_vecs) {
              a.k_vecs[3 * row] = acc[i];
              a.k_vecs[3 * row + 1] = acc[kACap + i];
              a.k_vecs[3 * row + 2] = acc[2 * kACap + i];
            }
            if (a.a_vor) a.a_vor[row] = acc[3 * kACap + i];
            if (a.a_eff) a.a_eff[row] = acc[4 * kACap + i];
            if (a.e_vertex) a.e_vertex[row] = sd.E;
          }
#pragma unroll
          for (int c = 0; c < 5; ++c) acc[c * kACap + i] = 0.0;
        } else {
          const double gx = acc[i], gy = acc[kACap + i], gz = acc[2 * kACap + i];
          double* go = a.grad + 3 * row;
          go[0] = gx; go[1] = gy; go[2] = gz;
          sums[PS_G_G] += gx * gx + gy * gy + gz * gz;
          acc[i] = 0.0; acc[kACap + i] = 0.0; acc[2 * kACap + i] = 0.0;
          if (do_volume && a.volgrad) {
            const double sixth = 1.0 / 6.0;  // the facets accumulated 6 dV/dx
            const double vx = sixth * acc[3 * kACap + i], vy = sixth * acc[4 * kACap + i], vz = sixth * acc[5 * kACap + i];
            double* vo = a.volgrad + 3 * row;
            vo[0] = vx; vo[1] = vy; vo[2] = vz;
            sums[PS_G_GC] += gx * vx + gy * vy + gz * vz;
            sums[PS_GC_GC] += vx * vx + vy * vy + vz * vz;
            acc[3 * kACap + i] = 0.0; acc[4 * kACap + i] = 0.0; acc[5 * kACap + i] = 0.0;
          }
          if (do_tilt && accAb) {
            if (a.tilt_grad) {  // tilt.py:163-170: dE/dt_v = k_t t_v A_bary(v)
              const double ab = accAb[i];
              a.tilt_grad[3 * row] = a.k_tilt * a.tilts[3 * row] * ab;
              a.tilt_grad[3 * row + 1] = a.k_tilt * a.tilts[3 * row + 1] * ab;
              a.tilt_grad[3 * row + 2] = a.k_tilt * a.tilts[3 * row + 2] * ab;
            }
            accAb[i] = 0.0;
          }
        }
      }
      mbar_arrive(&bar_free[b]);
    }
  } else {
    // ============================= consumers =============================
    const int grp = tid / T, lane = tid - grp * T;
    const int bar_mine = 1 + grp, bar_next = 1 + (grp + 1 == G ? 0 : grp + 1);
    const int ring = 2 * T;
#ifdef MS_DEBUG_VARIANTS  // timing experiments (libms_b200_dbg.so): parts of the loop switched off, results wrong
    const int dbg = a.debug;
#else
    constexpr int dbg = 0;
#endif
    const bool use_ring = G > 1 && !(dbg & 1);
    const bool dbg_sync = !(dbg & 1), dbg_acc = !(dbg & 2), dbg_compute = !(dbg & 4);
    if (use_ring && grp == G - 1) named_arrive(1, ring);  // group 0 owns the first token
    int t_rel = grp;   // my next round, relative to the first round of the current patch
    int64_t turns_done = 0;
    for (int j = 0; j < n_my; ++j) {
      const int b = j & 1;
      mbar_wait(&bar_full[b], unsigned((j >> 1) & 1));
      if (want_epi && j >= 2) mbar_wait(&bar_free[b], unsigned(((j >> 1) - 1) & 1));  // accumulator drained
      unsigned char* in = smem + size_t(b) * P::kInBytes;
      const PatchHdrS hs = *reinterpret_cast<const PatchHdrS*>(in + P::oHdr);
      const FacetRec* recs = reinterpret_cast<const FacetRec*>(in + P::oRecs);
      double* acc = reinterpret_cast<double*>(smem + P::oAcc + size_t(b) * P::kAccBytes);
      const int Pn = hs.n_owned;
      // a patch without facets still takes one (empty) round so that its epilogue is triggered
      const int n_turns = hs.n_rounds > 0 ? hs.n_rounds : 1;
      const double* slot_gamma = (!FAST && a.slot_gamma) ? a.slot_gamma + hs.slot_off : nullptr;

      LocalA la;
      LocalB lb;
      if (PASS == 0) {
        la.pos = reinterpret_cast<const double*>(in + P::oPos) + 3 * (hs.v_lo & 1);
        la.bfl = has_boundary ? bfl_base + size_t(b) * kPatchLocalCap : nullptr;
        la.t2 = do_tilt ? t2_base + size_t(b) * kPatchLocalCap : nullptr;
        la.acc = acc;
        la.P = Pn;
      } else {
        lb.pos = reinterpret_cast<const double*>(in + P::oPos) + 3 * (hs.v_lo & 1);
        lb.seed = reinterpret_cast<const double*>(in + P::oSeed) + kSeedStride * (hs.v_lo & 1);
        lb.bfl = has_boundary ? bfl_base + size_t(b) * kPatchLocalCap : nullptr;
        lb.t2 = do_tilt ? t2_base + size_t(b) * kPatchLocalCap : nullptr;
        lb.acc = acc;
        lb.accAb = ab_base ? ab_base + size_t(b) * kACap : nullptr;
        lb.P = Pn;
      }

      for (; t_rel < n_turns; t_rel += G) {
        const int slot = t_rel * T + lane;
        FacetRec rec;
        rec.a = rec.b = rec.c = 0; rec.flags = 0;
        if (slot < hs.n_slots) rec = load_rec(recs + slot);
        const bool valid = (rec.flags & REC_VALID) != 0;
        if (PASS == 0) {
          CornerA ca;
          if (valid && dbg_compute) {
            const double gam = slot_gamma ? slot_gamma[slot] : a.gamma_u;
            ca = facet_compute_a(ST, rec, gam, la, modules, a.k_tilt, sums);
          }
          if (use_ring) named_sync(bar_mine, ring); else if (dbg_sync) named_sync(1, T);
#ifdef MS_SELF_CHECK
          if (valid && do_bending) self_check_lock(a, b, rec, Pn, Pn + hs.n_halo, true);
#endif
          if (valid && do_bending && dbg_acc) facet_accumulate_a(ST, rec, ca, la, modules);
#ifdef MS_SELF_CHECK
          if (valid && do_bending) self_check_lock(a, b, rec, Pn, Pn + hs.n_halo, false);
#endif
        } else {
          FacetOutB out;
          if (valid && dbg_compute) {
            const double gam = slot_gamma ? slot_gamma[slot] : a.gamma_u;
            out = do_bending ? facet_compute_b<true>(ST, rec, gam, lb, modules, flags, a.k_tilt, scalars_here, sums)
                             : facet_compute_b<false>(ST, rec, gam, lb, modules, flags, a.k_tilt, scalars_here, sums);
          }
          if (use_ring) named_sync(bar_mine, ring); else if (dbg_sync) named_sync(1, T);
#ifdef MS_SELF_CHECK
          if (valid) self_check_lock(a, b, rec, Pn, Pn + hs.n_halo, true);
#endif
          if (valid && dbg_acc) facet_accumulate_b(ST, rec, out, lb, do_volume, do_tilt);
#ifdef MS_SELF_CHECK
          if (valid) self_check_lock(a, b, rec, Pn, Pn + hs.n_halo, false);
#endif
        }
        // the last round of the patch hands the accumulator (and the header) to the epilogue warps
        if (want_epi && t_rel == n_turns - 1) {
          if (lane == 0) mail[b] = hs;
          mbar_arrive(&bar_done[b]);
        }
        if (use_ring) named_arrive(bar_next, ring);
      }
      t_rel -= n_turns;
      turns_done += n_turns;
      // leaving the patch: its input buffer may be refilled
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(&bar_empty[b]);
    }
    // swallow the token left over by the last turn
    if (use_ring && int(turns_done % G) == grp) named_sync(bar_mine, ring);
  }

  block_sum<PS_COUNT>(sums, red, NC + 32, 15);
  if (tid == 0) {
    double* p = a.partials + (size_t(a.partial_row0) + blockIdx.x) * kPartialStride;
#pragma unroll
    for (int k = 0; k < PS_COUNT; ++k) p[k] = sums[k];
  }
  if (a.fin.ticket) {  // the last CTA to get here finalises the evaluation (warp-uniform: a kernel parameter)
    __shared__ int s_last;
    __shared__ double s_part[kFinRows][kPartialStride];
    const bool to_peers = a.fin.signal_flag || a.fin.publish_words || a.fin.push_words;
    if (tid == 0) {
      if (to_peers) __threadfence_system(); else __threadfence();
      s_last = atomicAdd(a.fin.ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      if (a.fin.scalars) finalize_scalars(a.fin, s_part, tid);
      if (a.fin.publish_words) {  // publish half of the all-reduce over peer memory (k_allreduce_publish)
        double* slot = reinterpret_cast<double*>(a.fin.publish_words + 8 + 16 * (a.fin.publish_epoch & 1ull));
        if (tid < kPartialStride) slot[tid] = a.fin.scalars[tid];
        __syncthreads();
      }
      if (a.fin.push_words) {  // push transport: scalars into this rank's slot of every rank's block, then its word
        const unsigned long long e = a.fin.publish_epoch;
        for (int i = tid; i < a.fin.push_slots * kPartialStride; i += NC + 64) {
          const int s = i / kPartialStride, k = i - s * kPartialStride;
          double* slot = reinterpret_cast<double*>(a.fin.push_words[s] + kPushScalarBase) +
                         (16 * int(e & 1ull) + a.fin.push_my_slot) * 16;
          slot[k] = a.fin.scalars[k];
        }
        __threadfence_system();
        __syncthreads();
        if (tid < a.fin.push_slots) {
          *reinterpret_cast<volatile unsigned long long*>(a.fin.push_words[tid] + kPushScalarFlagBase + a.fin.push_my_slot) = e;
          __threadfence_system();
        }
      }
      if (tid == 0) {
        *a.fin.ticket = 0u;
        if (to_peers) {
          __threadfence_system();
          if (a.fin.signal_flag) *reinterpret_cast<volatile unsigned long long*>(a.fin.signal_flag) = a.fin.signal_epoch;
          if (a.fin.publish_words)
            *reinterpret_cast<volatile unsigned long long*>(a.fin.publish_words + 2) = a.fin.publish_epoch;
          __threadfence_system();
        }
      }
      if (a.fin.gather_words) {  // the other half of the all-reduce, in place (k_allreduce_gather_coef)
        __shared__ int s_ok;
        const unsigned long long e = a.fin.publish_epoch;
        if (tid == 0) s_ok = 1;
        __syncthreads();
        for (int s = tid; s < a.fin.gather_slots; s += NC + 64) {
          const volatile unsigned long long* f = a.fin.gather_words[s] + 2;
          const long long t0 = clock64();
          while (*f < e) {
            if (clock64() - t0 > kWaitCycles) {
              atomicExch(a.fin.gather_error, 1);
              s_ok = 0;
              break;
            }
            __nanosleep(100);
          }
        }
        __syncthreads();
        if (s_ok) {
          __threadfence_system();
          if (tid < kPartialStride) {
            double acc = 0.0;
            for (int s = 0; s < a.fin.gather_slots; ++s)
              acc += __ldcv(reinterpret_cast<const double*>(a.fin.gather_words[s] + 8 + 16 * (e & 1ull)) + tid);
            a.fin.scalars[tid] = acc;
          }
          __syncthreads();
          if (tid == 0 && a.fin.gather_mode != -2)
            kkt_coefficient(a.fin.scalars, a.fin.gather_mode, a.fin.has_gc, a.fin.k_vol, a.fin.v_target);
        }
      }
    }
  }
}

// Fixed-order reduction of the per-CTA partial sums of pass A and pass B (one CTA of
// 64 x 12 threads: thread (row, k) sums slot k of rows row, row+64, ... and 12 threads then
// add the 64 row sums in index order).  Slot k comes from pass B's rows when bit k of
// b_mask is set, else from pass A's.
constexpr int kReduceRows = 64;
__global__ void __launch_bounds__(kReduceRows* kPartialStride)
    k_reduce_partials(const double* __restrict__ pa, int rows_a, const double* __restrict__ pb, int rows_b,
                      unsigned b_mask, double* scalars) {
  __shared__ double part[kReduceRows][kPartialStride];
  const int k = threadIdx.x % kPartialStride, row = threadIdx.x / kPartialStride;
  const bool from_b = (b_mask >> k) & 1u;
  const double* src = from_b ? pb : pa;
  const int count = from_b ? rows_b : rows_a;
  double v = 0.0;
  for (int p = row; p < count; p += kReduceRows) v += src[size_t(p) * kPartialStride + k];
  part[row][k] = v;
  __syncthreads();
  if (threadIdx.x < kPartialStride) {
    double t = 0.0;
    for (int r = 0; r < kReduceRows; ++r) t += part[r][threadIdx.x];
    scalars[threadIdx.x] = (threadIdx.x == PS_VOLUME6) ? t / 6.0 : t;
  }
}

// ---------------------------------------------------------------------------
// KKT projection helpers (runtime/constraint_manager.py:294-301).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dots(const double* __restrict__ g,
                                              const double* __restrict__ gc, int64_t n,
                                              double* block_partials) {
  __shared__ double red[32 * 3];
  double v[3] = {0.0, 0.0, 0.0};
  // fixed chunk per block -> fixed summation order
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = per * blockIdx.x, hi = (lo + per < n) ? lo + per : n;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double a = g[i], b = gc ? gc[i] : 0.0;
    v[0] += a * a;
    v[1] += a * b;
    v[2] += b * b;
  }
  block_sum<3>(v, red, 256, 0);
  if (threadIdx.x == 0) {
    block_partials[3 * blockIdx.x] = v[0];
    block_partials[3 * blockIdx.x + 1] = v[1];
    block_partials[3 * blockIdx.x + 2] = v[2];
  }
}

__global__ void __launch_bounds__(256) k_dots_final(const double* __restrict__ block_partials,
                                                    int n_blocks, double* scalars) {
  __shared__ double red[32 * 3];
  double v[3] = {0.0, 0.0, 0.0};
  for (int p = threadIdx.x; p < n_blocks; p += blockDim.x) {
    v[0] += block_partials[3 * p];
    v[1] += block_partials[3 * p + 1];
    v[2] += block_partials[3 * p + 2];
  }
  block_sum<3>(v, red, 256, 0);
  if (threadIdx.x == 0) {
    scalars[SC_G_G] = v[0];
    scalars[SC_G_GC] = v[1];
    scalars[SC_GC_GC] = v[2];
  }
}

__global__ void __launch_bounds__(256) k_project(double* g, const double* __restrict__ gc,
                                                 const uint8_t* __restrict__ fixed, int64_t nv,
                                                 double* scalars, int mode, double k_vol,
                                                 double v_target) {
  double coef = 0.0;
  if (gc) {
    if (mode == 0) {
      const double den = scalars[SC_GC_GC];
      coef = den > 1.0e-18 ? -(scalars[SC_G_GC] / den) : 0.0;
    } else {
      coef = k_vol * (scalars[SC_VOLUME] - v_target);
    }
  }
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i == 0) scalars[SC_LAMBDA] = (mode == 0) ? -coef : coef;
  if (i >= 3 * nv) return;
  double x = g[i];
  if (gc) x += coef * gc[i];
  if (fixed && fixed[i / 3]) x = 0.0;
  g[i] = x;
}

__global__ void k_kkt_coefficient(double* scalars, int mode, int has_gc, double k_vol, double v_target) {
  kkt_coefficient(scalars, mode, has_gc, k_vol, v_target);
}

__device__ __forceinline__ double projected_at(const double* __restrict__ g, const double* __restrict__ gc,
                                               const uint8_t* __restrict__ fixed, double coef, int64_t i) {
  if (fixed && fixed[i / 3]) return 0.0;
  double x = g[i];
  if (gc) x += coef * gc[i];
  return x;
}

__global__ void __launch_bounds__(256) k_apply_projection(double* g, const double* __restrict__ gc,
                                                          const uint8_t* __restrict__ fixed, int64_t nv,
                                                          const double* __restrict__ scalars) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= 3 * nv) return;
  g[i] = projected_at(g, gc, fixed, scalars[SC_COEF], i);
}

__global__ void __launch_bounds__(256) k_scale_projected(const double* __restrict__ g, const double* __restrict__ gc,
                                                         const uint8_t* __restrict__ fixed, int64_t nv,
                                                         const double* __restrict__ scalars, double scale, double* out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= 3 * nv) return;
  out[i] = scale * projected_at(g, gc, fixed, scalars[SC_COEF], i);
}

__global__ void __launch_bounds__(256) k_dots_projected(const double* __restrict__ g, const double* __restrict__ gc,
                                                        const uint8_t* __restrict__ fixed, const double* __restrict__ d,
                                                        int64_t n, const double* __restrict__ scalars, double* block_partials) {
  __shared__ double red[32 * 3];
  double v[3] = {0.0, 0.0, 0.0};
  const double coef = scalars[SC_COEF];
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = per * blockIdx.x, hi = (lo + per < n) ? lo + per : n;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const double a = projected_at(g, gc, fixed, coef, i), b = d[i];
    v[0] += a * a;
    v[1] += a * b;
    v[2] += b * b;
  }
  block_sum<3>(v, red, 256, 0);
  if (threadIdx.x == 0) {
    block_partials[3 * blockIdx.x] = v[0];
    block_partials[3 * blockIdx.x + 1] = v[1];
    block_partials[3 * blockIdx.x + 2] = v[2];
  }
}

__global__ void __launch_bounds__(256) k_gather_rows(const double* __restrict__ src, int width,
                                                     const int32_t* __restrict__ rows, int64_t n,
                                                     double* out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n * width) return;
  const int64_t r = i / width;
  const int c = int(i - r * width);
  out[i] = src[size_t(rows[r]) * width + c];
}

// out[rows[r], :] = src[r, :]  (inverse of k_gather_rows: internal row order -> caller's order)
__global__ void __launch_bounds__(256) k_scatter_rows(const double* __restrict__ src, int width,
                                                      const int32_t* __restrict__ rows, int64_t n,
                                                      double* out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n * width) return;
  const int64_t r = i / width;
  const int c = int(i - r * width);
  out[size_t(rows[r]) * width + c] = src[i];
}

// alpha_dev (device, may be null) replaces alpha: the device-controlled line search (ms_ctx_minimize)
__global__ void __launch_bounds__(256) k_axpy(const double* __restrict__ x,
                                              const double* __restrict__ d, double alpha,
                                              const double* __restrict__ alpha_dev, double* out, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (alpha_dev) alpha = *alpha_dev;
  if (i < n) out[i] = x[i] + alpha * d[i];
}

// ---------------------------------------------------------------------------
// Generic triangle-soup kernels (stateless shims): per-facet pass writes corner
// contributions, per-vertex pass gathers them through the corner CSR in fixed order.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool soup_facet(const SoupArgs& s, int f, int& i0, int& i1, int& i2) {
  i0 = s.tri[3 * size_t(f)] + s.shift;
  i1 = s.tri[3 * size_t(f) + 1] + s.shift;
  i2 = s.tri[3 * size_t(f) + 2] + s.shift;
  return i0 >= 0 && i0 < s.nv && i1 >= 0 && i1 < s.nv && i2 >= 0 && i2 < s.nv;
}

__device__ __forceinline__ void st3(double* p, size_t i, d3 v) {
  p[3 * i] = v.x; p[3 * i + 1] = v.y; p[3 * i + 2] = v.z;
}

__global__ void k_soup_surface(SoupArgs s, const double* __restrict__ gamma, double* corner,
                               double* facet_e) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= s.nf) return;
  int i0, i1, i2;
  d3 z = make_d3(0, 0, 0);
  CornerG cg; cg.g0 = z; cg.g1 = z; cg.g2 = z;
  double e = 0.0;
  if (soup_facet(s, f, i0, i1, i2)) {
    const FacetGeom g = facet_geom(ld3(s.pos, i0), ld3(s.pos, i1), ld3(s.pos, i2));
    if (g.S >= kSurfaceSkip) {
      BendIn b;
      cg = facet_pass_b<false>(g, gamma[f], 0.0, b, false);
      e = gamma[f] * (0.5 * g.S);
    }
  }
  st3(corner, 3 * size_t(f), cg.g0);
  st3(corner, 3 * size_t(f) + 1, cg.g1);
  st3(corner, 3 * size_t(f) + 2, cg.g2);
  facet_e[f] = e;
}

__global__ void k_soup_volume(SoupArgs s, double factor, double* corner, double* facet_v) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= s.nf) return;
  int i0, i1, i2;
  d3 z = make_d3(0, 0, 0);
  CornerG cg; cg.g0 = z; cg.g1 = z; cg.g2 = z;
  double v6 = 0.0;
  if (soup_facet(s, f, i0, i1, i2)) {
    const d3 v0 = ld3(s.pos, i0), v1 = ld3(s.pos, i1), v2 = ld3(s.pos, i2);
    cg = facet_volume_grad(v0, v1, v2);
    v6 = facet_volume6(v0, v1, v2);
  }
  st3(corner, 3 * size_t(f), factor * cg.g0);
  st3(corner, 3 * size_t(f) + 1, factor * cg.g1);
  st3(corner, 3 * size_t(f) + 2, factor * cg.g2);
  facet_v[f] = v6;
}

// corner payload: 4 doubles per corner (K.x,K.y,K.z,va)
__global__ void k_soup_curvature(SoupArgs s, double* corner, double* weights, double* va0,
                                 double* va1, double* va2) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= s.nf) return;
  int i0, i1, i2;
  CornerA c;
  d3 z = make_d3(0, 0, 0);
  c.K0 = z; c.K1 = z; c.K2 = z;
  c.va0 = c.va1 = c.va2 = 0.0;
  c.c0 = c.c1 = c.c2 = 0.0;
  if (soup_facet(s, f, i0, i1, i2)) {
    const FacetGeom g = facet_geom(ld3(s.pos, i0), ld3(s.pos, i1), ld3(s.pos, i2));
    c = facet_pass_a(g, false, false, false);
  }
  double* o = corner + 12 * size_t(f);
  o[0] = c.K0.x; o[1] = c.K0.y; o[2] = c.K0.z; o[3] = c.va0;
  o[4] = c.K1.x; o[5] = c.K1.y; o[6] = c.K1.z; o[7] = c.va1;
  o[8] = c.K2.x; o[9] = c.K2.y; o[10] = c.K2.z; o[11] = c.va2;
  weights[3 * size_t(f)] = c.c0; weights[3 * size_t(f) + 1] = c.c1; weights[3 * size_t(f) + 2] = c.c2;
  if (va0) va0[f] = c.va0;
  if (va1) va1[f] = c.va1;
  if (va2) va2[f] = c.va2;
}

__global__ void k_soup_laplacian(SoupArgs s, int dim, const double* __restrict__ weights,
                                 const double* __restrict__ field, double* corner) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= s.nf) return;
  int i0, i1, i2;
  const bool ok = soup_facet(s, f, i0, i1, i2);
  const double c0 = weights[3 * size_t(f)], c1 = weights[3 * size_t(f) + 1],
               c2 = weights[3 * size_t(f) + 2];
  double* o = corner + size_t(f) * 3 * dim;
  for (int d = 0; d < dim; ++d) {
    double a = 0.0, b = 0.0, c = 0.0;
    if (ok) {
      const double f0 = field[size_t(i0) * dim + d], f1 = field[size_t(i1) * dim + d],
                   f2 = field[size_t(i2) * dim + d];
      a = 0.5 * (c1 * (f0 - f2) + c2 * (f0 - f1));
      b = 0.5 * (c2 * (f1 - f0) + c0 * (f1 - f2));
      c = 0.5 * (c0 * (f2 - f1) + c1 * (f2 - f0));
    }
    o[d] = a; o[dim + d] = b; o[2 * dim + d] = c;
  }
}

// out[v*out_stride + d] (+)= sum over corners of v of corner[c*in_stride + d], d < dim
__global__ void k_gather(int nv, const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                         const double* __restrict__ corner, int in_stride, int in_off, int dim,
                         double* out, int out_stride, int accumulate) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  if (dim == 3) {  // the common case: one pass over the corner list, three running sums (same order per component)
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
    for (int j = ptr[v]; j < ptr[v + 1]; ++j) {
      const double* q = corner + size_t(idx[j]) * in_stride + in_off;
      a0 += q[0];
      a1 += q[1];
      a2 += q[2];
    }
    double* o = out + size_t(v) * out_stride;
    o[0] = accumulate ? o[0] + a0 : a0;
    o[1] = accumulate ? o[1] + a1 : a1;
    o[2] = accumulate ? o[2] + a2 : a2;
    return;
  }
  for (int d = 0; d < dim; ++d) {
    double acc = 0.0;
    for (int j = ptr[v]; j < ptr[v + 1]; ++j) acc += corner[size_t(idx[j]) * in_stride + in_off + d];
    double* o = out + size_t(v) * out_stride + d;
    *o = accumulate ? *o + acc : acc;
  }
}

__global__ void k_grad_cotan(int n, const double* __restrict__ u, const double* __restrict__ v,
                             double* gu, double* gv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  d3 a, b;
  grad_cotan(ld3(u, i), ld3(v, i), a, b);
  st3(gu, i, a);
  st3(gv, i, b);
}

__global__ void k_p1_divergence(SoupArgs s, const double* __restrict__ tilts, double* div,
                                double* area, double* g0, double* g1, double* g2) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= s.nf) return;
  int i0, i1, i2;
  P1 p;
  d3 z = make_d3(0, 0, 0);
  p.g0 = z; p.g1 = z; p.g2 = z; p.div = 0.0; p.area = 0.0;
  if (soup_facet(s, f, i0, i1, i2)) {
    const FacetGeom g = facet_geom(ld3(s.pos, i0), ld3(s.pos, i1), ld3(s.pos, i2));
    p = facet_p1(g, ld3(tilts, i0), ld3(tilts, i1), ld3(tilts, i2));
  }
  div[f] = p.div;
  area[f] = p.area;
  st3(g0, f, p.g0);
  st3(g1, f, p.g1);
  st3(g2, f, p.g2);
}

// barycentric-area-averaged vertex divergence (geometry/tilt_operators.py:414-465): fixed-order gather
__global__ void k_p1_vertex_divergence(SoupArgs s, const double* __restrict__ div, const double* __restrict__ area,
                                       double* div_v, double* area_v) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= s.nv) return;
  double num = 0.0, den = 0.0;
  for (int j = s.csr_ptr[v]; j < s.csr_ptr[v + 1]; ++j) {
    const int f = s.csr_idx[j] / 3;
    const double w = area[f] / 3.0;
    num += w * div[f];
    den += w;
  }
  div_v[v] = den > 1.0e-20 ? num / den : 0.0;
  area_v[v] = den;
}

// single-CTA fixed-order sum (stateless shims only; sizes are modest there)
__global__ void __launch_bounds__(256) k_sum(const double* __restrict__ x, int64_t n, double scale,
                                             double* out) {
  __shared__ double red[32];
  double v[1] = {0.0};
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) v[0] += x[i];
  block_sum<1>(v, red, 256, 0);
  if (threadIdx.x == 0) *out = v[0] * scale;
}

// Two-stage fixed-order sum for long arrays: block b sums the contiguous chunk b (threads strided inside
// it) into partial[b]; k_sum then adds the partials in index order.  Same result on every run.
__global__ void __launch_bounds__(256) k_sum_partial(const double* __restrict__ x, int64_t n, double* partial) {
  __shared__ double red[32];
  const int64_t chunk = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = chunk * blockIdx.x, hi = lo + chunk < n ? lo + chunk : n;
  double v[1] = {0.0};
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) v[0] += x[i];
  block_sum<1>(v, red, 256, 0);
  if (threadIdx.x == 0) partial[blockIdx.x] = v[0];
}

// ---- bending-tilt coupling (ms_bt.cuh): per-facet / per-vertex passes on global arrays ----
__global__ void __launch_bounds__(128) k_bt_facet_a(BtMesh m, double sign, double* corner4) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < m.nf) bt_facet_a(m, f, sign, corner4);
}

__global__ void __launch_bounds__(128) k_bt_vertex(BtMesh m, const double* __restrict__ k_vecs,
                                                   const double* __restrict__ a_vor,
                                                   const double* __restrict__ a_eff,
                                                   const double* __restrict__ corner4, double* seeds, double* base) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < m.nv) bt_vertex(m, v, k_vecs, a_vor, a_eff, corner4, seeds, base);
}

__global__ void __launch_bounds__(128) k_bt_facet_b(BtMesh m, const double* __restrict__ base, double sign,
                                                    double* corner3, double* facet_e) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < m.nf) facet_e[f] = bt_facet_b(m, f, base, sign, corner3);
}

// scalars[E_BENDING_TILT] <- *e_bt; the pass-A bending energy slot was only a by-product here
__global__ void k_bt_finalize(const double* e_bt, double* scalars) {
  scalars[SC_E_BENDING_TILT] = *e_bt;
  scalars[SC_E_BENDING] = 0.0;
}

// ---- leaflet tilt modules (ms_leaflet.cuh): three sweeps on global arrays + fixed-order gathers ----
__global__ void __launch_bounds__(128) k_lf_facet_a(LeafletMesh m, double* corner) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < m.nf) lf_facet_a(m, f, corner);
}

__global__ void __launch_bounds__(128) k_lf_vertex(LeafletMesh m, const double* __restrict__ corner, double* vbuf) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < m.nv) lf_vertex(m, v, corner, vbuf);
}

__global__ void __launch_bounds__(128) k_lf_facet_b(LeafletMesh m, const double* __restrict__ vbuf, int with_bt,
                                                    int with_tilt, int with_smooth, double* corner_shape,
                                                    double* corner_tilt,
                                                    double* facet_e /* [e_bt (nf) | e_tilt (nf) | e_smooth (nf)] */) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= m.nf) return;
  const LfEnergies e = lf_facet_b(m, f, vbuf, with_bt != 0, with_tilt != 0, with_smooth != 0, corner_shape, corner_tilt);
  facet_e[f] = e.e_bt;
  facet_e[size_t(m.nf) + f] = e.e_tilt;
  facet_e[2 * size_t(m.nf) + f] = e.e_smooth;
}

// ---- small meshes: the whole leaflet evaluation in ONE cooperative launch ----
// The three sweeps, the energy sums and the gathers of a mesh of a few thousand facets take a few microseconds
// each; as separate launches they cost ~50 us of launch latency and pipeline drain.  Here they are phases of one
// grid (all CTAs resident: cudaLaunchCooperativeKernel) separated by a grid barrier on a 64-bit ticket counter
// that only ever grows (no reset between launches: barrier k of this launch waits for base + k * gridDim.x).
__device__ __forceinline__ void lf_grid_barrier(unsigned long long* ticket, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ticket, 1ull);
    while (*reinterpret_cast<volatile unsigned long long*>(ticket) < target) {
    }
    __threadfence();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(128) k_lf_fused(LeafletMesh m, int with_bt, int with_tilt, int with_smooth, double* corner,
                                                  double* vbuf, double* corner_shape, double* corner_tilt,
                                                  double* block_e /* 3 * gridDim.x */, double* e_out3, double* grad,
                                                  int accumulate_grad, double* tilt_grad, int accumulate_tilt_grad,
                                                  unsigned long long* ticket, unsigned long long base) {
  __shared__ double red[32 * 3];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  unsigned long long target = base;
  if (with_bt) {
    for (int f = tid; f < m.nf; f += stride) lf_facet_a(m, f, corner);
    lf_grid_barrier(ticket, target += gridDim.x);
    for (int v = tid; v < m.nv; v += stride) lf_vertex(m, v, corner, vbuf);
    lf_grid_barrier(ticket, target += gridDim.x);
  }
  double e[3] = {0.0, 0.0, 0.0};
  for (int f = tid; f < m.nf; f += stride) {
    const LfEnergies r = lf_facet_b(m, f, vbuf, with_bt != 0, with_tilt != 0, with_smooth != 0,
                                    grad ? corner_shape : nullptr, tilt_grad ? corner_tilt : nullptr);
    e[0] += r.e_bt;
    e[1] += r.e_tilt;
    e[2] += r.e_smooth;
  }
  block_sum<3>(e, red, 128, 0);
  if (threadIdx.x == 0) {
    block_e[3 * blockIdx.x] = e[0];
    block_e[3 * blockIdx.x + 1] = e[1];
    block_e[3 * blockIdx.x + 2] = e[2];
  }
  lf_grid_barrier(ticket, target += gridDim.x);
  if (blockIdx.x == 0 && threadIdx.x < 3) {  // fixed order: block 0, 1, 2, ...
    double acc = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) acc += block_e[3 * b + threadIdx.x];
    e_out3[threadIdx.x] = acc;
  }
  for (int v = tid; v < m.nv; v += stride) {
    for (int which = 0; which < 2; ++which) {
      double* out = which == 0 ? grad : tilt_grad;
      if (!out) continue;
      const double* src = which == 0 ? corner_shape : corner_tilt;
      const bool acc = which == 0 ? accumulate_grad != 0 : accumulate_tilt_grad != 0;
      double a0 = 0.0, a1 = 0.0, a2 = 0.0;
      for (int j = m.csr_ptr[v]; j < m.csr_ptr[v + 1]; ++j) {
        const double* q = src + 3 * size_t(m.csr_idx[j]);
        a0 += q[0];
        a1 += q[1];
        a2 += q[2];
      }
      double* o = out + 3 * size_t(v);
      o[0] = acc ? o[0] + a0 : a0;
      o[1] = acc ? o[1] + a1 : a1;
      o[2] = acc ? o[2] + a2 : a2;
    }
  }
}

// Both leaflets of a small mesh in ONE cooperative launch: the work items of the two leaflets share every phase
// (item i < n belongs to the inner leaflet, i >= n to the outer one), so a tilt relaxation iteration costs one
// launch instead of two.  Same per-item code and the same gather order as k_lf_fused: the gradients are bitwise
// those of two separate evaluations (inner first, outer accumulated on top).
struct LfPairBuffers {
  double* corner[2];
  double* vbuf[2];
  double* shape[2];
  double* tilt[2];
  double* e_out3[2];
  double* tilt_grad[2];
};

__global__ void __launch_bounds__(128) k_lf_fused_pair(LeafletMesh m0, LeafletMesh m1, LfPairBuffers b, int with_bt,
                                                       int with_tilt, int with_smooth, double* block_e /* 6 * gridDim.x */,
                                                       double* grad, int accumulate_grad, int accumulate_tilt_grad,
                                                       unsigned long long* ticket, unsigned long long base) {
  __shared__ double red[32 * 6];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  const int nf = m0.nf, nv = m0.nv;
  unsigned long long target = base;
  if (with_bt) {
    for (int i = tid; i < 2 * nf; i += stride) {
      const int l = i >= nf;
      lf_facet_a(l ? m1 : m0, i - l * nf, b.corner[l]);
    }
    lf_grid_barrier(ticket, target += gridDim.x);
    for (int i = tid; i < 2 * nv; i += stride) {
      const int l = i >= nv;
      lf_vertex(l ? m1 : m0, i - l * nv, b.corner[l], b.vbuf[l]);
    }
    lf_grid_barrier(ticket, target += gridDim.x);
  }
  double e[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int i = tid; i < 2 * nf; i += stride) {
    const int l = i >= nf;
    const LfEnergies r = lf_facet_b(l ? m1 : m0, i - l * nf, b.vbuf[l], with_bt != 0, with_tilt != 0, with_smooth != 0,
                                    grad ? b.shape[l] : nullptr, b.tilt_grad[l] ? b.tilt[l] : nullptr);
    e[3 * l] += r.e_bt;
    e[3 * l + 1] += r.e_tilt;
    e[3 * l + 2] += r.e_smooth;
  }
  block_sum<6>(e, red, 128, 0);
  if (threadIdx.x == 0)
    for (int k = 0; k < 6; ++k) block_e[6 * blockIdx.x + k] = e[k];
  lf_grid_barrier(ticket, target += gridDim.x);
  if (blockIdx.x == 0 && threadIdx.x < 6) {  // fixed order: block 0, 1, 2, ...
    double acc = 0.0;
    for (unsigned blk = 0; blk < gridDim.x; ++blk) acc += block_e[6 * blk + threadIdx.x];
    b.e_out3[threadIdx.x / 3][threadIdx.x % 3] = acc;
  }
  for (int i = tid; i < 2 * nv; i += stride) {  // tilt gradients: one array per leaflet
    const int l = i >= nv, v = i - l * nv;
    double* out = b.tilt_grad[l];
    if (!out) continue;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
    for (int j = m0.csr_ptr[v]; j < m0.csr_ptr[v + 1]; ++j) {
      const double* q = b.tilt[l] + 3 * size_t(m0.csr_idx[j]);
      a0 += q[0];
      a1 += q[1];
      a2 += q[2];
    }
    double* o = out + 3 * size_t(v);
    o[0] = accumulate_tilt_grad ? o[0] + a0 : a0;
    o[1] = accumulate_tilt_grad ? o[1] + a1 : a1;
    o[2] = accumulate_tilt_grad ? o[2] + a2 : a2;
  }
  if (grad)
    for (int v = tid; v < nv; v += stride) {  // shape gradient: one array, inner leaflet first, outer on top
      double* o = grad + 3 * size_t(v);
      double g0 = accumulate_grad ? o[0] : 0.0, g1 = accumulate_grad ? o[1] : 0.0, g2 = accumulate_grad ? o[2] : 0.0;
      for (int l = 0; l < 2; ++l) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        for (int j = m0.csr_ptr[v]; j < m0.csr_ptr[v + 1]; ++j) {
          const double* q = b.shape[l] + 3 * size_t(m0.csr_idx[j]);
          a0 += q[0];
          a1 += q[1];
          a2 += q[2];
        }
        g0 = (l == 0 && !accumulate_grad) ? a0 : g0 + a0;
        g1 = (l == 0 && !accumulate_grad) ? a1 : g1 + a1;
        g2 = (l == 0 && !accumulate_grad) ? a2 : g2 + a2;
      }
      o[0] = g0;
      o[1] = g1;
      o[2] = g2;
    }
}

// ---- leaflet tilt relaxation helpers (runtime/steppers/tilt_relaxation.py:630-668,894-955) ----
// unit area-weighted vertex normals (Mesh.vertex_normals, geometry/triangle_ops.py:55-72): fixed-order gather
__global__ void __launch_bounds__(128) k_vertex_normals(int32_t nv, const int32_t* __restrict__ tri,
                                                        const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                        const double* __restrict__ pos, double* normals) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  d3 n = make_d3(0, 0, 0);
  for (int j = ptr[v]; j < ptr[v + 1]; ++j) {
    const int f = idx[j] / 3;
    const d3 a = ld3(pos, tri[3 * size_t(f)]), b = ld3(pos, tri[3 * size_t(f) + 1]), c = ld3(pos, tri[3 * size_t(f) + 2]);
    n = n + cross(b - a, c - a);
  }
  const double len = sqrt(dot(n, n));
  if (len >= 1.0e-12) n = (1.0 / len) * n;
  st3(normals, v, n);
}

// Evolver-style vertex averaging (ms_vertex_average.cuh): one thread per vertex over its corner list
__global__ void __launch_bounds__(128) k_vertex_average(const VaMesh m, double* __restrict__ out) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= m.nv) return;
  st3(out, v, va_vertex(m, v));
}

// --- equiangulation (ms_equiangulate.cuh): one thread per half-edge, sorted edge, or candidate ---
__global__ void __launch_bounds__(256) k_eq_keys(const EqMesh m, uint64_t* __restrict__ key, int32_t* __restrict__ h_out) {
  const int64_t h = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (h >= 3 * int64_t(m.nf)) return;
  key[h] = eq_key(m, eq_tail(m, h), eq_head(m, h));
  h_out[h] = int32_t(h);
}

__global__ void __launch_bounds__(256) k_eq_flag(const EqMesh m, uint8_t* __restrict__ flag) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= 3 * int64_t(m.nf)) return;
  int64_t h1 = 0, h2 = 0;
  flag[i] = eq_interior(m, i, h1, h2) && eq_should_flip(m, h1, h2);
}

__global__ void __launch_bounds__(256) k_eq_cands(const EqMesh m, int32_t nc, const int32_t* __restrict__ cand_pos,
                                                  int32_t* __restrict__ h1, int32_t* __restrict__ h2,
                                                  int32_t* __restrict__ slot_cand, uint64_t* __restrict__ nkey,
                                                  int32_t* __restrict__ id) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nc) return;
  const int32_t a = m.order[cand_pos[i]], b = m.order[cand_pos[i] + 1];
  h1[i] = a;
  h2[i] = b;
  slot_cand[a] = i;
  slot_cand[b] = i;
  nkey[i] = eq_key(m, eq_apex(m, a), eq_apex(m, b));
  id[i] = i;
}

__global__ void __launch_bounds__(256) k_eq_nkey_pos(int32_t nc, const int32_t* __restrict__ nkey_cand,
                                                     int32_t* __restrict__ nkey_pos) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nc) nkey_pos[nkey_cand[p]] = p;
}

// one Jacobi round; a round after the one that left no candidate undecided returns at once
__global__ void __launch_bounds__(256) k_eq_round(const EqCands s, const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                  const int32_t* __restrict__ prev_undecided, int32_t* undecided) {
  if (prev_undecided && *prev_undecided == 0) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint8_t st = i < s.n ? eq_round(s, in, i) : uint8_t(EQ_SELECTED);
  if (i < s.n) out[i] = st;
  const unsigned open = __ballot_sync(0xffffffffu, st == EQ_UNDECIDED);
  if (open && (threadIdx.x & 31) == 0) atomicAdd(undecided, __popc(open));
}

__global__ void __launch_bounds__(256) k_eq_apply(const EqCands s, const uint8_t* __restrict__ state, int32_t* tri,
                                                  int32_t* flips) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool sel = i < s.n && state[i] == EQ_SELECTED;
  if (sel) eq_apply(tri, s.h1[i], s.h2[i]);
  const unsigned mask = __ballot_sync(0xffffffffu, sel);
  if (mask && (threadIdx.x & 31) == 0) atomicAdd(flips, __popc(mask));
}

// --- refinement (ms_refine.cuh): one thread per sorted half-edge, vertex row or facet ---
__global__ void __launch_bounds__(256) k_rf_head_flags(const uint64_t* __restrict__ keys, int64_t n,
                                                       int32_t* __restrict__ flag) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = rf_head(keys, i);
}

// scan = inclusive sum of the head flags: sorted position i belongs to edge scan[i] - 1
__global__ void __launch_bounds__(256) k_rf_edges(const uint64_t* __restrict__ keys, const int32_t* __restrict__ order,
                                                  const int32_t* __restrict__ scan, int64_t n, int32_t* __restrict__ edge,
                                                  int32_t* __restrict__ head) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = scan[i] - 1;
  edge[order[i]] = e;
  if (rf_head(keys, i)) head[e] = int32_t(i);
  if (i == n - 1) head[e + 1] = int32_t(n);
}

// rows [0, nv): the old vertices; rows [nv, nv + n_edges): the midpoints
__global__ void __launch_bounds__(256) k_rf_vertices(const RfMesh r, const RfOut o) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < r.m.nv) rf_vertex(r, o, int32_t(i));
  else if (i < int64_t(r.m.nv) + r.n_edges) rf_midpoint(r, o, int32_t(i - r.m.nv));
}

__global__ void __launch_bounds__(256) k_rf_children(const RfMesh r, const RfOut o) {
  const int64_t f = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (f < r.m.nf) rf_children(r, o, int32_t(f));
}

// Bounding box of n positions: one box per block into boxes[1 + block], then boxes[0] from those (no atomics).
__device__ void rf_block_box(MortonBox b, MortonBox* out) {
  __shared__ MortonBox s[256];
  s[threadIdx.x] = b;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (int(threadIdx.x) < w) morton_box_merge(s[threadIdx.x], s[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = s[0];
}

__global__ void __launch_bounds__(256) k_rf_box_blocks(const double* __restrict__ pos, int64_t n, MortonBox* boxes) {
  MortonBox b = morton_box_empty();
  for (int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += int64_t(gridDim.x) * blockDim.x)
    morton_box_add(b, pos + 3 * v);
  rf_block_box(b, boxes + 1 + blockIdx.x);
}

__global__ void __launch_bounds__(256) k_rf_box_final(MortonBox* boxes, int n_blocks) {
  MortonBox b = morton_box_empty();
  for (int i = threadIdx.x; i < n_blocks; i += blockDim.x) morton_box_merge(b, boxes[1 + i]);
  rf_block_box(b, boxes);
}

__global__ void __launch_bounds__(256) k_rf_morton_keys(const double* __restrict__ pos, int64_t n,
                                                        const MortonBox* __restrict__ box, uint64_t* __restrict__ key,
                                                        int32_t* __restrict__ id) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= n) return;
  key[v] = morton_key(*box, pos + 3 * v);
  id[v] = int32_t(v);
}

__global__ void __launch_bounds__(256) k_rf_invert(const int32_t* __restrict__ perm, int64_t n, int32_t* __restrict__ inv) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) inv[perm[i]] = int32_t(i);
}

__global__ void __launch_bounds__(256) k_rf_renumber(const int32_t* __restrict__ rows, int64_t n,
                                                     const int32_t* __restrict__ inv, int32_t* __restrict__ out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = inv[rows[i]];
}

__global__ void __launch_bounds__(256) k_rf_gather_flags(const uint8_t* __restrict__ src, const int32_t* __restrict__ perm,
                                                         int64_t n, uint8_t* __restrict__ out, int32_t* __restrict__ out32) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t x = src[perm[i]];
  out[i] = x;
  if (out32) out32[i] = x ? 1 : 0;
}

// t -= (t.n) n  (runtime/projections/tilt.py:8-14)
__global__ void __launch_bounds__(256) k_project_tangent(int64_t nv, const double* __restrict__ normals, double* t) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const d3 n = ld3(normals, v), x = ld3(t, v);
  st3(t, v, axpy(-dot(x, n), n, x));
}

// trial = P(t - step g); rows with fixed tilts keep their value (projections/tilt.py:99-138)
__global__ void __launch_bounds__(256) k_tilt_trial(int64_t nv, const double* __restrict__ t, const double* __restrict__ g,
                                                    const double* __restrict__ normals, const uint8_t* __restrict__ fixed,
                                                    double step, double* trial) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const d3 x = ld3(t, v);
  if (fixed && fixed[v]) {
    st3(trial, v, x);
    return;
  }
  const d3 n = ld3(normals, v);
  const d3 y = axpy(-step, ld3(g, v), x);
  st3(trial, v, axpy(-dot(y, n), n, y));
}

// zero the gradient rows of fixed tilts; rowsq[v] = |g_v|^2 of the free rows (tilt_relaxation.py:856-871)
__global__ void __launch_bounds__(256) k_masked_row_norm2(int64_t nv, double* g, const uint8_t* __restrict__ fixed,
                                                          double* rowsq) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  if (fixed && fixed[v]) {
    st3(g, v, make_d3(0, 0, 0));
    rowsq[v] = 0.0;
    return;
  }
  const d3 x = ld3(g, v);
  rowsq[v] = dot(x, x);
}

// Jacobi preconditioner of the leaflet tilt CG (runtime/preconditioners.py:64-146): diag_v = k_tilt * barycentric
// area (facets of the leaflet when use_keep, else every facet) + 1/2 k_smooth * sum of the two opposite cotangents
// over every facet; diag <= 1e-12 and fixed rows -> 1; the inverse is stored.
__global__ void __launch_bounds__(128) k_leaflet_jacobi(LeafletMesh m, int use_keep, double k_smooth,
                                                        const uint8_t* __restrict__ fixed, double* minv) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= m.nv) return;
  double area = 0.0, cot = 0.0;
  for (int j = m.csr_ptr[v]; j < m.csr_ptr[v + 1]; ++j) {
    const int f = m.csr_idx[j] / 3, k = m.csr_idx[j] - 3 * f;
    int idx[3];
    if (!lf_facet_ok(m, f, idx)) continue;
    const FacetGeom g = facet_geom(lf_row(m.pos, idx[0]), lf_row(m.pos, idx[1]), lf_row(m.pos, idx[2]));
    if ((!use_keep || lf_kept(m, f)) && g.S >= kSurfaceSkip) area += 0.5 * g.S / 3.0;
    const CornerA c = facet_pass_a(g, false, false, false);
    cot += k == 0 ? c.c1 + c.c2 : (k == 1 ? c.c2 + c.c0 : c.c0 + c.c1);
  }
  double diag = m.k_tilt * area + 0.5 * k_smooth * cot;
  if (!(diag > 1.0e-12)) diag = 1.0;
  if (fixed && fixed[v]) diag = 1.0;
  minv[v] = 1.0 / diag;
}

// rows[v] = g_v . (minv_v g_v)  (the r.z of the preconditioned CG; minv == nullptr -> identity)
__global__ void __launch_bounds__(256) k_rz_rows(int64_t nv, const double* __restrict__ g, const double* __restrict__ minv,
                                                 double* rows) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const d3 x = ld3(g, v);
  rows[v] = dot(x, x) * (minv ? minv[v] : 1.0);
}

// dir = -minv g + beta dir   (restart: beta == 0 and the old direction is not read)
__global__ void __launch_bounds__(256) k_tilt_cg_direction(int64_t nv, const double* __restrict__ g,
                                                           const double* __restrict__ minv, double beta, int restart,
                                                           double* dir) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const d3 z = (minv ? -minv[v] : -1.0) * ld3(g, v);
  st3(dir, v, restart ? z : axpy(beta, ld3(dir, v), z));
}

// ---- halo exchange over NVLink peer memory ------------------------------------------------------------
// Every rank publishes "my owned rows of this array are written" by storing an epoch number into its flag
// word (k_halo_signal, stream-ordered after the producing kernel).  A consumer waits until every owner's flag
// has reached the epoch it expects and then copies its ghost rows straight out of the owners' arrays with
// peer loads (k_halo_pull): one kernel, no staging buffer, no host round trip.  The wait is bounded: after
// ~10 s (kWaitCycles) without the flag the kernel records an error instead of spinning forever.
__global__ void k_halo_signal(unsigned long long* flag, unsigned long long epoch) {
  __threadfence_system();
  *reinterpret_cast<volatile unsigned long long*>(flag) = epoch;
  __threadfence_system();
}

__device__ __forceinline__ void halo_wait_and_pull(int n_ghost, int width, const double* const* __restrict__ peer_base,
                                                   unsigned long long* const* __restrict__ peer_flag, int n_slots,
                                                   int flag_index, unsigned long long epoch,
                                                   const int32_t* __restrict__ owner, const int32_t* __restrict__ row,
                                                   double* dst, int* error) {
  __shared__ int ok;
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x) {
    if (!peer_flag[s] || !peer_base[s]) continue;  // only the owners of this rank's ghosts
    const volatile unsigned long long* f = peer_flag[s] + flag_index;
    const long long t0 = clock64();
    while (*f < epoch) {
      if (clock64() - t0 > kWaitCycles) {
        atomicExch(error, 1);
        ok = 0;
        break;
      }
      __nanosleep(200);
    }
  }
  __syncthreads();
  if (!ok) return;
  __threadfence_system();
  const int total = n_ghost * width;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int g = i / width, k = i - g * width;
    dst[i] = __ldcv(peer_base[owner[g]] + size_t(row[g]) * width + k);
  }
}

__global__ void __launch_bounds__(256) k_halo_pull(int n_ghost, int width, const double* const* __restrict__ peer_base,
                                                   unsigned long long* const* __restrict__ peer_flag, int n_slots,
                                                   int flag_index, unsigned long long epoch,
                                                   const int32_t* __restrict__ owner, const int32_t* __restrict__ row,
                                                   double* dst, int* error) {
  halo_wait_and_pull(n_ghost, width, peer_base, peer_flag, n_slots, flag_index, epoch, owner, row, dst, error);
}

// Signal and pull in ONE launch: block 0 raises this rank's flag (stream-ordered after the kernel that wrote the
// owned rows), every block then waits for the owners of the ghosts and copies.  Only for ranks that run
// concurrently (one process per GPU): contexts that share a stream would wait for a kernel queued behind them.
__global__ void __launch_bounds__(256) k_halo_exchange(unsigned long long* own_flag, int n_ghost, int width,
                                                       const double* const* __restrict__ peer_base,
                                                       unsigned long long* const* __restrict__ peer_flag, int n_slots,
                                                       int flag_index, unsigned long long epoch,
                                                       const int32_t* __restrict__ owner,
                                                       const int32_t* __restrict__ row, double* dst, int* error) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(own_flag) = epoch;
    __threadfence_system();
  }
  halo_wait_and_pull(n_ghost, width, peer_base, peer_flag, n_slots, flag_index, epoch, owner, row, dst, error);
}

// All-reduce (sum) of n <= 16 scalars over peer memory.  Word layout of every rank's exported block:
// [0..3] epoch flags, [8 + 16 p .. 8 + 16 p + 15] scalar slot of parity p.  Publish: copy this rank's scalars into
// the slot of the epoch's parity, then raise flag 2.  Gather: wait for every rank's flag, add the slots in RANK
// ORDER (the same order on every rank, so all ranks hold bitwise the same sums) and store them.  Two slots: a
// rank can publish epoch e+1 only after it has seen every flag of epoch e, and a peer can only lag behind reading
// epoch e, never e-1.
__global__ void k_allreduce_publish(const double* __restrict__ scalars, int n, unsigned long long* words,
                                    unsigned long long epoch) {
  double* slot = reinterpret_cast<double*>(words + 8 + 16 * (epoch & 1ull));
  if (int(threadIdx.x) < n) slot[threadIdx.x] = scalars[threadIdx.x];
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(words + 2) = epoch;
    __threadfence_system();
  }
}

__device__ __forceinline__ bool allreduce_gather(unsigned long long* const* __restrict__ peer_words, int n_slots, int n,
                                                 unsigned long long epoch, double* scalars, int* error) {
  __shared__ int ok;
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x) {
    const volatile unsigned long long* f = peer_words[s] + 2;
    const long long t0 = clock64();
    while (*f < epoch) {
      if (clock64() - t0 > kWaitCycles) {
        atomicExch(error, 1);
        ok = 0;
        break;
      }
      __nanosleep(200);
    }
  }
  __syncthreads();
  if (!ok) return false;
  __threadfence_system();
  if (int(threadIdx.x) < n) {
    double acc = 0.0;
    for (int s = 0; s < n_slots; ++s)
      acc += __ldcv(reinterpret_cast<const double*>(peer_words[s] + 8 + 16 * (epoch & 1ull)) + threadIdx.x);
    scalars[threadIdx.x] = acc;
  }
  return true;
}

__global__ void k_allreduce_gather(unsigned long long* const* __restrict__ peer_words, int n_slots, int n,
                                   unsigned long long epoch, double* scalars, int* error) {
  allreduce_gather(peer_words, n_slots, n, epoch, scalars, error);
}

// gather + the KKT coefficient from the GLOBAL sums (mode -2: energy-only evaluation, coefficient untouched)
__global__ void k_allreduce_gather_coef(unsigned long long* const* __restrict__ peer_words, int n_slots, int n,
                                        unsigned long long epoch, double* scalars, int mode, int has_gc, double k_vol,
                                        double v_target, int* error) {
  const bool ok = allreduce_gather(peer_words, n_slots, n, epoch, scalars, error);
  __syncthreads();
  if (ok && threadIdx.x == 0 && mode != -2) kkt_coefficient(scalars, mode, has_gc, k_vol, v_target);
}

__global__ void __launch_bounds__(256) k_row_norm2(const double* __restrict__ rows, int64_t n, double* out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = rows[3 * i], y = rows[3 * i + 1], z = rows[3 * i + 2];
  out[i] = x * x + y * y + z * z;
}

// ---- line-search helpers of the device-resident loop (runtime/steppers/line_search.py:267-541) ----
// minimum edge length squared over the facets (runtime/topology.py:174-199) and maximum row norm
// squared of the search direction; min / max are order independent, so atomics keep determinism.
__global__ void __launch_bounds__(256) k_min_edge2(const int32_t* __restrict__ tri, int32_t nf, int32_t nv,
                                                   const double* __restrict__ pos, unsigned long long* out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  double m = 1.0e300;
  if (f < nf) {
    const int i0 = tri[3 * size_t(f)], i1 = tri[3 * size_t(f) + 1], i2 = tri[3 * size_t(f) + 2];
    if (i0 >= 0 && i0 < nv && i1 >= 0 && i1 < nv && i2 >= 0 && i2 < nv) {
      const d3 a = ld3(pos, i0), b = ld3(pos, i1), c = ld3(pos, i2);
      const d3 e0 = c - b, e1 = a - c, e2 = b - a;
      m = fmin(dot(e0, e0), fmin(dot(e1, e1), dot(e2, e2)));
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmin(m, __shfl_down_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) atomicMin(out, (unsigned long long)__double_as_longlong(m));
}

__global__ void __launch_bounds__(256) k_max_row_norm2(const double* __restrict__ rows, int64_t n,
                                                       unsigned long long* out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  double m = 0.0;
  if (i < n) {
    const double x = rows[3 * i], y = rows[3 * i + 1], z = rows[3 * i + 2];
    m = x * x + y * y + z * z;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// flag |= 1 when a facet normal turns by more than acos(cos_limit) between `old_pos` and `new_pos`, or
// collapses (runtime/topology.py:13-48)
__global__ void __launch_bounds__(256) k_normal_change(const int32_t* __restrict__ tri, int32_t nf, int32_t nv,
                                                       const double* __restrict__ old_pos,
                                                       const double* __restrict__ new_pos, double cos_limit,
                                                       int* flag) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nf) return;
  const int i0 = tri[3 * size_t(f)], i1 = tri[3 * size_t(f) + 1], i2 = tri[3 * size_t(f) + 2];
  if (!(i0 >= 0 && i0 < nv && i1 >= 0 && i1 < nv && i2 >= 0 && i2 < nv)) return;
  const d3 a = ld3(old_pos, i0), b = ld3(old_pos, i1), c = ld3(old_pos, i2);
  const d3 n0 = cross(b - a, c - a);
  const double m0 = sqrt(dot(n0, n0));
  if (!(m0 > 1.0e-12)) return;  // facets that were degenerate before the step are not judged
  const d3 a1 = ld3(new_pos, i0), b1 = ld3(new_pos, i1), c1 = ld3(new_pos, i2);
  const d3 n1 = cross(b1 - a1, c1 - a1);
  const double m1 = sqrt(dot(n1, n1));
  bool bad = m1 < 1.0e-12;
  if (!bad) {
    // clamp without fmin / fmax, which would turn a NaN (a non-finite trial vertex) into a passing -1
    double d = dot(n0, n1) / (m0 * m1);
    if (d > 1.0) d = 1.0;
    if (d < -1.0) d = -1.0;
    bad = !(d >= cos_limit);
  }
  if (bad) atomicOr(flag, 1);
}

// Per-vertex Polak-Ribiere direction (runtime/steppers/conjugate_gradient.py:84-104):
//   beta_v = g_v.(g_v - g'_v) / (g'_v.g'_v + 1e-20);  d_v = -g_v + beta_v d'_v, or -g_v where beta_v < 0;
// fixed rows get a zero direction.  restart (device, may be null) set: d = -1 * g on every row, as launch_scale.
__global__ void __launch_bounds__(256) k_cg_direction(const double* __restrict__ g, const double* __restrict__ pg,
                                                      const double* __restrict__ pd,
                                                      const uint8_t* __restrict__ fixed, int64_t nv, double* d,
                                                      const int32_t* __restrict__ restart) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const double gx = g[3 * v], gy = g[3 * v + 1], gz = g[3 * v + 2];
  if (restart && *restart) {
    const double scale = -1.0;
    d[3 * v] = scale * gx; d[3 * v + 1] = scale * gy; d[3 * v + 2] = scale * gz;
    return;
  }
  const double px = pg[3 * v], py = pg[3 * v + 1], pz = pg[3 * v + 2];
  const double numer = gx * (gx - px) + gy * (gy - py) + gz * (gz - pz);
  const double denom = (px * px + py * py + pz * pz) + 1.0e-20;
  const double beta = numer / denom;
  double dx = -gx, dy = -gy, dz = -gz;
  if (!(beta < 0.0)) {
    dx += beta * pd[3 * v]; dy += beta * pd[3 * v + 1]; dz += beta * pd[3 * v + 2];
  }
  if (fixed && fixed[v]) dx = dy = dz = 0.0;
  d[3 * v] = dx; d[3 * v + 1] = dy; d[3 * v + 2] = dz;
}

// y[v,:] += alpha * x[v,:] on the rows that are not fixed (constraint projection of the positions).  x may be y
// (ms_ctx_axpy with dst == src), so it is not __restrict__; each thread reads and writes only its own element.
__global__ void __launch_bounds__(256) k_axpy_rows(const double* x, double alpha, const double* __restrict__ alpha_dev,
                                                   const uint8_t* __restrict__ fixed, int64_t nv, double* y) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= 3 * nv) return;
  if (alpha_dev) alpha = *alpha_dev;
  if (fixed && fixed[i / 3]) return;
  y[i] += alpha * x[i];
}

__global__ void __launch_bounds__(256) k_scale(const double* __restrict__ x, double scale, double* out, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = scale * x[i];
}

inline int blocks_for(int64_t n, int t) { return int((n + t - 1) / t); }

}  // namespace

namespace {
int g_num_sms = 0;

// compile-time kernel kind of a launch (see k_patch)
int kernel_kind(const PatchLaunch& a) {
  const bool diag = a.k_vecs || a.a_vor || a.a_eff || a.e_vertex;
  if (a.modules == kFastModules && a.flags == 0 && !a.is_boundary && !a.slot_gamma && !a.kappa && !a.c0 && !diag &&
      a.seeds && a.volgrad)
    return 1;
  if ((a.modules & ~uint32_t(MS_MOD_SURFACE | MS_MOD_VOLUME)) == 0 && a.modules != 0 && !a.slot_gamma && !diag &&
      a.volgrad)
    return 2;
  if (!(a.modules & MS_MOD_TILT) && (a.modules & MS_MOD_BENDING) && a.seeds) return 3;  // run-time parameters, no tilt
  return 0;
}

template <int PASS>
size_t patch_smem_bytes(const PatchLaunch& a) {
  if (kernel_kind(a) == 1 || kernel_kind(a) == 2) return Plan<PASS>::oOpt;
  const bool tilt = (a.modules & MS_MOD_TILT) && a.tilts;
  return Plan<PASS>::oOpt + opt_bytes(a.is_boundary != nullptr, tilt, tilt && PASS == 1);
}

}  // namespace

size_t pass_a_smem_bytes(const PatchLaunch& a) { return patch_smem_bytes<0>(a); }
size_t pass_b_smem_bytes(const PatchLaunch& a) { return patch_smem_bytes<1>(a); }

cudaError_t configure_kernels() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const int max_dyn = 227 * 1024;
  const void* fns[] = {(const void*)k_patch<0, 0, kConsumerThreads>, (const void*)k_patch<0, 1, kConsumerThreads>,
                       (const void*)k_patch<0, 2, kConsumerThreads>, (const void*)k_patch<1, 0, kConsumerThreads>,
                       (const void*)k_patch<1, 1, kConsumerThreads>, (const void*)k_patch<1, 2, kConsumerThreads>,
                       (const void*)k_patch<0, 3, kConsumerThreads>, (const void*)k_patch<1, 3, kConsumerThreads>};
  for (const void* f : fns) {
    cudaFuncAttributes attr;
    e = cudaFuncGetAttributes(&attr, f);
    if (e != cudaSuccess) return e;
    // static (finalisation scratch) + dynamic shared memory share the 227 KB a CTA may opt in to
    e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn - int(attr.sharedSizeBytes));
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

int patch_grid(const PatchLaunch& a) {
  int sms = g_num_sms > 0 ? g_num_sms : 148;
  if (a.max_ctas > 0 && a.max_ctas < sms) sms = a.max_ctas;
  return a.patch_count < sms ? a.patch_count : sms;
}

cudaError_t launch_pass_a(const PatchLaunch& a, cudaStream_t st) {
  if (a.patch_count <= 0) return cudaSuccess;
  const size_t smem = patch_smem_bytes<0>(a);
  const int grid = patch_grid(a);
  switch (kernel_kind(a)) {
    case 1: k_patch<0, 1, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, true, false); break;
    case 2: k_patch<0, 2, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, false, false); break;
    case 3: k_patch<0, 3, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, false, false); break;
    default: k_patch<0, 0, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, false, false);
  }
  return cudaGetLastError();
}

cudaError_t launch_pass_b(const PatchLaunch& a, bool bending, bool scalars_here, cudaStream_t st) {
  if (a.patch_count <= 0) return cudaSuccess;
  const size_t smem = patch_smem_bytes<1>(a);
  const int grid = patch_grid(a);
  const int kind = kernel_kind(a);
  if (kind == 1 && bending && !scalars_here)
    k_patch<1, 1, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, true, false);
  else if (kind == 2 && !bending)
    k_patch<1, 2, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, false, scalars_here);
  else if (kind == 3 && bending && !scalars_here)
    k_patch<1, 3, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, bending, scalars_here);
  else
    k_patch<1, 0, kConsumerThreads><<<grid, kConsumerThreads + 64, smem, st>>>(a, bending, scalars_here);
  return cudaGetLastError();
}

cudaError_t launch_reduce_partials(const double* pa, int rows_a, const double* pb, int rows_b, unsigned b_mask,
                                   double* scalars, cudaStream_t st) {
  k_reduce_partials<<<1, kReduceRows * kPartialStride, 0, st>>>(pa, rows_a, pb, rows_b, b_mask, scalars);
  return cudaGetLastError();
}

cudaError_t launch_dots(const double* g, const double* gc, int64_t n, double* block_partials,
                        int n_blocks, double* scalars, cudaStream_t st) {
  k_dots<<<n_blocks, 256, 0, st>>>(g, gc, n, block_partials);
  k_dots_final<<<1, 256, 0, st>>>(block_partials, n_blocks, scalars);
  return cudaGetLastError();
}

cudaError_t launch_project(double* g, const double* gc, const uint8_t* fixed, int64_t nv,
                           double* scalars, int mode, double k_vol, double v_target,
                           cudaStream_t st) {
  if (nv <= 0) return cudaSuccess;
  k_project<<<blocks_for(3 * nv, 256), 256, 0, st>>>(g, gc, fixed, nv, scalars, mode, k_vol, v_target);
  return cudaGetLastError();
}

cudaError_t launch_kkt_coefficient(double* scalars, int mode, int has_gc, double k_vol, double v_target, cudaStream_t st) {
  k_kkt_coefficient<<<1, 1, 0, st>>>(scalars, mode, has_gc, k_vol, v_target);
  return cudaGetLastError();
}

cudaError_t launch_apply_projection(double* g, const double* gc, const uint8_t* fixed, int64_t nv, const double* scalars,
                                    cudaStream_t st) {
  if (nv <= 0) return cudaSuccess;
  k_apply_projection<<<blocks_for(3 * nv, 256), 256, 0, st>>>(g, gc, fixed, nv, scalars);
  return cudaGetLastError();
}

cudaError_t launch_scale_projected(const double* g, const double* gc, const uint8_t* fixed, int64_t nv,
                                   const double* scalars, double scale, double* out, cudaStream_t st) {
  if (nv <= 0) return cudaSuccess;
  k_scale_projected<<<blocks_for(3 * nv, 256), 256, 0, st>>>(g, gc, fixed, nv, scalars, scale, out);
  return cudaGetLastError();
}

cudaError_t launch_dots_projected(const double* g, const double* gc, const uint8_t* fixed, const double* d, int64_t nv,
                                  double* block_partials, int n_blocks, double* scalars, cudaStream_t st) {
  k_dots_projected<<<n_blocks, 256, 0, st>>>(g, gc, fixed, d, 3 * nv, scalars, block_partials);
  k_dots_final<<<1, 256, 0, st>>>(block_partials, n_blocks, scalars);
  return cudaGetLastError();
}

cudaError_t launch_gather_rows(const double* src, int width, const int32_t* rows, int64_t n,
                               double* out, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  k_gather_rows<<<blocks_for(n * width, 256), 256, 0, st>>>(src, width, rows, n, out);
  return cudaGetLastError();
}

cudaError_t launch_scatter_rows(const double* src, int width, const int32_t* rows, int64_t n,
                                double* out, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  k_scatter_rows<<<blocks_for(n * width, 256), 256, 0, st>>>(src, width, rows, n, out);
  return cudaGetLastError();
}

cudaError_t launch_axpy(const double* x, const double* d, double alpha, double* out, int64_t n,
                        cudaStream_t st, const double* alpha_dev) {
  if (n <= 0) return cudaSuccess;
  k_axpy<<<blocks_for(n, 256), 256, 0, st>>>(x, d, alpha, alpha_dev, out, n);
  return cudaGetLastError();
}

cudaError_t launch_soup_surface(const SoupArgs& s, const double* gamma, double* corner,
                                double* facet_e, double* grad, double* energy_out,
                                cudaStream_t st) {
  if (s.nf > 0) k_soup_surface<<<blocks_for(s.nf, 128), 128, 0, st>>>(s, gamma, corner, facet_e);
  if (s.nv > 0 && s.nf > 0)
    k_gather<<<blocks_for(s.nv, 128), 128, 0, st>>>(s.nv, s.csr_ptr, s.csr_idx, corner, 3, 0, 3, grad, 3, 1);
  k_sum<<<1, 256, 0, st>>>(facet_e, s.nf, 1.0, energy_out);
  return cudaGetLastError();
}

cudaError_t launch_soup_volume(const SoupArgs& s, double factor, double* corner, double* facet_v,
                               double* grad, double* volume_out, cudaStream_t st) {
  if (s.nf > 0) k_soup_volume<<<blocks_for(s.nf, 128), 128, 0, st>>>(s, factor, corner, facet_v);
  if (s.nv > 0 && s.nf > 0 && grad)
    k_gather<<<blocks_for(s.nv, 128), 128, 0, st>>>(s.nv, s.csr_ptr, s.csr_idx, corner, 3, 0, 3, grad, 3, 1);
  k_sum<<<1, 256, 0, st>>>(facet_v, s.nf, 1.0 / 6.0, volume_out);
  return cudaGetLastError();
}

cudaError_t launch_soup_curvature(const SoupArgs& s, double* corner, double* k_vecs,
                                  double* vertex_areas, double* weights, double* va0, double* va1,
                                  double* va2, cudaStream_t st) {
  if (s.nf > 0) k_soup_curvature<<<blocks_for(s.nf, 128), 128, 0, st>>>(s, corner, weights, va0, va1, va2);
  if (s.nv > 0) {
    // with nf == 0 every CSR range is empty and the gathers write zeros
    k_gather<<<blocks_for(s.nv, 128), 128, 0, st>>>(s.nv, s.csr_ptr, s.csr_idx, corner, 4, 0, 3, k_vecs, 3, 0);
    k_gather<<<blocks_for(s.nv, 128), 128, 0, st>>>(s.nv, s.csr_ptr, s.csr_idx, corner, 4, 3, 1, vertex_areas, 1, 0);
  }
  return cudaGetLastError();
}

cudaError_t launch_soup_laplacian(const SoupArgs& s, int32_t dim, const double* weights,
                                  const double* field, double* corner, double* out,
                                  cudaStream_t st) {
  if (s.nf > 0) k_soup_laplacian<<<blocks_for(s.nf, 128), 128, 0, st>>>(s, dim, weights, field, corner);
  if (s.nv > 0)
    k_gather<<<blocks_for(s.nv, 128), 128, 0, st>>>(s.nv, s.csr_ptr, s.csr_idx, corner, dim, 0, dim, out, dim, 0);
  return cudaGetLastError();
}

cudaError_t launch_grad_cotan(int32_t n, const double* u, const double* v, double* gu, double* gv,
                              cudaStream_t st) {
  if (n > 0) k_grad_cotan<<<blocks_for(n, 128), 128, 0, st>>>(n, u, v, gu, gv);
  return cudaGetLastError();
}

cudaError_t launch_p1_divergence(const SoupArgs& s, const double* tilts, double* div, double* area,
                                 double* g0, double* g1, double* g2, cudaStream_t st) {
  if (s.nf > 0) k_p1_divergence<<<blocks_for(s.nf, 128), 128, 0, st>>>(s, tilts, div, area, g0, g1, g2);
  return cudaGetLastError();
}

cudaError_t launch_p1_vertex_divergence(const SoupArgs& s, const double* div, const double* area, double* div_v,
                                       double* area_v, cudaStream_t st) {
  if (s.nv > 0) k_p1_vertex_divergence<<<blocks_for(s.nv, 128), 128, 0, st>>>(s, div, area, div_v, area_v);
  return cudaGetLastError();
}

cudaError_t launch_row_norm2(const double* rows, int64_t n, double* out, cudaStream_t st) {
  if (n > 0) k_row_norm2<<<blocks_for(n, 256), 256, 0, st>>>(rows, n, out);
  return cudaGetLastError();
}

cudaError_t launch_sum(const double* x, int64_t n, double scale, double* out, cudaStream_t st) {
  k_sum<<<1, 256, 0, st>>>(x, n, scale, out);
  return cudaGetLastError();
}

// sum of x[0..n) * scale -> *out; scratch holds kSumBlocks doubles (used for long arrays only)
static void sum_fixed_order(const double* x, int64_t n, double scale, double* out, double* scratch, cudaStream_t st) {
  if (n < (int64_t(1) << 16)) {
    k_sum<<<1, 256, 0, st>>>(x, n, scale, out);
  } else {
    k_sum_partial<<<kSumBlocks, 256, 0, st>>>(x, n, scratch);
    k_sum<<<1, 256, 0, st>>>(scratch, kSumBlocks, scale, out);
  }
}

cudaError_t launch_bt_stage(const BtMesh& m, double sign, const double* k_vecs, const double* a_vor,
                            const double* a_eff, double* corner /* 12*nf doubles */, double* seeds, double* base,
                            double* facet_e, double* e_out, bool tilt_grads, cudaStream_t st) {
  if (m.nf > 0) k_bt_facet_a<<<blocks_for(m.nf, 128), 128, 0, st>>>(m, sign, corner);
  if (m.nv > 0) k_bt_vertex<<<blocks_for(m.nv, 128), 128, 0, st>>>(m, k_vecs, a_vor, a_eff, corner, seeds, base);
  // the corner buffer is free again: it now receives the tilt-gradient contributions (9 per facet)
  if (m.nf > 0) k_bt_facet_b<<<blocks_for(m.nf, 128), 128, 0, st>>>(m, base, sign, tilt_grads ? corner : nullptr, facet_e);
  sum_fixed_order(facet_e, m.nf, 1.0, e_out, e_out + 1, st);
  return cudaGetLastError();
}

cudaError_t launch_bt_tilt_gather(const BtMesh& m, const double* corner3, double* tilt_grad, bool accumulate,
                                  cudaStream_t st) {
  if (m.nv > 0)
    k_gather<<<blocks_for(m.nv, 128), 128, 0, st>>>(m.nv, m.csr_ptr, m.csr_idx, corner3, 3, 0, 3, tilt_grad, 3,
                                                     accumulate ? 1 : 0);
  return cudaGetLastError();
}

cudaError_t launch_bt_finalize(const double* e_bt, double* scalars, cudaStream_t st) {
  k_bt_finalize<<<1, 1, 0, st>>>(e_bt, scalars);
  return cudaGetLastError();
}

cudaError_t launch_leaflet(const LeafletMesh& m, bool with_bt, bool with_tilt, bool with_smooth, double* corner,
                           double* vbuf, double* corner_shape, double* corner_tilt, double* facet_e, double* e_out3,
                           double* sum_scratch, double* grad,
                           bool accumulate_grad, double* tilt_grad, bool accumulate_tilt_grad, cudaStream_t st) {
  if (with_bt) {
    if (m.nf > 0) k_lf_facet_a<<<blocks_for(m.nf, 128), 128, 0, st>>>(m, corner);
    if (m.nv > 0) k_lf_vertex<<<blocks_for(m.nv, 128), 128, 0, st>>>(m, corner, vbuf);
  }
  if (m.nf > 0)
    k_lf_facet_b<<<blocks_for(m.nf, 128), 128, 0, st>>>(m, vbuf, with_bt ? 1 : 0, with_tilt ? 1 : 0, with_smooth ? 1 : 0,
                                                        grad ? corner_shape : nullptr, tilt_grad ? corner_tilt : nullptr,
                                                        facet_e);
  for (int k = 0; k < 3; ++k)
    sum_fixed_order(facet_e + k * size_t(m.nf), m.nf, 1.0, e_out3 + k, sum_scratch + k * kSumBlocks, st);
  if (m.nv > 0 && grad)
    k_gather<<<blocks_for(m.nv, 128), 128, 0, st>>>(m.nv, m.csr_ptr, m.csr_idx, corner_shape, 3, 0, 3, grad, 3,
                                                     accumulate_grad ? 1 : 0);
  if (m.nv > 0 && tilt_grad)
    k_gather<<<blocks_for(m.nv, 128), 128, 0, st>>>(m.nv, m.csr_ptr, m.csr_idx, corner_tilt, 3, 0, 3, tilt_grad, 3,
                                                     accumulate_tilt_grad ? 1 : 0);
  return cudaGetLastError();
}

// Cooperative single-launch variant for small meshes.  Returns cudaErrorNotSupported when the device cannot launch
// cooperatively or the grid would not be resident; the caller then uses launch_leaflet.  *ticket_base is the
// host-side mirror of the ticket counter (advanced by the barriers this launch performs).
cudaError_t launch_leaflet_fused(const LeafletMesh& m, bool with_bt, bool with_tilt, bool with_smooth, double* corner,
                                 double* vbuf, double* corner_shape, double* corner_tilt, double* block_e, int max_blocks,
                                 double* e_out3, double* grad, bool accumulate_grad, double* tilt_grad,
                                 bool accumulate_tilt_grad, unsigned long long* ticket, unsigned long long* ticket_base,
                                 cudaStream_t st) {
  static int resident = -1;
  if (resident < 0) {
    int dev = 0, coop = 0, per_sm = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lf_fused, 128, 0);
    resident = coop ? per_sm * sms : 0;
  }
  int blocks = blocks_for(m.nf > m.nv ? m.nf : m.nv, 128);
  if (blocks > max_blocks) blocks = max_blocks;
  if (blocks > resident) blocks = resident;
  if (blocks <= 0) return cudaErrorNotSupported;
  LeafletMesh mm = m;
  int bt = with_bt ? 1 : 0, tl = with_tilt ? 1 : 0, sm = with_smooth ? 1 : 0, ag = accumulate_grad ? 1 : 0,
      at = accumulate_tilt_grad ? 1 : 0;
  unsigned long long base = *ticket_base;
  void* args[] = {&mm, &bt, &tl, &sm, &corner, &vbuf, &corner_shape, &corner_tilt, &block_e, &e_out3, &grad, &ag,
                  &tilt_grad, &at, &ticket, &base};
  cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_lf_fused), dim3(blocks), dim3(128), args, 0, st);
  if (e == cudaSuccess) *ticket_base = base + (unsigned long long)(blocks) * (with_bt ? 3ull : 1ull);
  return e;
}

// Inner and outer leaflet of a small mesh in one cooperative launch (see k_lf_fused_pair); the arrays of index 0
// belong to m0, of index 1 to m1.  cudaErrorNotSupported -> evaluate the leaflets one after the other.
cudaError_t launch_leaflet_fused_pair(const LeafletMesh& m0, const LeafletMesh& m1, bool with_bt, bool with_tilt,
                                      bool with_smooth, double* const corner[2], double* const vbuf[2],
                                      double* const shape[2], double* const tilt[2], double* const e_out3[2],
                                      double* const tilt_grad[2], double* block_e, int max_blocks, double* grad,
                                      bool accumulate_grad, bool accumulate_tilt_grad, unsigned long long* ticket,
                                      unsigned long long* ticket_base, cudaStream_t st) {
  static int resident = -1;
  if (resident < 0) {
    int dev = 0, coop = 0, per_sm = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lf_fused_pair, 128, 0);
    resident = coop ? per_sm * sms : 0;
  }
  int blocks = blocks_for(2 * int64_t(m0.nf > m0.nv ? m0.nf : m0.nv), 128);
  if (blocks > max_blocks) blocks = max_blocks;
  if (blocks > resident) blocks = resident;
  if (blocks <= 0) return cudaErrorNotSupported;
  LeafletMesh a = m0, b = m1;
  LfPairBuffers buf;
  for (int l = 0; l < 2; ++l) {
    buf.corner[l] = corner[l];
    buf.vbuf[l] = vbuf[l];
    buf.shape[l] = shape[l];
    buf.tilt[l] = tilt[l];
    buf.e_out3[l] = e_out3[l];
    buf.tilt_grad[l] = tilt_grad[l];
  }
  int bt = with_bt ? 1 : 0, tl = with_tilt ? 1 : 0, sm = with_smooth ? 1 : 0, ag = accumulate_grad ? 1 : 0,
      at = accumulate_tilt_grad ? 1 : 0;
  unsigned long long base = *ticket_base;
  void* args[] = {&a, &b, &buf, &bt, &tl, &sm, &block_e, &grad, &ag, &at, &ticket, &base};
  cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_lf_fused_pair), dim3(blocks), dim3(128), args, 0, st);
  if (e == cudaSuccess) *ticket_base = base + (unsigned long long)(blocks) * (with_bt ? 3ull : 1ull);
  return e;
}

cudaError_t launch_vertex_normals(int32_t nv, const int32_t* tri, const int32_t* csr_ptr, const int32_t* csr_idx,
                                  const double* pos, double* normals, cudaStream_t st) {
  if (nv > 0) k_vertex_normals<<<blocks_for(nv, 128), 128, 0, st>>>(nv, tri, csr_ptr, csr_idx, pos, normals);
  return cudaGetLastError();
}

cudaError_t launch_vertex_average(const VaMesh& m, double* out, cudaStream_t st) {
  if (m.nv > 0) k_vertex_average<<<blocks_for(m.nv, 128), 128, 0, st>>>(m, out);
  return cudaGetLastError();
}

int eq_key_bits(int32_t nv) {
  const uint64_t top = nv > 1 ? uint64_t(nv) * uint64_t(nv) - 1 : 1;
  int bits = 0;
  while (bits < 64 && (top >> bits)) ++bits;
  return bits;
}

cudaError_t eq_temp_bytes(int64_t n_half_edges, size_t* bytes) {
  size_t a = 0, b = 0;
  const int n = int(n_half_edges);
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                                  (const int32_t*)nullptr, (int32_t*)nullptr, n);
  if (e != cudaSuccess) return e;
  e = cub::DeviceSelect::Flagged(nullptr, b, cub::CountingInputIterator<int32_t>(0), (const uint8_t*)nullptr,
                                 (int32_t*)nullptr, (int32_t*)nullptr, n);
  *bytes = a > b ? a : b;
  return e;
}

cudaError_t launch_eq_sort_edges(const EqMesh& m, uint64_t* key_in, int32_t* h_in, uint64_t* keys, int32_t* order,
                                 void* temp, size_t temp_bytes, cudaStream_t st) {
  const int64_t n = 3 * int64_t(m.nf);
  if (n == 0) return cudaSuccess;
  k_eq_keys<<<blocks_for(n, 256), 256, 0, st>>>(m, key_in, h_in);
  if (cudaError_t e = cudaGetLastError()) return e;
  return cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_in, keys, h_in, order, int(n), 0, eq_key_bits(m.nv), st);
}

cudaError_t launch_eq_candidates(const EqMesh& m, uint8_t* flag, int32_t* cand_pos, int32_t* n_cand, void* temp,
                                 size_t temp_bytes, cudaStream_t st) {
  const int64_t n = 3 * int64_t(m.nf);
  if (n == 0) return cudaMemsetAsync(n_cand, 0, sizeof(int32_t), st);
  k_eq_flag<<<blocks_for(n, 256), 256, 0, st>>>(m, flag);
  if (cudaError_t e = cudaGetLastError()) return e;
  return cub::DeviceSelect::Flagged(temp, temp_bytes, cub::CountingInputIterator<int32_t>(0), flag, cand_pos, n_cand,
                                    int(n), st);
}

cudaError_t launch_eq_conflicts(const EqMesh& m, int32_t nc, const int32_t* cand_pos, const EqCands& s,
                                uint64_t* nkey_in, int32_t* id_in, void* temp, size_t temp_bytes, cudaStream_t st) {
  if (cudaError_t e = cudaMemsetAsync(const_cast<int32_t*>(s.slot_cand), 0xff, 3 * size_t(m.nf) * sizeof(int32_t), st)) return e;
  if (nc == 0) return cudaSuccess;
  k_eq_cands<<<blocks_for(nc, 256), 256, 0, st>>>(m, nc, cand_pos, const_cast<int32_t*>(s.h1), const_cast<int32_t*>(s.h2),
                                                  const_cast<int32_t*>(s.slot_cand), nkey_in, id_in);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, nkey_in, const_cast<uint64_t*>(s.nkey), id_in,
                                                      const_cast<int32_t*>(s.nkey_cand), nc, 0, eq_key_bits(m.nv), st))
    return e;
  k_eq_nkey_pos<<<blocks_for(nc, 256), 256, 0, st>>>(nc, s.nkey_cand, const_cast<int32_t*>(s.nkey_pos));
  return cudaGetLastError();
}

cudaError_t launch_eq_round(const EqCands& s, const uint8_t* in, uint8_t* out, const int32_t* prev_undecided,
                            int32_t* undecided, cudaStream_t st) {
  if (s.n > 0) k_eq_round<<<blocks_for(s.n, 256), 256, 0, st>>>(s, in, out, prev_undecided, undecided);
  return cudaGetLastError();
}

cudaError_t launch_eq_apply(const EqCands& s, const uint8_t* state, int32_t* tri, int32_t* flips, cudaStream_t st) {
  if (s.n > 0) k_eq_apply<<<blocks_for(s.n, 256), 256, 0, st>>>(s, state, tri, flips);
  return cudaGetLastError();
}

cudaError_t rf_temp_bytes(int64_t n, size_t* bytes) {
  size_t a = 0, b = 0;
  if (cudaError_t e = eq_temp_bytes(n, &a)) return e;
  cudaError_t e = cub::DeviceScan::InclusiveSum(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, int(n));
  *bytes = std::max(a, b);
  return e;
}

cudaError_t launch_rf_edges(const EqMesh& m, int32_t* flag, int32_t* scan, int32_t* edge, int32_t* head, void* temp,
                            size_t temp_bytes, cudaStream_t st) {
  const int64_t n = 3 * int64_t(m.nf);
  if (n == 0) return cudaSuccess;
  k_rf_head_flags<<<blocks_for(n, 256), 256, 0, st>>>(m.keys, n, flag);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (cudaError_t e = cub::DeviceScan::InclusiveSum(temp, temp_bytes, flag, scan, int(n), st)) return e;
  k_rf_edges<<<blocks_for(n, 256), 256, 0, st>>>(m.keys, m.order, scan, n, edge, head);
  return cudaGetLastError();
}

cudaError_t launch_rf_build(const RfMesh& r, const RfOut& o, cudaStream_t st) {
  const int64_t nv_out = int64_t(r.m.nv) + r.n_edges;
  if (nv_out > 0) k_rf_vertices<<<blocks_for(nv_out, 256), 256, 0, st>>>(r, o);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (r.m.nf > 0) k_rf_children<<<blocks_for(r.m.nf, 256), 256, 0, st>>>(r, o);
  return cudaGetLastError();
}

cudaError_t launch_rf_morton(const double* pos, int32_t n, MortonBox* boxes, uint64_t* key_in, int32_t* id_in,
                             uint64_t* key_out, int32_t* perm, int32_t* inv, void* temp, size_t temp_bytes,
                             cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  const int nb = std::min(kRfBoxBlocks, blocks_for(n, 256));
  k_rf_box_blocks<<<nb, 256, 0, st>>>(pos, n, boxes);
  k_rf_box_final<<<1, 256, 0, st>>>(boxes, nb);
  k_rf_morton_keys<<<blocks_for(n, 256), 256, 0, st>>>(pos, n, boxes, key_in, id_in);
  if (cudaError_t e = cudaGetLastError()) return e;
  // 3 x 21 key bits; the radix sort is stable, so equal keys keep ascending ids, as std::stable_sort orders them
  if (cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_in, key_out, id_in, perm, n, 0, 63, st)) return e;
  k_rf_invert<<<blocks_for(n, 256), 256, 0, st>>>(perm, n, inv);
  return cudaGetLastError();
}

cudaError_t launch_rf_renumber(const int32_t* rows, int64_t n, const int32_t* inv, int32_t* out, cudaStream_t st) {
  if (n > 0) k_rf_renumber<<<blocks_for(n, 256), 256, 0, st>>>(rows, n, inv, out);
  return cudaGetLastError();
}

cudaError_t launch_rf_gather_flags(const uint8_t* src, const int32_t* perm, int64_t n, uint8_t* out, int32_t* out32,
                                   cudaStream_t st) {
  if (n > 0) k_rf_gather_flags<<<blocks_for(n, 256), 256, 0, st>>>(src, perm, n, out, out32);
  return cudaGetLastError();
}

cudaError_t launch_project_tangent(int64_t nv, const double* normals, double* t, cudaStream_t st) {
  if (nv > 0) k_project_tangent<<<blocks_for(nv, 256), 256, 0, st>>>(nv, normals, t);
  return cudaGetLastError();
}

cudaError_t launch_tilt_trial(int64_t nv, const double* t, const double* g, const double* normals, const uint8_t* fixed,
                              double step, double* trial, cudaStream_t st) {
  if (nv > 0) k_tilt_trial<<<blocks_for(nv, 256), 256, 0, st>>>(nv, t, g, normals, fixed, step, trial);
  return cudaGetLastError();
}

cudaError_t launch_masked_norm2(int64_t nv, double* g, const uint8_t* fixed, double* rowsq, double* out,
                                double* sum_scratch /* kSumBlocks */, cudaStream_t st) {
  if (nv > 0) k_masked_row_norm2<<<blocks_for(nv, 256), 256, 0, st>>>(nv, g, fixed, rowsq);
  sum_fixed_order(rowsq, nv, 1.0, out, sum_scratch, st);
  return cudaGetLastError();
}

cudaError_t launch_leaflet_jacobi(const LeafletMesh& m, bool use_keep, double k_smooth, const uint8_t* fixed, double* minv,
                                  cudaStream_t st) {
  if (m.nv > 0) k_leaflet_jacobi<<<blocks_for(m.nv, 128), 128, 0, st>>>(m, use_keep ? 1 : 0, k_smooth, fixed, minv);
  return cudaGetLastError();
}

cudaError_t launch_rz(int64_t nv, const double* g, const double* minv, double* rows, double* out,
                      double* sum_scratch /* kSumBlocks */, cudaStream_t st) {
  if (nv > 0) k_rz_rows<<<blocks_for(nv, 256), 256, 0, st>>>(nv, g, minv, rows);
  sum_fixed_order(rows, nv, 1.0, out, sum_scratch, st);
  return cudaGetLastError();
}

cudaError_t launch_tilt_cg_direction(int64_t nv, const double* g, const double* minv, double beta, bool restart, double* dir,
                                     cudaStream_t st) {
  if (nv > 0) k_tilt_cg_direction<<<blocks_for(nv, 256), 256, 0, st>>>(nv, g, minv, beta, restart ? 1 : 0, dir);
  return cudaGetLastError();
}

cudaError_t launch_halo_signal(unsigned long long* flag, unsigned long long epoch, cudaStream_t st) {
  k_halo_signal<<<1, 1, 0, st>>>(flag, epoch);
  return cudaGetLastError();
}

cudaError_t launch_halo_pull(int n_ghost, int width, const double* const* peer_base, unsigned long long* const* peer_flag,
                             int n_slots, int flag_index, unsigned long long epoch, const int32_t* owner,
                             const int32_t* row, double* dst, int* error, cudaStream_t st) {
  if (n_ghost <= 0) return cudaSuccess;
  const int blocks = (n_ghost * width + 255) / 256;
  k_halo_pull<<<blocks < 64 ? blocks : 64, 256, 0, st>>>(n_ghost, width, peer_base, peer_flag, n_slots, flag_index, epoch,
                                                          owner, row, dst, error);
  return cudaGetLastError();
}

// ---- push transport --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_halo_push(int n_rows, int width, const double* __restrict__ src,
                                                   double* const* __restrict__ peer_base,
                                                   const int32_t* __restrict__ dst_slot, const int32_t* __restrict__ src_row,
                                                   const int32_t* __restrict__ dst_row,
                                                   unsigned long long* const* __restrict__ peer_flags, int n_slots,
                                                   uint64_t dst_mask, int my_slot, int kind, unsigned long long epoch,
                                                   unsigned int* ticket) {
  const int total = n_rows * width;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int g = i / width, k = i - g * width;
    peer_base[dst_slot[g]][size_t(dst_row[g]) * width + k] = src[size_t(src_row[g]) * width + k];
  }
  __threadfence_system();
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  __threadfence_system();
  if (threadIdx.x == 0) *ticket = 0u;
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x)
    if ((dst_mask >> s) & 1ull) {
      *reinterpret_cast<volatile unsigned long long*>(peer_flags[s] + kPushFlagBase + 64 * kind + my_slot) = epoch;
    }
  __threadfence_system();
}

__global__ void k_allreduce_local_coef(unsigned long long* own_words, int n_slots, int n, unsigned long long epoch,
                                       double* scalars, int mode, int has_gc, double k_vol, double v_target, int* error) {
  __shared__ int ok;
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  for (int s = threadIdx.x; s < n_slots; s += blockDim.x) {
    const volatile unsigned long long* f = own_words + kPushScalarFlagBase + s;
    const long long t0 = clock64();
    while (*f < epoch) {
      if (clock64() - t0 > kWaitCycles) {
        atomicExch(error, 1);
        ok = 0;
        break;
      }
      __nanosleep(100);
    }
  }
  __syncthreads();
  if (!ok) return;
  __threadfence_system();
  if (int(threadIdx.x) < n) {
    const volatile double* base = reinterpret_cast<const volatile double*>(own_words + kPushScalarBase);
    double acc = 0.0;
    for (int s = 0; s < n_slots; ++s) acc += base[(16 * int(epoch & 1ull) + s) * 16 + threadIdx.x];
    scalars[threadIdx.x] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0 && mode != -2) kkt_coefficient(scalars, mode, has_gc, k_vol, v_target);
}

cudaError_t launch_halo_push(int n_rows, int width, const double* src, double* const* peer_base, const int32_t* dst_slot,
                             const int32_t* src_row, const int32_t* dst_row, unsigned long long* const* peer_flags,
                             int n_slots, uint64_t dst_mask, int my_slot, int kind, unsigned long long epoch,
                             unsigned int* ticket, cudaStream_t st) {
  int blocks = (n_rows * width + 255) / 256;
  blocks = blocks < 1 ? 1 : (blocks > 64 ? 64 : blocks);
  k_halo_push<<<blocks, 256, 0, st>>>(n_rows, width, src, peer_base, dst_slot, src_row, dst_row, peer_flags, n_slots,
                                      dst_mask, my_slot, kind, epoch, ticket);
  return cudaGetLastError();
}

cudaError_t launch_allreduce_local_coef(double* scalars, int n, unsigned long long* own_words, int n_slots,
                                        unsigned long long epoch, int mode, int has_gc, double k_vol, double v_target,
                                        int* error, cudaStream_t st) {
  k_allreduce_local_coef<<<1, 64, 0, st>>>(own_words, n_slots, n, epoch, scalars, mode, has_gc, k_vol, v_target, error);
  return cudaGetLastError();
}

cudaError_t launch_halo_exchange(unsigned long long* own_flag, int n_ghost, int width, const double* const* peer_base,
                                 unsigned long long* const* peer_flag, int n_slots, int flag_index,
                                 unsigned long long epoch, const int32_t* owner, const int32_t* row, double* dst,
                                 int* error, cudaStream_t st) {
  const int blocks = (n_ghost * width + 255) / 256;
  k_halo_exchange<<<blocks < 64 ? (blocks > 0 ? blocks : 1) : 64, 256, 0, st>>>(own_flag, n_ghost, width, peer_base, peer_flag,
                                                                               n_slots, flag_index, epoch, owner, row, dst,
                                                                               error);
  return cudaGetLastError();
}

cudaError_t launch_allreduce_gather_coef(double* scalars, int n, unsigned long long* const* peer_words, int n_slots,
                                         unsigned long long epoch, int mode, int has_gc, double k_vol, double v_target,
                                         int* error, cudaStream_t st) {
  k_allreduce_gather_coef<<<1, 64, 0, st>>>(peer_words, n_slots, n, epoch, scalars, mode, has_gc, k_vol, v_target, error);
  return cudaGetLastError();
}

cudaError_t launch_allreduce_peer(double* scalars, int n, unsigned long long* own_words, unsigned long long* const* peer_words,
                                  int n_slots, unsigned long long epoch, int* error, cudaStream_t st) {
  k_allreduce_publish<<<1, 32, 0, st>>>(scalars, n, own_words, epoch);
  k_allreduce_gather<<<1, 64, 0, st>>>(peer_words, n_slots, n, epoch, scalars, error);
  return cudaGetLastError();
}

// First launches load the kernels' code (lazy module loading), which may synchronise the device: do them once,
// with no work, before contexts start waiting for each other.
cudaError_t launch_halo_warmup(unsigned long long* words, double* scalars, int* error, unsigned int* push_ticket,
                               cudaStream_t st) {
  k_halo_signal<<<1, 1, 0, st>>>(words + 3, 0ull);
  k_halo_pull<<<1, 256, 0, st>>>(0, 3, nullptr, nullptr, 0, 0, 0ull, nullptr, nullptr, nullptr, error);
  k_allreduce_publish<<<1, 32, 0, st>>>(scalars, 0, words, 0ull);
  k_allreduce_gather<<<1, 64, 0, st>>>(nullptr, 0, 0, 0ull, scalars, error);
  // every kernel a lock-step sequence may launch for the first time while a peer's kernel is already waiting: the
  // lazy load of a kernel can need the device, which a waiting kernel of the same process holds
  k_allreduce_gather_coef<<<1, 64, 0, st>>>(nullptr, 0, 0, 0ull, scalars, -2, 0, 0.0, 0.0, error);
  k_halo_exchange<<<1, 256, 0, st>>>(words + 3, 0, 3, nullptr, nullptr, 0, 0, 0ull, nullptr, nullptr, nullptr, error);
  k_reduce_partials<<<1, kReduceRows * kPartialStride, 0, st>>>(nullptr, 0, nullptr, 0, 0u, scalars);
  k_kkt_coefficient<<<1, 1, 0, st>>>(scalars, -1, 0, 0.0, 0.0);
  // push transport: no row, no destination (the single block takes the ticket and puts it back to 0); no rank to wait
  // for, no scalar written
  k_halo_push<<<1, 256, 0, st>>>(0, 3, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0ull, 0, 0, 0ull,
                                 push_ticket);
  k_allreduce_local_coef<<<1, 64, 0, st>>>(words, 0, 0, 0ull, scalars, -2, 0, 0.0, 0.0, error);
  return cudaGetLastError();
}

cudaError_t launch_min_edge2(const int32_t* tri, int32_t nf, int32_t nv, const double* pos,
                             unsigned long long* out, cudaStream_t st) {
  if (nf > 0) k_min_edge2<<<blocks_for(nf, 256), 256, 0, st>>>(tri, nf, nv, pos, out);
  return cudaGetLastError();
}

cudaError_t launch_max_row_norm2(const double* rows, int64_t n, unsigned long long* out, cudaStream_t st) {
  if (n > 0) k_max_row_norm2<<<blocks_for(n, 256), 256, 0, st>>>(rows, n, out);
  return cudaGetLastError();
}

cudaError_t launch_normal_change(const int32_t* tri, int32_t nf, int32_t nv, const double* old_pos,
                                 const double* new_pos, double cos_limit, int* flag, cudaStream_t st) {
  if (nf > 0) k_normal_change<<<blocks_for(nf, 256), 256, 0, st>>>(tri, nf, nv, old_pos, new_pos, cos_limit, flag);
  return cudaGetLastError();
}

cudaError_t launch_cg_direction(const double* g, const double* pg, const double* pd, const uint8_t* fixed,
                                int64_t nv, double* d, cudaStream_t st, const int32_t* restart_dev) {
  if (nv > 0) k_cg_direction<<<blocks_for(nv, 256), 256, 0, st>>>(g, pg, pd, fixed, nv, d, restart_dev);
  return cudaGetLastError();
}

cudaError_t launch_axpy_rows(const double* x, double alpha, const uint8_t* fixed, int64_t nv, double* y,
                             cudaStream_t st, const double* alpha_dev) {
  if (nv > 0) k_axpy_rows<<<blocks_for(3 * nv, 256), 256, 0, st>>>(x, alpha, alpha_dev, fixed, nv, y);
  return cudaGetLastError();
}

namespace {
// initial words of the line-search reductions: min edge^2 = 1e300, max |d|^2 = 0, guard flag, spare
__global__ void k_ls_init(unsigned long long* bits) {
  if (threadIdx.x == 0) {
    bits[0] = (unsigned long long)__double_as_longlong(1.0e300);
    bits[1] = (unsigned long long)__double_as_longlong(0.0);
    bits[2] = bits[3] = 0ull;
  }
}

// one thread: advance the loop of ms_ctx_minimize to its next action and open that action's IF node
__global__ void k_min_control(MinOpts o, MinState* s, const double* scalars, const unsigned long long* ls_bits, int32_t nf,
                              double* hist, int32_t hist_cap, int32_t proj_grad, int32_t ran_a_grad, MinHandles h) {
  if (threadIdx.x != 0) return;
  MinInput in;
  in.sc = scalars;
  ms_min_ls_stats(ls_bits, scalars, nf, in.ls);
  in.ok = reinterpret_cast<const int*>(ls_bits + 2)[0] == 0;
  const int32_t act = ms_min_step(o, *s, in, hist, hist_cap, proj_grad, ran_a_grad);
  for (int k = 0; k < MN_ACTIONS; ++k)
    if (h.present & (1u << k)) cudaGraphSetConditional(h.act[k], act == k ? 1u : 0u);
  cudaGraphSetConditional(h.run, act == MN_DONE ? 0u : 1u);
}
}  // namespace

cudaError_t launch_ls_init(unsigned long long* bits, cudaStream_t st) {
  k_ls_init<<<1, 32, 0, st>>>(bits);
  return cudaGetLastError();
}

cudaError_t launch_min_control(const MinOpts& o, MinState* s, const double* scalars, const unsigned long long* ls_bits,
                               int32_t nf, double* hist, int32_t hist_cap, int32_t proj_grad, int32_t ran_a_grad,
                               const MinHandles& h, cudaStream_t st) {
  k_min_control<<<1, 32, 0, st>>>(o, s, scalars, ls_bits, nf, hist, hist_cap, proj_grad, ran_a_grad, h);
  return cudaGetLastError();
}

cudaError_t launch_scale(const double* x, double scale, double* out, int64_t n, cudaStream_t st) {
  if (n > 0) k_scale<<<blocks_for(n, 256), 256, 0, st>>>(x, scale, out, n);
  return cudaGetLastError();
}

// --- patch packing (ms_pack_device.cuh): one warp per chunk, one thread per corner / vertex row / slot ---
namespace {

struct PkWarp {
  __device__ int lane() const { return int(threadIdx.x & 31); }
  __device__ int size() const { return 32; }
  __device__ void sync() const { __syncwarp(); }
  __device__ uint32_t ballot(bool p) const { return __ballot_sync(0xffffffffu, p); }
  __device__ uint32_t lt_mask() const { return (1u << lane()) - 1u; }
  __device__ int bcast(int x) const { return __shfl_sync(0xffffffffu, x, 0); }
  __device__ uint64_t min64(uint64_t x) const {
    for (int o = 16; o > 0; o >>= 1) {
      const uint64_t y = __shfl_xor_sync(0xffffffffu, x, o);
      x = y < x ? y : x;
    }
    return x;
  }
};

__global__ void __launch_bounds__(256) k_pk_corner_keys(const int32_t* __restrict__ tri, int32_t nv, int64_t n,
                                                        int32_t* __restrict__ key, int32_t* __restrict__ id) {
  const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= n) return;
  key[c] = pk_corner_key(tri, nv, c);
  id[c] = int32_t(c);
}

// ptr[v] = first sorted position whose key is >= v
__global__ void __launch_bounds__(256) k_pk_csr_ptr(const int32_t* __restrict__ skey, int64_t n, int32_t nv,
                                                    int32_t* __restrict__ ptr) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v > nv) return;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) / 2;
    if (skey[mid] < v) lo = mid + 1; else hi = mid;
  }
  ptr[v] = int32_t(lo);
}

__global__ void __launch_bounds__(256) k_pk_bounds(const PackParams p, const int32_t* __restrict__ csr_ptr,
                                                   int32_t n_owned, unsigned long long* __restrict__ bounds) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= n_owned) return;
  const int64_t chunk = pk_chunk_rows(p), c = v / chunk;
  const int32_t c1 = int32_t((c + 1) * chunk < n_owned ? (c + 1) * chunk : n_owned);
  int64_t window, deg;
  pk_row_bounds(p, csr_ptr, int32_t(v), c1, &window, &deg);
  atomicMax(bounds + 3 * c, (unsigned long long)window);
  atomicMax(bounds + 3 * c + 1, (unsigned long long)deg);
  if (v == c * chunk) bounds[3 * c + 2] = (unsigned long long)(csr_ptr[c1] - csr_ptr[v]);
}

__global__ void __launch_bounds__(256) k_pk_valid(const int32_t* __restrict__ tri, int32_t nv, int32_t nf,
                                                  unsigned long long* __restrict__ n_valid) {
  const int64_t f = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool ok = f < nf && pk_valid(tri + 3 * f, nv);
  const unsigned mask = __ballot_sync(0xffffffffu, ok);
  if (mask && (threadIdx.x & 31) == 0) atomicAdd(n_valid, (unsigned long long)__popc(mask));
}

__global__ void __launch_bounds__(32) k_pk_chunks(const PkMesh m, int32_t* scratch, const PkStage st, PkChunk* chunks) {
  PkWarp w;
  const int64_t c = blockIdx.x, chunk = pk_chunk_rows(m.prm);
  const int32_t v1 = int32_t((c + 1) * chunk < m.n_owned ? (c + 1) * chunk : m.n_owned);
  pk_chunk(w, m, scratch, st, chunks[c], int32_t(c * chunk), v1);
}

// one block per chunk: its headers (offsets made global), halo ids and listed records into the concatenation
__global__ void __launch_bounds__(256) k_pk_concat(const PkStage st, const PkChunk* __restrict__ chunks,
                                                   const int64_t* __restrict__ bases, PatchHeader* hdr, int32_t* halo,
                                                   FacetRec* recs, int32_t* slot_facet) {
  const PkChunk& k = chunks[blockIdx.x];
  const int64_t hb = bases[3 * blockIdx.x], lb = bases[3 * blockIdx.x + 1], sb = bases[3 * blockIdx.x + 2];
  for (int64_t j = threadIdx.x; j < k.n_patches; j += blockDim.x) {
    PatchHeader h = st.hdr[k.hdr_off + j];
    h.halo_off += int32_t(lb);
    h.slot_off += sb;
    hdr[hb + j] = h;
  }
  for (int64_t j = threadIdx.x; j < k.n_halo; j += blockDim.x) halo[lb + j] = st.halo[k.halo_off + j];
  for (int64_t e = k.ent_off + threadIdx.x; e < k.ent_off + k.n_listed; e += blockDim.x) {
    recs[sb + st.ent_slot[e]] = st.ent_rec[e];
    slot_facet[sb + st.ent_slot[e]] = st.ent_fac[e];
  }
}

// one block per patch, one thread per (round, half-warp)
__global__ void __launch_bounds__(128) k_pk_hw_excess(const PatchHeader* __restrict__ hdr, const FacetRec* __restrict__ recs,
                                                      int32_t T, unsigned long long* out) {
  const PatchHeader h = hdr[blockIdx.x];
  const int nhw = pk_n_hw(T);
  int64_t groups = 0, excess = 0;
  for (int64_t g = threadIdx.x; g < int64_t(h.n_rounds) * nhw; g += blockDim.x) {
    const int hw = int(g % nhw);
    pk_hw_excess(recs + h.slot_off + (g / nhw) * T + hw * 16, T - hw * 16 < 16 ? T - hw * 16 : 16, &groups, &excess);
  }
  if (groups) atomicAdd(out, (unsigned long long)groups);
  if (excess) atomicAdd(out + 1, (unsigned long long)excess);
}

__global__ void __launch_bounds__(256) k_pk_slot_gamma(const int32_t* __restrict__ slot_facet, int64_t n,
                                                       const double* __restrict__ gamma, double* __restrict__ out) {
  const int64_t s = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int32_t f = slot_facet[s];
  out[s] = f >= 0 ? gamma[f] : 0.0;
}

__global__ void __launch_bounds__(256) k_pk_inject(const PatchHeader* __restrict__ hdr, int32_t n, FacetRec* recs) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const PatchHeader h = hdr[p];
  if (h.n_rounds > 0 && (recs[h.slot_off].flags & REC_VALID)) recs[h.slot_off + 1] = recs[h.slot_off];
}

int pk_key_bits(int32_t nv) {
  int bits = 1;
  while (bits < 31 && (uint32_t(nv) >> bits)) ++bits;
  return bits;
}

}  // namespace

cudaError_t pk_temp_bytes(int64_t n_corners, size_t* bytes) {
  return cub::DeviceRadixSort::SortPairs(nullptr, *bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                         (const int32_t*)nullptr, (int32_t*)nullptr, int(n_corners));
}

cudaError_t launch_pk_corner_csr(const int32_t* tri, int32_t nv, int32_t nf, int32_t* key_in, int32_t* id_in,
                                 int32_t* key_out, int32_t* csr_idx, int32_t* csr_ptr, void* temp, size_t temp_bytes,
                                 cudaStream_t st) {
  const int64_t n = 3 * int64_t(nf);
  if (n > 0) {
    k_pk_corner_keys<<<blocks_for(n, 256), 256, 0, st>>>(tri, nv, n, key_in, id_in);
    if (cudaError_t e = cudaGetLastError()) return e;
    if (cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_in, key_out, id_in, csr_idx, int(n), 0,
                                                        pk_key_bits(nv), st))
      return e;
  }
  k_pk_csr_ptr<<<blocks_for(int64_t(nv) + 1, 256), 256, 0, st>>>(key_out, n, nv, csr_ptr);
  return cudaGetLastError();
}

cudaError_t launch_pk_bounds(const PackParams& p, const int32_t* csr_ptr, int32_t n_owned, const int32_t* tri,
                             int32_t nv, int32_t nf, unsigned long long* bounds, int64_t n_chunks,
                             unsigned long long* n_valid, cudaStream_t st) {
  if (cudaError_t e = cudaMemsetAsync(bounds, 0, (3 * size_t(n_chunks) + 1) * sizeof(unsigned long long), st)) return e;
  if (n_owned > 0) k_pk_bounds<<<blocks_for(n_owned, 256), 256, 0, st>>>(p, csr_ptr, n_owned, bounds);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (nf > 0) k_pk_valid<<<blocks_for(nf, 256), 256, 0, st>>>(tri, nv, nf, n_valid);
  return cudaGetLastError();
}

cudaError_t launch_pk_chunks(const PkMesh& m, int32_t* scratch, const PkStage& stage, PkChunk* chunks, int64_t n_chunks,
                             cudaStream_t st) {
  if (n_chunks > 0) k_pk_chunks<<<unsigned(n_chunks), 32, 0, st>>>(m, scratch, stage, chunks);
  return cudaGetLastError();
}

cudaError_t launch_pk_concat(const PkStage& stage, const PkChunk* chunks, const int64_t* bases, int64_t n_chunks,
                             PatchHeader* hdr, int32_t* halo, FacetRec* recs, int32_t* slot_facet, int64_t n_slots,
                             cudaStream_t st) {
  if (n_slots > 0) {
    if (cudaError_t e = cudaMemsetAsync(recs, 0, size_t(n_slots) * sizeof(FacetRec), st)) return e;
    if (cudaError_t e = cudaMemsetAsync(slot_facet, 0xff, size_t(n_slots) * sizeof(int32_t), st)) return e;
  }
  if (n_chunks > 0) k_pk_concat<<<unsigned(n_chunks), 256, 0, st>>>(stage, chunks, bases, hdr, halo, recs, slot_facet);
  return cudaGetLastError();
}

cudaError_t launch_pk_hw_excess(const PatchHeader* hdr, int32_t n_patches, const FacetRec* recs, int32_t threads,
                                unsigned long long* out, cudaStream_t st) {
  if (cudaError_t e = cudaMemsetAsync(out, 0, 2 * sizeof(unsigned long long), st)) return e;
  if (n_patches > 0) k_pk_hw_excess<<<unsigned(n_patches), 128, 0, st>>>(hdr, recs, threads, out);
  return cudaGetLastError();
}

cudaError_t launch_pk_slot_gamma(const int32_t* slot_facet, int64_t n, const double* gamma, double* out, cudaStream_t st) {
  if (n > 0) k_pk_slot_gamma<<<blocks_for(n, 256), 256, 0, st>>>(slot_facet, n, gamma, out);
  return cudaGetLastError();
}

cudaError_t launch_pk_inject(const PatchHeader* hdr, int32_t n_patches, FacetRec* recs, cudaStream_t st) {
  if (n_patches > 0) k_pk_inject<<<blocks_for(n_patches, 256), 256, 0, st>>>(hdr, n_patches, recs);
  return cudaGetLastError();
}

}  // namespace ms
