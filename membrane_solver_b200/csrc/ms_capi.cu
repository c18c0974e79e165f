// C-ABI layer (include/ms_b200.h): context with device-resident mesh buffers and
// the stateless per-kernel shims.  Replaces the dispatch of
// fortran_kernels/loader.py for the energy+gradient path.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/ms_b200.h"
#include "ms_kernels.cuh"
#include "ms_pack.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU(expr)                                                                         \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      return fail(-100 - int(_e), std::string(#expr) + ": " + cudaGetErrorString(_e));   \
  } while (0)

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  int ensure(size_t count) {
    if (count <= n && p) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    if (count == 0) return 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
    if (e != cudaSuccess) return fail(-100 - int(e), std::string("cudaMalloc: ") + cudaGetErrorString(e));
    n = count;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  void swap(DevBuf& o) {
    std::swap(p, o.p);
    std::swap(n, o.n);
  }
  ~DevBuf() { release(); }
};

bool g_configured[64] = {false};

// NVTX range around the launches of one phase (visible in Nsight Systems / ncu --nvtx; a no-op without a tool)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

}  // namespace

struct ms_ctx {
  ~ms_ctx() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    for (cudaEvent_t e : mn_ev)
      if (e) cudaEventDestroy(e);
    if (h_min_state) cudaFreeHost(h_min_state);
    if (h_min_hist) cudaFreeHost(h_min_hist);
    if (mn_stream) cudaStreamDestroy(mn_stream);
  }
  int device = 0;
  cudaStream_t stream = nullptr;
  bool have_topology = false;
  bool has_positions = false;  // MS_ARR_POSITIONS has been written since the topology was set
  int32_t nv = 0, nf = 0;
  int32_t n_owned = 0;  // vertex rows owned by this context's patches (== nv unless partitioned)
  ms::PackParams pack_params;
  ms::PackedMesh packed;  // headers, halo ids and statistics; the records and slot facets live on the device only
  int64_t n_slots = 0;    // record slots of the packing (d_recs, d_slot_facet)
  std::vector<int32_t> v_lo;

  DevBuf<ms::PatchHeader> d_patches;
  DevBuf<int32_t> d_halo;
  DevBuf<ms::FacetRec> d_recs;
  DevBuf<int32_t> d_slot_facet;  // facet row of each record slot, -1 for an empty one
  DevBuf<double> d_slot_gamma;
  DevBuf<uint8_t> d_boundary, d_fixed;
  DevBuf<int32_t> d_boundary32;  // boundary flags as int32: staged into shared memory with 4-byte cp.async
  DevBuf<double> d_tilt_sq;      // |t|^2 per vertex, refreshed before every evaluation that uses the tilts
  DevBuf<double> d_kappa, d_c0;
  DevBuf<double> d_pos, d_trial, d_dir, d_tilts, d_seeds, d_partials_a, d_partials_b, d_grad, d_volgrad,
      d_tilt_grad, d_scalars, d_dot_partials, d_kvecs, d_avor, d_aeff, d_evert;
  bool ran_pass_a = false;  // the last evaluation ran pass A (its per-CTA sums are current)
  // Deferred KKT projection: MS_ARR_GRAD holds the raw energy gradient and scalars[SC_COEF] the coefficient; the
  // projected gradient g + coef * gC (fixed rows zeroed) is formed by whoever consumes it (direction, dots) or
  // materialised in place on first access through the ABI (flush_projection).
  struct PendingProjection {
    bool active = false, use_gc = false, use_fixed = false;
  } proj;
  DevBuf<unsigned int> d_ticket;  // [0] last-CTA ticket of the fused finalisation, [1] push kernel, [2] in-kernel pulls
  unsigned int pull_arrived = 0;  // host mirror of d_ticket[2]: CTAs that have reported so far
  DevBuf<int> d_self_check;       // violation counters of the self-check build (ms_ctx_self_check)
  bool has_gamma = false, has_kappa = false, has_c0 = false, has_boundary = false,
       has_fixed = false, has_body = false;
  double gamma_u = 1.0, kappa_u = 0.0, c0_u = 0.0, k_tilt = 0.0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> events;
  DevBuf<uint8_t> d_flush;
  DevBuf<int32_t> d_send_rows;  // rows other partitions read from this one (halo exchange)
  // partitions: patches whose halo lies entirely in the owned rows (interior) first, then the patches that
  // reference ghost rows (boundary) -- the interior ones can run while the halo exchange is in flight
  DevBuf<int32_t> d_patch_order;
  int32_t n_interior = 0;
  int32_t max_ctas = 0;  // 0 = one persistent CTA per SM
  // pipelined host evaluation: chunks of the position upload overlap the patch kernels.  orderA lists the
  // patches by the last vertex row they read; orderB by how many orderA patches must have run pass A first.
  bool pipe_ready = false;
  std::vector<int32_t> pipe_need_a, pipe_need_b;  // sorted keys of orderA / orderB
  DevBuf<int32_t> d_order_a, d_order_b;
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> pipe_events;
  // internal vertex order: row i of every device array holds the caller's vertex perm[i]
  std::vector<double> order_hint;       // positions given by ms_ctx_set_vertex_order_hint (consumed by set_topology)
  std::vector<int32_t> perm;            // new -> old; empty = identity
  DevBuf<int32_t> d_perm;
  DevBuf<double> d_stage;               // staging for permuted uploads / downloads (5*nv doubles)
  // triangle rows + corner CSR on the device (built on first use), bending-tilt buffers
  std::vector<int32_t> h_tri;
  bool bt_ready = false, tri_ready = false, csr_ready = false;
  DevBuf<double> d_cg_prev_g, d_cg_prev_d;  // conjugate-gradient memory (previous gradient / direction)
  DevBuf<unsigned long long> d_ls_bits;  // line-search reductions: [min edge^2, max |d|^2] as bit patterns, [flag]
  DevBuf<int32_t> d_tri, d_csr_ptr, d_csr_idx;
  DevBuf<double> d_bt_corner, d_bt_base, d_bt_facet_e, d_bt_e;
  DevBuf<int32_t> d_va_group;  // pin groups of ms_ctx_vertex_average (internal order)
  // host copies that outlive a re-pack of flipped rows (ms_ctx_equiangulate): per-facet gamma and body membership
  std::vector<double> h_gamma;
  std::vector<uint8_t> h_body;
  // the last ms_ctx_equiangulate: selection rounds of every sweep run; ms of sweeps, D2H of the rows, device pack, commit
  std::vector<int32_t> eq_rounds;
  double eq_ms[4] = {0, 0, 0, 0};
  double rf_ms[4] = {0, 0, 0, 0};  // the last ms_ctx_refine: device ms, D2H of rows and order, device pack, commit
  int64_t n_send_rows = 0;
  // leaflet tilt modules (ms_leaflet.cuh): per-leaflet selections, parameters and tilt fields
  struct Leaflet {
    bool set = false;
    bool has_keep = false, has_interior = false, has_base_zero = false, has_kappa = false, has_c0 = false,
         has_weight = false, has_consistent = false;
    DevBuf<uint8_t> keep, interior, base_zero, consistent;
    DevBuf<double> kappa, c0, weight, tilts, tilt_grad, trial, dir, minv;
    bool has_minv = false;
    DevBuf<uint8_t> fixed;
    bool has_fixed = false;
    double kappa_u = 0.0, c0_u = 0.0, k_tilt = 0.0, k_smooth = 0.0, sign = 1.0;
    int32_t consistent_u = 0;
  } leaflet[3];  // inner leaflet, outer leaflet, single tilt field
  DevBuf<double> d_lf_corner, d_lf_vbuf, d_lf_shape, d_lf_tilt, d_lf_facet_e, d_lf_e;
  DevBuf<double> d_lf_corner2, d_lf_vbuf2, d_lf_shape2, d_lf_tilt2;  // second leaflet of a paired evaluation
  DevBuf<double> d_vnormals, d_rowsq, d_norm_out, d_lf_block_e;
  DevBuf<unsigned long long> d_lf_ticket;
  unsigned long long lf_ticket_base = 0;
  bool lf_fused_ok = true;
  // halo exchange over peer memory: opened peer arrays, flag words, ghost source table
  struct PeerTable {
    std::vector<void*> opened;                       // every pointer returned by cudaIpcOpenMemHandle
    std::vector<const double*> pos, trial, seeds;    // per owner slot
    std::vector<unsigned long long*> flags;
    DevBuf<const double*> d_pos, d_trial, d_seeds;
    DevBuf<unsigned long long*> d_flags;
    DevBuf<int32_t> d_owner, d_row;
    // push transport: for every row another rank lists as a ghost -- that rank's slot, the row here, the row there
    DevBuf<int32_t> d_push_slot, d_push_src, d_push_dst;
    int32_t n_push = 0, my_slot = -1;
    uint64_t push_mask = 0;    // ranks this one pushes to == ranks it receives from (1-ring ghosts are symmetric)
    bool push_ready = false;
    int32_t n_slots = 0;
    bool tables_current = false;
  } peers;
  DevBuf<unsigned long long> d_flag_words;           // this rank's flag words (exported)
  DevBuf<int> d_halo_error;
  unsigned long long flag_epoch[4] = {0, 0, 0, 0};
  bool vnormals_ready = false;
  // ms_ctx_minimize: loop state and history on the device, the capture stream of its graph, its statistics
  DevBuf<ms::MinState> d_min_state;
  DevBuf<double> d_min_hist;
  ms::MinState* h_min_state = nullptr;  // pinned staging: the copies around the graph do not block the host
  double* h_min_hist = nullptr;
  size_t h_min_hist_n = 0;
  cudaStream_t mn_stream = nullptr;
  cudaEvent_t mn_ev[2] = {nullptr, nullptr};
  int64_t mn_counts[7] = {0, 0, 0, 0, 0, 0, 0};
  double mn_ms[2] = {0, 0};
};

namespace {

constexpr int kDotBlocks = 592;  // 4 CTAs per SM on 148 SMs

int use_device(const ms_ctx* c) {
  CU(cudaSetDevice(c->device));
  return 0;
}

int check_ctx(const ms_ctx* c, bool need_topology) {
  if (!c) return fail(-1, "null context");
  if (need_topology && !c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  return use_device(c);
}

// Materialise a deferred projection in MS_ARR_GRAD (see ms_ctx::proj).
int flush_projection(ms_ctx* c) {
  if (!c->proj.active) return 0;
  c->proj.active = false;
  CU(ms::launch_apply_projection(c->d_grad.p, c->proj.use_gc ? c->d_volgrad.p : nullptr,
                                 c->proj.use_fixed ? c->d_fixed.p : nullptr, c->n_owned, c->d_scalars.p, c->stream));
  return 0;
}

double* array_ptr(ms_ctx* c, int which, int64_t* len) {
  const int64_t nv = c->nv;
  switch (which) {
    case MS_ARR_POSITIONS: *len = 3 * nv; return c->d_pos.p;
    case MS_ARR_GRAD: *len = 3 * nv; return c->d_grad.p;
    case MS_ARR_VOLGRAD: *len = 3 * nv; return c->d_volgrad.p;
    case MS_ARR_SEEDS: *len = ms::kSeedStride * nv; return c->d_seeds.p;
    case MS_ARR_TILTS: *len = 3 * nv; return c->d_tilts.p;
    case MS_ARR_TILT_GRAD: *len = 3 * nv; return c->d_tilt_grad.p;
    case MS_ARR_SCALARS: *len = MS_SC_COUNT; return c->d_scalars.p;
    case MS_ARR_K_VECS: *len = 3 * nv; return c->d_kvecs.p;
    case MS_ARR_A_VOR: *len = nv; return c->d_avor.p;
    case MS_ARR_A_EFF: *len = nv; return c->d_aeff.p;
    case MS_ARR_E_VERTEX: *len = nv; return c->d_evert.p;
    case MS_ARR_TRIAL: *len = 3 * nv; return c->d_trial.p;
    case MS_ARR_DIRECTION: *len = 3 * nv; return c->d_dir.p;
    case MS_ARR_TILTS_IN: *len = 3 * nv; return c->leaflet[0].tilts.p;
    case MS_ARR_TILTS_OUT: *len = 3 * nv; return c->leaflet[1].tilts.p;
    case MS_ARR_TILT_GRAD_IN: *len = 3 * nv; return c->leaflet[0].tilt_grad.p;
    case MS_ARR_TILT_GRAD_OUT: *len = 3 * nv; return c->leaflet[1].tilt_grad.p;
    case MS_ARR_TILTS_FIELD: *len = 3 * nv; return c->leaflet[2].tilts.p;
    case MS_ARR_TILT_GRAD_FIELD: *len = 3 * nv; return c->leaflet[2].tilt_grad.p;
    default: *len = 0; return nullptr;
  }
}

// Lazily allocate the optional arrays the first time they are addressed.
int ensure_array(ms_ctx* c, int which) {
  const size_t nv = size_t(c->nv);
  switch (which) {
    case MS_ARR_TILTS: return c->d_tilts.ensure(3 * nv);
    case MS_ARR_TILT_GRAD: return c->d_tilt_grad.ensure(3 * nv);
    case MS_ARR_K_VECS: return c->d_kvecs.ensure(3 * nv);
    case MS_ARR_A_VOR: return c->d_avor.ensure(nv);
    case MS_ARR_A_EFF: return c->d_aeff.ensure(nv);
    case MS_ARR_E_VERTEX: return c->d_evert.ensure(nv);
    case MS_ARR_TRIAL: return c->d_trial.ensure(3 * nv);
    case MS_ARR_DIRECTION: return c->d_dir.ensure(3 * nv);
    case MS_ARR_TILTS_IN: return c->leaflet[0].tilts.ensure(3 * nv);
    case MS_ARR_TILTS_OUT: return c->leaflet[1].tilts.ensure(3 * nv);
    case MS_ARR_TILT_GRAD_IN: return c->leaflet[0].tilt_grad.ensure(3 * nv);
    case MS_ARR_TILT_GRAD_OUT: return c->leaflet[1].tilt_grad.ensure(3 * nv);
    case MS_ARR_TILTS_FIELD: return c->leaflet[2].tilts.ensure(3 * nv);
    case MS_ARR_TILT_GRAD_FIELD: return c->leaflet[2].tilt_grad.ensure(3 * nv);
    default: return 0;
  }
}

int fill_launch(ms_ctx* c, const ms_eval_opts* o, ms::PatchLaunch& a) {
  const int n_patches = int(c->packed.patches.size());
  int begin = o->patch_count < 0 ? 0 : o->patch_begin;
  int count = o->patch_count < 0 ? n_patches : o->patch_count;
  if (begin < 0 || count < 0 || begin + count > n_patches) return fail(-3, "patch range out of bounds");
  std::memset(&a, 0, sizeof(a));
#ifdef MS_DEBUG_VARIANTS
  {
    static const int dbg = [] { const char* e = std::getenv("MS_DEBUG_VARIANT"); return e ? std::atoi(e) : 0; }();
    a.debug = dbg;
  }
#endif
  if (o->patch_count == MS_PATCHES_INTERIOR || o->patch_count == MS_PATCHES_BOUNDARY) {
    // the two halves of one evaluation: interior patches, then the patches that read ghost rows; their
    // per-CTA sums occupy consecutive partial rows: [0, grid_i) and [grid_i, grid_i + grid_b)
    a.patch_list = c->d_patch_order.p;
    begin = o->patch_count == MS_PATCHES_INTERIOR ? 0 : c->n_interior;
    count = o->patch_count == MS_PATCHES_INTERIOR ? c->n_interior : n_patches - c->n_interior;
    ms::PatchLaunch inner;
    std::memset(&inner, 0, sizeof(inner));
    inner.patch_count = c->n_interior;
    inner.max_ctas = c->max_ctas;
    a.partial_row0 = o->patch_count == MS_PATCHES_INTERIOR ? 0 : ms::patch_grid(inner);
  }
  a.patches = c->d_patches.p;
  a.halo_ids = c->d_halo.p;
  a.recs = c->d_recs.p;
  a.slot_gamma = c->has_gamma ? c->d_slot_gamma.p : nullptr;
  a.patch_begin = begin;
  a.patch_count = count;
  a.max_ctas = c->max_ctas;
  a.threads = c->packed.params.threads;
  a.max_owned = c->packed.max_owned;
  a.max_local = c->packed.max_local;
  a.max_slots = c->packed.max_slots;
  a.max_rounds = c->packed.max_rounds;
  if (o->use_trial) {
    if (!c->d_trial.p) return fail(-4, "use_trial set but no trial positions exist (ms_ctx_make_trial)");
    a.pos = c->d_trial.p;
  } else {
    a.pos = c->d_pos.p;
  }
  a.tilts = c->d_tilts.p;
  a.is_boundary = c->has_boundary ? c->d_boundary.p : nullptr;
  a.boundary32 = c->has_boundary ? c->d_boundary32.p : nullptr;
  a.tilt_sq = nullptr;
  a.kappa = c->has_kappa ? c->d_kappa.p : nullptr;
  a.c0 = c->has_c0 ? c->d_c0.p : nullptr;
  a.gamma_u = c->gamma_u;
  a.kappa_u = c->kappa_u;
  a.c0_u = c->c0_u;
  a.k_tilt = c->k_tilt;
  a.modules = o->modules;
  a.flags = o->flags;
  a.seeds = c->d_seeds.p;
  a.partials = nullptr;  // set by the pass entry points
  a.grad = c->d_grad.p;
  a.volgrad = c->d_volgrad.p;
  a.self_check = c->d_self_check.p;
  if ((o->modules & MS_MOD_TILT)) {
    if (!c->d_tilts.p) return fail(-5, "tilt module requested but no tilts were uploaded");
    // |t|^2 per vertex for the producer's asynchronous staging (the tilts may have been changed through
    // ms_ctx_device_ptr, so it is refreshed per launch; 32 B per vertex of traffic)
    if (int rc = c->d_tilt_sq.ensure(size_t(c->nv) + 1)) return rc;
    CU(ms::launch_row_norm2(c->d_tilts.p, c->nv, c->d_tilt_sq.p, c->stream));
    a.tilt_sq = c->d_tilt_sq.p;
    if (o->want_grad) {
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD)) return rc;
      a.tilt_grad = c->d_tilt_grad.p;
    }
  }
  if (o->diagnostics) {
    for (int w : {MS_ARR_K_VECS, MS_ARR_A_VOR, MS_ARR_A_EFF, MS_ARR_E_VERTEX})
      if (int rc = ensure_array(c, w)) return rc;
    a.k_vecs = c->d_kvecs.p;
    a.a_vor = c->d_avor.p;
    a.a_eff = c->d_aeff.p;
    a.e_vertex = c->d_evert.p;
  }
  if (o->modules & MS_MOD_BENDING_TILT) {
    if (o->modules & MS_MOD_BENDING) return fail(-6, "bending and bending_tilt share the seed array; evaluate them separately");
    if (c->n_owned != c->nv) return fail(-6, "bending_tilt is not available on partitioned (multi-GPU) contexts");
    if (!c->d_tilts.p) return fail(-5, "bending_tilt requested but no tilts were uploaded");
    // the patch kernels see it as bending: pass A delivers K, A_vor, A_eff, pass B back-propagates
    // the seeds computed by the coupling stage (ms_bt.cuh)
    a.modules = (o->modules & ~uint32_t(MS_MOD_BENDING_TILT)) | MS_MOD_BENDING;
    for (int w : {MS_ARR_K_VECS, MS_ARR_A_VOR, MS_ARR_A_EFF})
      if (int rc = ensure_array(c, w)) return rc;
    a.k_vecs = c->d_kvecs.p;
    a.a_vor = c->d_avor.p;
    a.a_eff = c->d_aeff.p;
    if (o->want_grad || o->want_tilt_grad)
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD)) return rc;
  }
  return 0;
}

bool needs_bending(const ms_eval_opts* o) { return (o->modules & (MS_MOD_BENDING | MS_MOD_BENDING_TILT)) != 0; }
bool has_bt(const ms_eval_opts* o) { return (o->modules & MS_MOD_BENDING_TILT) != 0; }
bool wants_tilt_grad(const ms_eval_opts* o) { return o->want_grad || o->want_tilt_grad; }

// triangle rows (internal vertex order) on the device, uploaded on first use
int ensure_tri(ms_ctx* c) {
  const size_t nf = size_t(c->nf);
  if (c->tri_ready) return 0;
  if (int rc = c->d_tri.ensure(3 * nf + 1)) return rc;
  if (nf) CU(cudaMemcpy(c->d_tri.p, c->h_tri.data(), 3 * nf * sizeof(int32_t), cudaMemcpyHostToDevice));
  c->tri_ready = true;
  return 0;
}

// The vertex -> corner CSR (corner id 3 f + k, facet-major; ms::build_corner_csr) of device rows, by one stable sort of
// the corner keys: ptr gets nv + 1 offsets, idx 3 nf + 1 entries.
int corner_csr_device(ms_ctx* c, int32_t nv, int32_t nf, const int32_t* tri, DevBuf<int32_t>& ptr, DevBuf<int32_t>& idx) {
  const size_t n = 3 * size_t(nf);
  size_t tb = 0;
  CU(ms::pk_temp_bytes(int64_t(n), &tb));
  DevBuf<int32_t> key_in, id_in, key_out;
  DevBuf<uint8_t> temp;
  for (int rc : {key_in.ensure(n + 1), id_in.ensure(n + 1), key_out.ensure(n + 1), temp.ensure(tb + 1), ptr.ensure(size_t(nv) + 1),
                 idx.ensure(n + 1)})
    if (rc) return rc;
  CU(ms::launch_pk_corner_csr(tri, nv, nf, key_in.p, id_in.p, key_out.p, idx.p, ptr.p, temp.p, tb, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // the scratch is released on return
  return 0;
}

// triangle rows and the vertex -> corner CSR on the device, once per topology (the packing leaves its CSR behind)
int ensure_corner_csr(ms_ctx* c) {
  if (c->csr_ready) return 0;
  if (int rc = ensure_tri(c)) return rc;
  if (int rc = corner_csr_device(c, c->nv, c->nf, c->d_tri.p, c->d_csr_ptr, c->d_csr_idx)) return rc;
  c->csr_ready = true;
  return 0;
}

int bt_prepare(ms_ctx* c, ms::BtMesh& m) {
  const size_t nv = size_t(c->nv), nf = size_t(c->nf);
  if (int rc = ensure_corner_csr(c)) return rc;
  if (!c->bt_ready) {
    if (int rc = c->d_bt_corner.ensure(12 * nf + 1)) return rc;
    if (int rc = c->d_bt_base.ensure(nv + 1)) return rc;
    if (int rc = c->d_bt_facet_e.ensure(nf + 1)) return rc;
    if (int rc = c->d_bt_e.ensure(1 + ms::kSumBlocks)) return rc;
    c->bt_ready = true;
  }
  m.nv = c->nv;
  m.nf = c->nf;
  m.tri = c->d_tri.p;
  m.pos = nullptr;  // set by the caller (positions or trial)
  m.tilts = c->d_tilts.p;
  m.is_boundary = c->has_boundary ? c->d_boundary.p : nullptr;
  m.kappa = c->has_kappa ? c->d_kappa.p : nullptr;
  m.c0 = c->has_c0 ? c->d_c0.p : nullptr;
  m.kappa_u = c->kappa_u;
  m.c0_u = c->c0_u;
  m.csr_ptr = c->d_csr_ptr.p;
  m.csr_idx = c->d_csr_idx.p;
  return 0;
}

// Asynchronous device -> host copy of a per-vertex array in the CALLER's vertex order.
int download_rows(ms_ctx* c, const double* src_dev, double* host, int width) {
  const size_t n = size_t(c->nv) * size_t(width);
  if (!n) return 0;
  if (c->perm.empty()) {
    CU(cudaMemcpyAsync(host, src_dev, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    return 0;
  }
  CU(ms::launch_scatter_rows(src_dev, width, c->d_perm.p, c->nv, c->d_stage.p, c->stream));
  CU(cudaMemcpyAsync(host, c->d_stage.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  return 0;
}

// Morton (Z-curve) order of the hint positions: contiguous row ranges become compact surface
// patches, which is what keeps the ring-facet recomputation of the patch kernels small.
// ms_ctx_refine computes the same order on the device (ms_refine.cuh).
void morton_permutation(const std::vector<double>& pos, int32_t nv, std::vector<int32_t>& perm) {
  ms::MortonBox box = ms::morton_box_empty();
  for (int32_t v = 0; v < nv; ++v) ms::morton_box_add(box, &pos[3 * size_t(v)]);
  std::vector<uint64_t> key(size_t(nv), 0);
  for (int32_t v = 0; v < nv; ++v) key[size_t(v)] = ms::morton_key(box, &pos[3 * size_t(v)]);
  perm.resize(size_t(nv));
  std::iota(perm.begin(), perm.end(), 0);
  std::stable_sort(perm.begin(), perm.end(), [&](int32_t a, int32_t b) { return key[size_t(a)] < key[size_t(b)]; });
  bool identity = true;
  for (int32_t i = 0; i < nv && identity; ++i) identity = perm[size_t(i)] == i;
  if (identity) perm.clear();
}

// A packing built on the device (ms_pack_device.cuh): headers with the closing sentinel, halo ids, records and slot
// facets on the device; headers, halo ids and statistics also in `host` (its recs / slot_facet stay empty); and the
// corner CSR of the rows it packed.
struct DevPacking {
  ms::PackedMesh host;
  int64_t n_slots = 0;
  DevBuf<ms::PatchHeader> patches;
  DevBuf<int32_t> halo, slot_facet, csr_ptr, csr_idx;
  DevBuf<ms::FacetRec> recs;
};

// ms::pack_patches on the device, with its return codes (0, -1, -2, -3); other codes are CUDA or internal failures.
// tri and body (nf bytes or nullptr) are device arrays.  Changes nothing in the context.
int pack_device(ms_ctx* c, int32_t nv, int32_t n_owned, int32_t nf, const int32_t* tri, const uint8_t* body,
                const ms::PackParams& prm, DevPacking& out) {
  if (n_owned < 0 || n_owned > nv) n_owned = nv;
  if (nv < 0 || nf < 0 || (nf > 0 && !tri) || prm.threads <= 0 || prm.max_owned <= 0 || prm.max_local <= 0 ||
      prm.max_local > 65535 || prm.max_slots < prm.threads || prm.fill_pct < 10 || prm.fill_pct > 100)
    return -1;
  cudaStream_t st = c->stream;
  ms::PackedMesh& pk = out.host;
  pk = ms::PackedMesh();
  pk.nv = nv;
  pk.nf = nf;
  pk.params = prm;
  pk.n_owned_vertices = n_owned;
  if (int rc = corner_csr_device(c, nv, nf, tri, out.csr_ptr, out.csr_idx)) return rc;
  const int64_t chunk = ms::pk_chunk_rows(prm), n_chunks = (int64_t(n_owned) + chunk - 1) / chunk;
  std::vector<unsigned long long> hb(3 * size_t(n_chunks) + 1);
  {
    DevBuf<unsigned long long> bounds;
    if (int rc = bounds.ensure(hb.size())) return rc;
    CU(ms::launch_pk_bounds(prm, out.csr_ptr.p, n_owned, tri, nv, nf, bounds.p, n_chunks, bounds.p + 3 * n_chunks, st));
    CU(cudaMemcpyAsync(hb.data(), bounds.p, hb.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  pk.n_valid = int64_t(hb[3 * size_t(n_chunks)]);
  const std::vector<int64_t> b64(hb.begin(), hb.end() - 1);
  std::vector<ms::PkChunk> ck(static_cast<size_t>(n_chunks));
  const ms::PkPlan plan = ms::pk_plan(prm, n_owned, b64.data(), ck.data(), n_chunks);
  // scratch and staging, released on return
  DevBuf<int64_t> scratch, s_slot, bases;
  DevBuf<ms::PatchHeader> s_hdr;
  DevBuf<int32_t> s_halo, s_fac;
  DevBuf<ms::FacetRec> s_rec;
  DevBuf<ms::PkChunk> d_ck;
  DevBuf<unsigned long long> hx;
  for (int rc : {scratch.ensure(size_t(plan.scratch_words / 2) + 1), s_slot.ensure(size_t(plan.ent) + 1),
                 bases.ensure(3 * size_t(n_chunks) + 1), s_hdr.ensure(size_t(plan.hdr) + 1),
                 s_halo.ensure(size_t(plan.halo) + 1), s_fac.ensure(size_t(plan.ent) + 1), s_rec.ensure(size_t(plan.ent) + 1),
                 d_ck.ensure(size_t(n_chunks) + 1), hx.ensure(2)})
    if (rc) return rc;
  const ms::PkStage stage{s_hdr.p, s_halo.p, s_rec.p, s_fac.p, s_slot.p};
  const ms::PkMesh m{nv, nf, n_owned, tri, body, out.csr_ptr.p, out.csr_idx.p, prm};
  if (n_chunks) CU(cudaMemcpyAsync(d_ck.p, ck.data(), ck.size() * sizeof(ms::PkChunk), cudaMemcpyHostToDevice, st));
  CU(ms::launch_pk_chunks(m, reinterpret_cast<int32_t*>(scratch.p), stage, d_ck.p, n_chunks, st));
  if (n_chunks) CU(cudaMemcpyAsync(ck.data(), d_ck.p, ck.size() * sizeof(ms::PkChunk), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (const ms::PkChunk& k : ck) {  // the first failing chunk decides, as on the host
    if (k.rc == ms::kPkInternal) return fail(-9, "device packer: a scratch bound did not hold");
    if (k.rc) return k.rc;
  }
  std::vector<int64_t> hbase(3 * size_t(n_chunks));
  int64_t np = 0, nh = 0, ns = 0;
  for (size_t i = 0; i < ck.size(); ++i) {
    const ms::PkChunk& k = ck[i];
    hbase[3 * i] = np;
    hbase[3 * i + 1] = nh;
    hbase[3 * i + 2] = ns;
    np += k.n_patches;
    nh += k.n_halo;
    ns += k.n_slots;
    pk.max_owned = std::max(pk.max_owned, k.max_owned);
    pk.max_local = std::max(pk.max_local, k.max_local);
    pk.max_rounds = std::max(pk.max_rounds, k.max_rounds);
    pk.max_slots = std::max(pk.max_slots, k.max_slots);
    pk.n_round_slots += k.n_round_slots;
    pk.n_listed += k.n_listed;
    pk.n_lane_conflicts += k.n_lane_conflicts;
  }
  if (nh > INT32_MAX) return fail(-8, "the packing has more than 2^31 - 1 halo entries");
  for (int rc : {out.patches.ensure(size_t(np) + 1), out.halo.ensure(size_t(nh) + 1), out.recs.ensure(size_t(ns) + 1),
                 out.slot_facet.ensure(size_t(ns) + 1)})
    if (rc) return rc;
  if (n_chunks) CU(cudaMemcpyAsync(bases.p, hbase.data(), hbase.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  CU(ms::launch_pk_concat(stage, d_ck.p, bases.p, n_chunks, out.patches.p, out.halo.p, out.recs.p, out.slot_facet.p, ns, st));
  ms::PatchHeader end;  // sentinel header: closes the record range of the last patch
  std::memset(&end, 0, sizeof(end));
  end.v_lo = n_owned;
  end.halo_off = int32_t(nh);
  end.slot_off = ns;
  CU(cudaMemcpyAsync(out.patches.p + np, &end, sizeof(end), cudaMemcpyHostToDevice, st));
  CU(ms::launch_pk_hw_excess(out.patches.p, int32_t(np), out.recs.p, prm.threads, hx.p, st));
  unsigned long long hw[2] = {0, 0};
  CU(cudaMemcpyAsync(hw, hx.p, sizeof(hw), cudaMemcpyDeviceToHost, st));
  pk.patches.resize(size_t(np));
  pk.halo_ids.resize(size_t(nh));
  if (np) CU(cudaMemcpyAsync(pk.patches.data(), out.patches.p, size_t(np) * sizeof(ms::PatchHeader), cudaMemcpyDeviceToHost, st));
  if (nh) CU(cudaMemcpyAsync(pk.halo_ids.data(), out.halo.p, size_t(nh) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  pk.n_hw_groups = int64_t(hw[0]);
  pk.n_hw_excess = int64_t(hw[1]);
  out.n_slots = ns;
  return 0;
}

// Packs device triangle rows (internal vertex order) into `out` with the context's pack parameters.  A vertex of
// valence V needs V rounds, i.e. V * threads record slots, and a patch holds at most kPatchSlotCap of them: meshes with
// high-valence vertices (a disk centre, a cone apex) are packed with narrower rounds (96 -> 64 -> 32 lanes: valence
// up to 16 / 24 / 48).  body: nf bytes on the device or nullptr.  Changes nothing in the context.
int pack_rows(ms_ctx* c, int32_t nv, int32_t n_owned, int32_t nf, const int32_t* tri, const uint8_t* body,
              DevPacking& out) {
  ms::PackParams used_params = c->pack_params;
  int prc = pack_device(c, nv, n_owned, nf, tri, body, used_params, out);
  while (prc == -3 && used_params.threads > 32) {
    used_params.threads = used_params.threads > 64 ? 64 : 32;
    prc = pack_device(c, nv, n_owned, nf, tri, body, used_params, out);
  }
  if (prc == -2) return fail(-8, "a vertex neighbourhood exceeds max_local; raise it with ms_ctx_set_pack_params");
  if (prc == -3) return fail(-8, "a vertex has more than 48 incident facets: its rounds do not fit a patch");
  if (prc == -1) return fail(-1, "pack_patches failed");
  if (prc) return prc;
  const ms::PackedMesh& pk = out.host;
  if (pk.max_owned > ms::kPatchOwnedCap || pk.max_local > ms::kPatchLocalCap || pk.max_slots > ms::kPatchSlotCap)
    return fail(-8, "a patch exceeds the compiled shared-memory capacities");
  return 0;
}

// Makes `packed` the context's packing: patch ranges, interior-then-boundary patch order, and the device arrays
// (headers, halo ids, records, slot facets, corner CSR) it built.  The caller has dropped the connectivity state.
int upload_packing(ms_ctx* c, DevPacking&& packed, int32_t n_owned) {
  c->packed = std::move(packed.host);
  const ms::PackedMesh& pk = c->packed;
  const size_t np = pk.patches.size();
  c->v_lo.resize(np + 1);
  for (size_t p = 0; p < np; ++p) c->v_lo[p] = pk.patches[p].v_lo;
  c->v_lo[np] = n_owned;
  {
    std::vector<int32_t> order;
    std::vector<int32_t> boundary;
    for (size_t p = 0; p < np; ++p) {
      const ms::PatchHeader& h = pk.patches[p];
      bool ghost = false;
      for (int32_t j = 0; j < h.n_halo && !ghost; ++j) ghost = pk.halo_ids[size_t(h.halo_off) + size_t(j)] >= n_owned;
      (ghost ? boundary : order).push_back(int32_t(p));
    }
    c->n_interior = int32_t(order.size());
    order.insert(order.end(), boundary.begin(), boundary.end());
    if (int rc = c->d_patch_order.ensure(order.size() + 1)) return rc;
    if (!order.empty()) CU(cudaMemcpy(c->d_patch_order.p, order.data(), order.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  c->n_slots = packed.n_slots;
  c->d_patches.swap(packed.patches);
  c->d_halo.swap(packed.halo);
  c->d_recs.swap(packed.recs);
  c->d_slot_facet.swap(packed.slot_facet);
  c->d_csr_ptr.swap(packed.csr_ptr);
  c->d_csr_idx.swap(packed.csr_idx);
  c->csr_ready = true;
#ifdef MS_SELF_CHECK
  if (std::getenv("MS_SELF_CHECK_INJECT")) {
    // negative control of the self-check: slot 1 of every patch's first round repeats slot 0, so two lanes of one
    // warp read-modify-write the same owned rows at once -- the row locks must report it
    CU(ms::launch_pk_inject(c->d_patches.p, int32_t(np), c->d_recs.p, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
#endif
  return 0;
}

// Per-facet surface tension of the record slots (slot_gamma): the context's host copy gathered through the device
// slot facets.
int upload_slot_gamma(ms_ctx* c) {
  DevBuf<double> gamma;
  if (int rc = gamma.ensure(size_t(c->nf) + 1)) return rc;
  if (int rc = c->d_slot_gamma.ensure(size_t(c->n_slots) + 1)) return rc;
  if (c->nf)
    CU(cudaMemcpyAsync(gamma.p, c->h_gamma.data(), size_t(c->nf) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CU(ms::launch_pk_slot_gamma(c->d_slot_facet.p, c->n_slots, gamma.p, c->d_slot_gamma.p, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // gamma is released on return
  return 0;
}

// Forgets everything derived from the connectivity: it is rebuilt on first use (triangle rows, corner CSR,
// bending-tilt buffers, pipelined-evaluation orders) or must be set again by the caller (leaflet selections, vertex
// normals).  The conjugate-gradient history and a pending projection go too.
void drop_connectivity_state(ms_ctx* c) {
  c->proj.active = false;
  c->bt_ready = false;
  c->tri_ready = false;
  c->csr_ready = false;
  c->pipe_ready = false;
  for (auto& lf : c->leaflet) {
    lf.set = lf.has_fixed = lf.has_minv = false;
    lf.trial.release(); lf.dir.release(); lf.minv.release();
    lf.fixed.release();
  }
  c->vnormals_ready = false;
  c->d_vnormals.release();
  c->d_rowsq.release();
  c->d_lf_corner.release(); c->d_lf_vbuf.release(); c->d_lf_shape.release(); c->d_lf_tilt.release();
  c->d_lf_corner2.release(); c->d_lf_vbuf2.release(); c->d_lf_shape2.release(); c->d_lf_tilt2.release();
  c->d_lf_facet_e.release();
  c->d_cg_prev_g.release();
  c->d_cg_prev_d.release();
}

template <typename T>
std::vector<T> permuted(const T* src, const std::vector<int32_t>& perm) {
  std::vector<T> out(perm.size());
  for (size_t i = 0; i < perm.size(); ++i) out[i] = src[size_t(perm[i])];
  return out;
}

bool per_vertex_array(int which) {
  return which != MS_ARR_SCALARS;
}

template <typename T>
int upload_optional(ms_ctx* c, const T* host, size_t n, bool per_vertex, DevBuf<T>& dst, bool& has) {
  has = host != nullptr;
  if (!host) return 0;
  std::vector<T> tmp;
  if (per_vertex && !c->perm.empty()) {
    tmp = permuted(host, c->perm);
    host = tmp.data();
  }
  if (int rc = dst.ensure(n + 1)) return rc;
  if (n) CU(cudaMemcpy(dst.p, host, n * sizeof(T), cudaMemcpyHostToDevice));
  return 0;
}

}  // namespace

extern "C" {

const char* ms_last_error(void) { return g_err.c_str(); }
int ms_version(void) { return 100; }

int ms_device_count(int* count) {
  if (!count) return fail(-1, "null argument");
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) {
    *count = 0;
    return fail(-100 - int(e), std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
  }
  return 0;
}

int ms_ctx_create(int device, ms_ctx** out) {
  if (!out) return fail(-1, "null argument");
  *out = nullptr;
  int n = 0;
  if (int rc = ms_device_count(&n)) return rc;
  if (n <= 0) return fail(-7, "no CUDA device: the B200 path has no CPU fallback");
  if (device < 0 || device >= n) return fail(-1, "device index out of range");
  CU(cudaSetDevice(device));
  if (device < 64 && !g_configured[device]) {
    CU(ms::configure_kernels());
    g_configured[device] = true;
  }
  std::unique_ptr<ms_ctx> c(new ms_ctx());  // released on every failure path below
  c->device = device;
  CU(cudaEventCreate(&c->ev0));
  CU(cudaEventCreate(&c->ev1));
  if (int rc = c->d_scalars.ensure(MS_SC_COUNT)) return rc;
  CU(cudaMemset(c->d_scalars.p, 0, MS_SC_COUNT * sizeof(double)));
  if (int rc = c->d_dot_partials.ensure(3 * kDotBlocks)) return rc;
#ifdef MS_SELF_CHECK
  if (int rc = c->d_self_check.ensure(4)) return rc;
  CU(cudaMemset(c->d_self_check.p, 0, 4 * sizeof(int)));
#endif
  *out = c.release();
  return 0;
}

int ms_ctx_destroy(ms_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (cudaEvent_t e : c->events)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->pipe_events)
    if (e) cudaEventDestroy(e);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (void* p : c->peers.opened)
    if (p) cudaIpcCloseMemHandle(p);
  delete c;
  return 0;
}

int ms_ctx_set_stream(ms_ctx* c, void* s) {
  if (!c) return fail(-1, "null context");
  c->stream = reinterpret_cast<cudaStream_t>(s);
  return 0;
}

int ms_ctx_set_pack_params(ms_ctx* c, int32_t threads, int32_t max_owned, int32_t max_local) {
  if (!c) return fail(-1, "null context");
  if (threads < 32 || threads > 256 || threads % 32) return fail(-1, "threads must be a multiple of 32 in [32,256]");
  if (max_owned < 1 || max_local < max_owned) return fail(-1, "bad patch sizes");
  if (max_owned > ms::kPatchOwnedCap || max_local > ms::kPatchLocalCap)
    return fail(-1, "patch sizes exceed the compiled shared-memory capacities (512 owned / 896 local)");
  c->pack_params.threads = threads;
  c->pack_params.max_owned = max_owned;
  c->pack_params.max_local = max_local;
  return 0;
}

int ms_ctx_set_pack_tuning(ms_ctx* c, int32_t fill_pct, int32_t repair_sweeps) {
  if (!c) return fail(-1, "null context");
  if (fill_pct < 10 || fill_pct > 100 || repair_sweeps < 0 || repair_sweeps > 8) return fail(-1, "bad tuning values");
  c->pack_params.fill_pct = fill_pct;
  c->pack_params.repair_sweeps = repair_sweeps;
  return 0;
}

int ms_ctx_set_max_ctas(ms_ctx* c, int32_t max_ctas) {
  if (!c) return fail(-1, "null context");
  if (max_ctas < 0) return fail(-1, "max_ctas must be >= 0");
  c->max_ctas = max_ctas;
  return 0;
}

int ms_ctx_set_vertex_order_hint(ms_ctx* c, int32_t nv, const double* pos) {
  if (!c) return fail(-1, "null context");
  c->order_hint.clear();
  if (pos && nv > 0) c->order_hint.assign(pos, pos + 3 * size_t(nv));
  return 0;
}

int ms_ctx_get_permutation(const ms_ctx* c, int32_t* perm_new_to_old) {
  if (!c || !perm_new_to_old) return fail(-1, "null argument");
  if (!c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  for (int32_t i = 0; i < c->nv; ++i) perm_new_to_old[i] = c->perm.empty() ? i : c->perm[size_t(i)];
  return 0;
}

int ms_ctx_set_topology(ms_ctx* c, int32_t nv, int32_t nf, const int32_t* tri,
                        const uint8_t* is_boundary, const uint8_t* body_mask,
                        const uint8_t* fixed_mask) {
  return ms_ctx_set_topology_partition(c, nv, nv, nf, tri, is_boundary, body_mask, fixed_mask);
}

int ms_ctx_set_topology_partition(ms_ctx* c, int32_t nv, int32_t n_owned, int32_t nf,
                                  const int32_t* tri, const uint8_t* is_boundary,
                                  const uint8_t* body_mask, const uint8_t* fixed_mask) {
  NvtxRange range("ms_b200 set_topology (pack + upload)");
  if (int rc = check_ctx(c, false)) return rc;
  if (nv < 0 || nf < 0 || (nf > 0 && !tri) || n_owned < 0 || n_owned > nv)
    return fail(-1, "bad topology arguments");
  c->have_topology = false;
  c->proj.active = false;
  c->n_owned = n_owned;
  // internal vertex order from the hint (single-context meshes only; partitions arrive ordered)
  c->perm.clear();
  if (c->order_hint.size() == 3 * size_t(nv) && n_owned == nv && nv > 1)
    morton_permutation(c->order_hint, nv, c->perm);
  c->order_hint.clear();
  c->order_hint.shrink_to_fit();
  std::vector<int32_t> tri_internal;
  std::vector<uint8_t> boundary_internal, fixed_internal;
  if (!c->perm.empty()) {
    std::vector<int32_t> inv(size_t(nv), 0);
    for (int32_t i = 0; i < nv; ++i) inv[size_t(c->perm[size_t(i)])] = i;
    tri_internal.assign(tri, tri + 3 * size_t(nf));
    for (auto& x : tri_internal)
      if (x >= 0 && x < nv) x = inv[size_t(x)];  // out-of-range indices stay out of range (facet skipped)
    tri = tri_internal.data();
    if (is_boundary) { boundary_internal = permuted(is_boundary, c->perm); is_boundary = boundary_internal.data(); }
    if (fixed_mask) { fixed_internal = permuted(fixed_mask, c->perm); fixed_mask = fixed_internal.data(); }
    if (int rc = c->d_perm.ensure(size_t(nv))) return rc;
    CU(cudaMemcpy(c->d_perm.p, c->perm.data(), size_t(nv) * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (int rc = c->d_stage.ensure(size_t(ms::kSeedStride) * size_t(nv))) return rc;
  }
  // the internal-order rows (and the body flags) go up once and are packed there
  DevBuf<int32_t> tri_dev;
  DevBuf<uint8_t> body_dev;
  if (int rc = tri_dev.ensure(3 * size_t(nf) + 1)) return rc;
  if (nf) CU(cudaMemcpy(tri_dev.p, tri, 3 * size_t(nf) * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (body_mask) {
    if (int rc = body_dev.ensure(size_t(nf) + 1)) return rc;
    if (nf) CU(cudaMemcpy(body_dev.p, body_mask, size_t(nf), cudaMemcpyHostToDevice));
  }
  DevPacking packed;
  if (int rc = pack_rows(c, nv, n_owned, nf, tri_dev.p, body_mask ? body_dev.p : nullptr, packed)) return rc;
  c->nv = nv;
  c->nf = nf;
  c->h_tri.assign(tri, tri + 3 * size_t(nf));
  if (body_mask) c->h_body.assign(body_mask, body_mask + size_t(nf)); else c->h_body.clear();
  c->h_gamma.clear();
  c->has_positions = false;
  drop_connectivity_state(c);
  for (auto& lf : c->leaflet) {  // per-leaflet tilt fields are sized for the previous vertex count
    lf.tilts.release(); lf.tilt_grad.release();
  }
  c->d_tri.swap(tri_dev);
  c->tri_ready = true;  // d_tri holds the rows
  if (int rc = upload_packing(c, std::move(packed), n_owned)) return rc;

  c->has_boundary = is_boundary != nullptr;
  c->has_fixed = fixed_mask != nullptr;
  c->has_body = body_mask != nullptr;
  if (is_boundary) {
    if (int rc = c->d_boundary.ensure(size_t(nv))) return rc;
    if (nv) CU(cudaMemcpy(c->d_boundary.p, is_boundary, size_t(nv), cudaMemcpyHostToDevice));
    std::vector<int32_t> b32(size_t(nv) + 1, 0);
    for (int32_t v = 0; v < nv; ++v) b32[size_t(v)] = is_boundary[v] ? 1 : 0;
    if (int rc = c->d_boundary32.ensure(size_t(nv) + 1)) return rc;
    CU(cudaMemcpy(c->d_boundary32.p, b32.data(), b32.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  if (fixed_mask) {
    if (int rc = c->d_fixed.ensure(size_t(nv))) return rc;
    if (nv) CU(cudaMemcpy(c->d_fixed.p, fixed_mask, size_t(nv), cudaMemcpyHostToDevice));
  }
  const size_t n3 = 3 * size_t(nv);
  if (int rc = c->d_pos.ensure(n3)) return rc;
  if (int rc = c->d_grad.ensure(n3)) return rc;
  if (int rc = c->d_volgrad.ensure(n3)) return rc;
  if (int rc = c->d_seeds.ensure(size_t(ms::kSeedStride) * size_t(nv))) return rc;
  {  // one row of running sums per persistent CTA, pass and sub-launch (the pipelined host evaluation
     // issues up to 32 sub-launches of <= 148 CTAs per pass)
    const size_t rows = 5120;  // >= 148 CTAs x (32 + 1) sub-launches
    if (int rc = c->d_partials_a.ensure(rows * ms::kPartialStride)) return rc;
    if (int rc = c->d_partials_b.ensure(rows * ms::kPartialStride)) return rc;
    CU(cudaMemset(c->d_partials_a.p, 0, rows * ms::kPartialStride * sizeof(double)));
    CU(cudaMemset(c->d_partials_b.p, 0, rows * ms::kPartialStride * sizeof(double)));
  }
  if (n3) {
    CU(cudaMemset(c->d_grad.p, 0, n3 * sizeof(double)));
    CU(cudaMemset(c->d_volgrad.p, 0, n3 * sizeof(double)));
  }
  // per-entity parameter arrays belong to the previous topology
  c->has_gamma = c->has_kappa = c->has_c0 = false;
  c->d_tilts.release();
  c->d_tilt_sq.release();
  c->d_tilt_grad.release();
  c->d_trial.release();
  c->d_dir.release();
  c->d_kvecs.release();
  c->d_avor.release();
  c->d_aeff.release();
  c->d_evert.release();
  c->have_topology = true;
  return 0;
}

int ms_ctx_set_fixed_mask(ms_ctx* c, const uint8_t* fixed_mask) {
  if (int rc = check_ctx(c, true)) return rc;
  // the mask takes part in a pending projection: apply it with the OLD mask first
  if (int rc = flush_projection(c)) return rc;
  const size_t nv = size_t(c->nv);
  c->has_fixed = fixed_mask != nullptr && nv > 0;
  if (!c->has_fixed) return 0;
  std::vector<uint8_t> tmp;
  if (!c->perm.empty()) {
    tmp = permuted(fixed_mask, c->perm);
    fixed_mask = tmp.data();
  }
  if (int rc = c->d_fixed.ensure(nv)) return rc;
  CU(cudaMemcpyAsync(c->d_fixed.p, fixed_mask, nv, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // tmp goes out of scope
  return 0;
}

int ms_ctx_pack_info(const ms_ctx* c, ms_pack_info* info) {
  if (!c || !info) return fail(-1, "null argument");
  if (!c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  const ms::PackedMesh& pk = c->packed;
  info->nv = c->nv;
  info->nf = c->nf;
  info->n_patches = int32_t(pk.patches.size());
  info->threads = pk.params.threads;
  info->max_owned = pk.max_owned;
  info->max_local = pk.max_local;
  info->max_rounds = pk.max_rounds;
  info->max_slots = pk.max_slots;
  info->n_slots = c->n_slots;
  info->n_listed = pk.n_listed;
  info->n_valid = pk.n_valid;
  info->n_halo = int64_t(pk.halo_ids.size());
  info->n_round_slots = pk.n_round_slots;
  info->n_lane_conflicts = pk.n_lane_conflicts;
  info->n_hw_groups = pk.n_hw_groups;
  info->n_hw_excess = pk.n_hw_excess;
  return 0;
}

int ms_ctx_get_packing(const ms_ctx* c, void* headers, int32_t* halo_ids, void* recs, int32_t* slot_facet) {
  if (int rc = check_ctx(c, true)) return rc;
  const ms::PackedMesh& pk = c->packed;
  if (headers && !pk.patches.empty()) std::memcpy(headers, pk.patches.data(), pk.patches.size() * sizeof(ms::PatchHeader));
  if (halo_ids && !pk.halo_ids.empty()) std::memcpy(halo_ids, pk.halo_ids.data(), pk.halo_ids.size() * sizeof(int32_t));
  const size_t ns = size_t(c->n_slots);
  if (recs && ns) CU(cudaMemcpyAsync(recs, c->d_recs.p, ns * sizeof(ms::FacetRec), cudaMemcpyDeviceToHost, c->stream));
  if (slot_facet && ns)
    CU(cudaMemcpyAsync(slot_facet, c->d_slot_facet.p, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int ms_ctx_patch_ranges(const ms_ctx* c, int32_t* v_lo) {
  if (!c || !v_lo) return fail(-1, "null argument");
  if (!c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  std::memcpy(v_lo, c->v_lo.data(), c->v_lo.size() * sizeof(int32_t));
  return 0;
}

int ms_ctx_halo_rows(const ms_ctx* c, int32_t patch_begin, int32_t patch_count, int32_t own_lo,
                     int32_t own_hi, int32_t* out, int64_t* n) {
  if (!c || !n) return fail(-1, "null argument");
  if (!c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  const ms::PackedMesh& pk = c->packed;
  if (patch_begin < 0 || patch_count < 0 || size_t(patch_begin) + size_t(patch_count) > pk.patches.size())
    return fail(-3, "patch range out of bounds");
  std::vector<uint8_t> seen(size_t(c->nv), 0);
  for (int32_t p = patch_begin; p < patch_begin + patch_count; ++p) {
    const ms::PatchHeader& h = pk.patches[size_t(p)];
    for (int32_t j = 0; j < h.n_halo; ++j) {
      const int32_t v = pk.halo_ids[size_t(h.halo_off) + size_t(j)];
      if (v < own_lo || v >= own_hi) seen[size_t(v)] = 1;
    }
  }
  int64_t k = 0;
  for (int32_t v = 0; v < c->nv; ++v)
    if (seen[size_t(v)]) {
      if (out) out[k] = v;
      ++k;
    }
  *n = k;
  return 0;
}

int ms_ctx_set_surface_tension(ms_ctx* c, const double* gamma, double gamma_uniform) {
  if (int rc = check_ctx(c, true)) return rc;
  c->gamma_u = gamma_uniform;
  c->has_gamma = false;
  c->h_gamma.clear();
  if (!gamma) return 0;
  c->h_gamma.assign(gamma, gamma + size_t(c->nf));
  if (int rc = upload_slot_gamma(c)) return rc;
  c->has_gamma = true;
  return 0;
}

int ms_ctx_set_bending_params(ms_ctx* c, const double* kappa, const double* c0, double kappa_u,
                              double c0_u) {
  if (int rc = check_ctx(c, true)) return rc;
  c->kappa_u = kappa_u;
  c->c0_u = c0_u;
  c->has_kappa = kappa != nullptr;
  c->has_c0 = c0 != nullptr;
  const size_t nv = size_t(c->nv);
  std::vector<double> tmp;
  if (kappa) {
    if (!c->perm.empty()) { tmp = permuted(kappa, c->perm); kappa = tmp.data(); }
    if (int rc = c->d_kappa.ensure(nv)) return rc;
    if (nv) CU(cudaMemcpy(c->d_kappa.p, kappa, nv * sizeof(double), cudaMemcpyHostToDevice));
  }
  if (c0) {
    if (!c->perm.empty()) { tmp = permuted(c0, c->perm); c0 = tmp.data(); }
    if (int rc = c->d_c0.ensure(nv)) return rc;
    if (nv) CU(cudaMemcpy(c->d_c0.p, c0, nv * sizeof(double), cudaMemcpyHostToDevice));
  }
  return 0;
}

int ms_ctx_set_tilt_rigidity(ms_ctx* c, double k_tilt) {
  if (!c) return fail(-1, "null context");
  c->k_tilt = k_tilt;
  return 0;
}

int ms_ctx_upload(ms_ctx* c, int which, const double* host, int64_t offset, int64_t count) {
  if (int rc = check_ctx(c, true)) return rc;
  if (which == MS_ARR_GRAD) c->proj.active = false;
  // gC takes part in a pending projection: apply it with the OLD gC first
  if (which == MS_ARR_VOLGRAD)
    if (int rc = flush_projection(c)) return rc;
  if (!host && count > 0) return fail(-1, "null host pointer");
  if (int rc = ensure_array(c, which)) return rc;
  int64_t len = 0;
  double* d = array_ptr(c, which, &len);
  if (!d && len > 0) return fail(-1, "array is not allocated");
  if (offset < 0 || count < 0 || offset + count > len) return fail(-1, "upload range out of bounds");
  if (which == MS_ARR_POSITIONS) c->has_positions = true;
  if (!c->perm.empty() && per_vertex_array(which) && count) {
    // the caller's rows are in its own vertex order: land in the staging buffer, gather into internal order
    if (offset != 0 || count != len) return fail(-1, "partial uploads are not available on an internally reordered mesh");
    CU(cudaMemcpyAsync(c->d_stage.p, host, size_t(count) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CU(ms::launch_gather_rows(c->d_stage.p, int(len / c->nv), c->d_perm.p, c->nv, d, c->stream));
    return 0;
  }
  if (count) CU(cudaMemcpyAsync(d + offset, host, size_t(count) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int ms_ctx_get_array(ms_ctx* c, int which, double* host, int64_t offset, int64_t count) {
  if (int rc = check_ctx(c, true)) return rc;
  if (which == MS_ARR_GRAD)
    if (int rc = flush_projection(c)) return rc;
  if (!host && count > 0) return fail(-1, "null host pointer");
  int64_t len = 0;
  double* d = array_ptr(c, which, &len);
  if (!d && len > 0) return fail(-1, "array has not been produced yet");
  if (offset < 0 || count < 0 || offset + count > len) return fail(-1, "download range out of bounds");
  if (!c->perm.empty() && per_vertex_array(which) && count) {
    if (offset != 0 || count != len) return fail(-1, "partial downloads are not available on an internally reordered mesh");
    if (int rc = download_rows(c, d, host, int(len / c->nv))) return rc;
  } else if (count) {
    CU(cudaMemcpyAsync(host, d + offset, size_t(count) * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

void* ms_ctx_device_ptr(ms_ctx* c, int which) {
  if (!c || !c->have_topology) return nullptr;
  if (use_device(c)) return nullptr;
  if (ensure_array(c, which)) return nullptr;
  // the caller sees the projected gradient, and may write gC only after the projection that uses it
  if ((which == MS_ARR_GRAD || which == MS_ARR_VOLGRAD) && flush_projection(c)) return nullptr;
  if (which == MS_ARR_POSITIONS) c->has_positions = true;             // the caller may write through it
  int64_t len = 0;
  return array_ptr(c, which, &len);
}

int64_t ms_ctx_array_len(const ms_ctx* c, int which) {
  if (!c || !c->have_topology) return 0;
  int64_t len = 0;
  array_ptr(const_cast<ms_ctx*>(c), which, &len);
  return len;
}

int ms_ctx_set_positions(ms_ctx* c, const double* pos_host) {
  return ms_ctx_upload(c, MS_ARR_POSITIONS, pos_host, 0, 3 * int64_t(c ? c->nv : 0));
}

int ms_ctx_set_tilts(ms_ctx* c, const double* tilts_host) {
  return ms_ctx_upload(c, MS_ARR_TILTS, tilts_host, 0, 3 * int64_t(c ? c->nv : 0));
}

// b_mask of the fixed-order sum: which scalar slots come from pass B's rows (see reduce_rows)
static unsigned reduce_b_mask(const ms_eval_opts* o) {
  const bool ran_a = needs_bending(o) || !o->want_grad;
  unsigned b_mask = 0;
  if (o->want_grad) {
    b_mask = (1u << MS_SC_G_G) | (1u << MS_SC_G_GC) | (1u << MS_SC_GC_GC);
    if (!ran_a) b_mask = 0xfffu;
  }
  return b_mask;
}

// the constraint / fixed-row projection an evaluation asks for
static void projection_of(const ms_ctx* c, const ms_eval_opts* o, bool& use_gc, bool& use_fixed) {
  use_gc = o->want_grad && o->constraint_mode >= 0 && (o->modules & MS_MOD_VOLUME);
  use_fixed = o->want_grad && o->apply_fixed && c->has_fixed;
}

// fused finalisation: the last CTA of `a`'s launch reduces the rows and writes the KKT coefficient
static int attach_finalize(ms_ctx* c, const ms_eval_opts* o, ms::PatchLaunch& a) {
  if (!c->d_ticket.p) {
    if (int rc = c->d_ticket.ensure(4)) return rc;
    CU(cudaMemsetAsync(c->d_ticket.p, 0, 4 * sizeof(unsigned int), c->stream));
  }
  const bool ran_a = needs_bending(o) || !o->want_grad;
  const int rows = ms::patch_grid(a);
  bool use_gc, use_fixed;
  projection_of(c, o, use_gc, use_fixed);
  a.fin.ticket = c->d_ticket.p;
  a.fin.partials_a = c->d_partials_a.p;
  a.fin.partials_b = c->d_partials_b.p;
  a.fin.rows_a = ran_a ? rows : 0;
  a.fin.rows_b = o->want_grad ? rows : 0;
  a.fin.b_mask = reduce_b_mask(o);
  a.fin.constraint_mode = o->want_grad ? o->constraint_mode : -2;
  a.fin.has_gc = use_gc ? 1 : 0;
  a.fin.k_vol = o->k_vol;
  a.fin.v_target = o->v_target;
  a.fin.scalars = c->d_scalars.p;
  return 0;
}

static int eval_pass_a_impl(ms_ctx* c, const ms_eval_opts* o, bool finalize) {
  NvtxRange range("ms_b200 pass A");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o) return fail(-1, "null options");
  ms::PatchLaunch a;
  if (int rc = fill_launch(c, o, a)) return rc;
  // Pass A is needed for the bending seeds and for energies; surface/volume-only
  // gradient evaluations do everything in pass B.
  a.partials = c->d_partials_a.p;
  c->ran_pass_a = needs_bending(o) || !o->want_grad;
  if (finalize)
    if (int rc = attach_finalize(c, o, a)) return rc;
  if (c->ran_pass_a) CU(ms::launch_pass_a(a, c->stream));
  if (has_bt(o)) {
    ms::BtMesh m;
    if (int rc = bt_prepare(c, m)) return rc;
    m.pos = a.pos;
    CU(ms::launch_bt_stage(m, 1.0, c->d_kvecs.p, c->d_avor.p, c->d_aeff.p, c->d_bt_corner.p, c->d_seeds.p,
                           c->d_bt_base.p, c->d_bt_facet_e.p, c->d_bt_e.p, wants_tilt_grad(o), c->stream));
  }
  return 0;
}

static int eval_pass_b_impl(ms_ctx* c, const ms_eval_opts* o, bool finalize) {
  NvtxRange range("ms_b200 pass B");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o) return fail(-1, "null options");
  // a tilt-only evaluation (want_grad == 0, want_tilt_grad == 1) still needs pass B for the tilt
  // magnitude module, whose tilt gradient comes from the barycentric areas accumulated there
  const bool run_b = o->want_grad || (o->want_tilt_grad && (o->modules & MS_MOD_TILT));
  ms::PatchLaunch a;
  if (int rc = fill_launch(c, o, a)) return rc;
  a.partials = c->d_partials_b.p;
  if (run_b) {
    c->proj.active = false;  // MS_ARR_GRAD is overwritten with a new raw gradient
    if ((o->modules & MS_MOD_TILT) && !a.tilt_grad) {
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD)) return rc;
      a.tilt_grad = c->d_tilt_grad.p;
    }
    if (finalize)
      if (int rc = attach_finalize(c, o, a)) return rc;
    CU(ms::launch_pass_b(a, needs_bending(o), !needs_bending(o), c->stream));
  }
  if (has_bt(o) && wants_tilt_grad(o)) {
    ms::BtMesh m;
    if (int rc = bt_prepare(c, m)) return rc;
    m.pos = a.pos;
    CU(ms::launch_bt_tilt_gather(m, c->d_bt_corner.p, c->d_tilt_grad.p, run_b && (o->modules & MS_MOD_TILT), c->stream));
  }
  return 0;
}

int ms_ctx_eval_pass_a(ms_ctx* c, const ms_eval_opts* o) { return eval_pass_a_impl(c, o, false); }
int ms_ctx_eval_pass_b(ms_ctx* c, const ms_eval_opts* o) { return eval_pass_b_impl(c, o, false); }

int ms_ctx_eval_finish(ms_ctx* c, const ms_eval_opts* o) {
  if (int rc = ms_ctx_eval_reduce(c, o)) return rc;
  return ms_ctx_eval_project(c, o);
}

static int reduce_rows(ms_ctx* c, const ms_eval_opts* o, int rows_a, int rows_b) {
  // energies, area, volume come from pass A when it ran, else from pass B; <g,g>, <g,gC>, <gC,gC>
  // and the tilt energy come from pass B when a gradient was requested -- one fixed-order sum
  const bool ran_a = needs_bending(o) || !o->want_grad;
  const unsigned b_mask = reduce_b_mask(o);
  CU(ms::launch_reduce_partials(c->d_partials_a.p, ran_a ? rows_a : 0, c->d_partials_b.p, o->want_grad ? rows_b : 0,
                                b_mask, c->d_scalars.p, c->stream));
  if (has_bt(o)) CU(ms::launch_bt_finalize(c->d_bt_e.p, c->d_scalars.p, c->stream));
  return 0;
}

int ms_ctx_eval_reduce(ms_ctx* c, const ms_eval_opts* o) {
  NvtxRange range("ms_b200 reduce");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o) return fail(-1, "null options");
  ms::PatchLaunch a;
  if (int rc = fill_launch(c, o, a)) return rc;
  // a split evaluation (interior + boundary launches) leaves its sums in rows [0, grid_i + grid_b)
  int rows = ms::patch_grid(a);
  if (o->patch_count == MS_PATCHES_INTERIOR || o->patch_count == MS_PATCHES_BOUNDARY) {
    ms::PatchLaunch inner = a, outer = a;
    inner.patch_count = c->n_interior;
    outer.patch_count = int(c->packed.patches.size()) - c->n_interior;
    rows = ms::patch_grid(inner) + ms::patch_grid(outer);
  }
  return reduce_rows(c, o, rows, rows);
}

int ms_ctx_eval_project(ms_ctx* c, const ms_eval_opts* o) {
  NvtxRange range("ms_b200 kkt coefficient");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o) return fail(-1, "null options");
  if (!o->want_grad) return 0;  // energy-only evaluation: a pending projection (and its coefficient) stays as it is
  bool use_gc, use_fixed;
  projection_of(c, o, use_gc, use_fixed);
  // one thread: scalars[SC_COEF], scalars[SC_LAMBDA]; the projection itself is applied by the consumer of the
  // gradient (direction, dot products) or materialised on first access (flush_projection)
  CU(ms::launch_kkt_coefficient(c->d_scalars.p, o->constraint_mode, use_gc ? 1 : 0, o->k_vol, o->v_target, c->stream));
  c->proj.active = use_gc || use_fixed;
  c->proj.use_gc = use_gc;
  c->proj.use_fixed = use_fixed;
  return 0;
}

int ms_ctx_eval_stage(ms_ctx* c, const ms_eval_opts* o, int32_t stage);

int ms_ctx_eval_async(ms_ctx* c, const ms_eval_opts* o) {
  if (!c || !o) return fail(-1, "null argument");
  // whole-mesh evaluations finalise inside the last pass (last-CTA ticket): no reduce / project launches
  const bool fuse = o->patch_count == -1 && c->have_topology && !c->packed.patches.empty();
  if (!fuse) {
    if (int rc = ms_ctx_eval_pass_a(c, o)) return rc;
    if (int rc = ms_ctx_eval_pass_b(c, o)) return rc;
    return ms_ctx_eval_finish(c, o);
  }
  if (int rc = ms_ctx_eval_stage(c, o, 0)) return rc;
  return ms_ctx_eval_stage(c, o, 1);
}

int ms_ctx_eval_stage(ms_ctx* c, const ms_eval_opts* o, int32_t stage) {
  if (!c || !o) return fail(-1, "null argument");
  if (stage < 0 || stage > 1) return fail(-1, "stage must be 0 (pass A) or 1 (pass B + finalisation)");
  if (o->patch_count != -1 || !c->have_topology || c->packed.patches.empty())
    return fail(-1, "ms_ctx_eval_stage evaluates whole, non-empty meshes");
  if (stage == 0) return eval_pass_a_impl(c, o, !o->want_grad);
  if (int rc = eval_pass_b_impl(c, o, o->want_grad != 0)) return rc;
  if (has_bt(o)) CU(ms::launch_bt_finalize(c->d_bt_e.p, c->d_scalars.p, c->stream));
  if (o->want_grad) {
    bool use_gc, use_fixed;
    projection_of(c, o, use_gc, use_fixed);
    c->proj.active = use_gc || use_fixed;
    c->proj.use_gc = use_gc;
    c->proj.use_fixed = use_fixed;
  }
  return 0;
}

int ms_ctx_self_check(ms_ctx* c, int32_t* counters3) {
  if (int rc = check_ctx(c, false)) return rc;
  if (!counters3) return fail(-1, "null argument");
#ifdef MS_SELF_CHECK
  if (!c->d_self_check.p) {
    if (int rc = c->d_self_check.ensure(4)) return rc;
    CU(cudaMemset(c->d_self_check.p, 0, 4 * sizeof(int)));
  }
  CU(cudaMemcpyAsync(counters3, c->d_self_check.p, 3 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
#else
  counters3[0] = counters3[1] = counters3[2] = -1;
  return fail(-10, "this library was built without MS_SELF_CHECK (build membrane_solver_b200/libms_b200_checked.so)");
#endif
}

int ms_ctx_read_scalars(ms_ctx* c, double* scalars16) {
  if (int rc = check_ctx(c, false)) return rc;
  if (!scalars16) return fail(-1, "null argument");
  CU(cudaMemcpyAsync(scalars16, c->d_scalars.p, MS_SC_COUNT * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int ms_ctx_eval(ms_ctx* c, const ms_eval_opts* o, double* scalars16) {
  if (int rc = ms_ctx_eval_async(c, o)) return rc;
  return ms_ctx_read_scalars(c, scalars16);
}

// ---- leaflet tilt modules ------------------------------------------------------------------------------
int ms_ctx_set_leaflet(ms_ctx* c, int32_t leaflet, const ms_leaflet_desc* d) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!d || leaflet < 0 || leaflet > 2) return fail(-1, "bad leaflet arguments");
  if (c->n_owned != c->nv) return fail(-5, "leaflet modules are not available on a partitioned context");
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  const size_t nv = size_t(c->nv), nf = size_t(c->nf);
  L.set = false;
  if (int rc = upload_optional(c, d->facet_keep, nf, false, L.keep, L.has_keep)) return rc;
  if (int rc = upload_optional(c, d->interior, nv, true, L.interior, L.has_interior)) return rc;
  if (int rc = upload_optional(c, d->base_zero, nv, true, L.base_zero, L.has_base_zero)) return rc;
  if (int rc = upload_optional(c, d->kappa, nv, true, L.kappa, L.has_kappa)) return rc;
  if (int rc = upload_optional(c, d->c0, nv, true, L.c0, L.has_c0)) return rc;
  if (int rc = upload_optional(c, d->tilt_row_weight, nv, true, L.weight, L.has_weight)) return rc;
  if (int rc = upload_optional(c, d->facet_consistent, nf, false, L.consistent, L.has_consistent)) return rc;
  L.kappa_u = d->kappa_default;
  L.c0_u = d->c0_default;
  L.k_tilt = d->k_tilt;
  L.k_smooth = d->k_smooth;
  L.sign = d->div_sign;
  L.consistent_u = d->consistent_default;
  L.set = true;
  return 0;
}

// 15 result doubles (3 leaflet slots x {E_bending_tilt, E_tilt, E_tilt_smoothness, |g|^2, r.z}) in one block, so
// that one copy brings everything back, followed by the scratch of the two-stage sums
static int ensure_leaflet_results(ms_ctx* c) {
  if (c->d_lf_e.p) return 0;
  const size_t n = 16 + 3 * size_t(ms::kSumBlocks);
  if (int rc = c->d_lf_e.ensure(n)) return rc;
  CU(cudaMemset(c->d_lf_e.p, 0, n * sizeof(double)));
  return 0;
}

static void fill_leaflet_mesh(ms_ctx* c, ms_ctx::Leaflet& L, bool use_trial, ms::LeafletMesh& m) {
  m.nv = c->nv;
  m.nf = c->nf;
  m.tri = c->d_tri.p;
  m.pos = use_trial ? c->d_trial.p : c->d_pos.p;
  m.tilts = L.tilts.p;
  m.keep = L.has_keep ? L.keep.p : nullptr;
  m.is_boundary = c->has_boundary ? c->d_boundary.p : nullptr;
  m.interior = L.has_interior ? L.interior.p : nullptr;
  m.base_zero = L.has_base_zero ? L.base_zero.p : nullptr;
  m.kappa = L.has_kappa ? L.kappa.p : nullptr;
  m.c0 = L.has_c0 ? L.c0.p : nullptr;
  m.kappa_u = L.kappa_u;
  m.c0_u = L.c0_u;
  m.row_weight = L.has_weight ? L.weight.p : nullptr;
  m.consistent = L.has_consistent ? L.consistent.p : nullptr;
  m.consistent_u = L.consistent_u;
  m.k_tilt = L.k_tilt;
  m.k_smooth = L.k_smooth;
  m.sign = L.sign;
  m.csr_ptr = c->d_csr_ptr.p;
  m.csr_idx = c->d_csr_idx.p;
}

int ms_ctx_eval_leaflet(ms_ctx* c, int32_t leaflet, uint32_t modules, int32_t want_grad, int32_t want_tilt_grad,
                        uint32_t accumulate, int32_t use_trial, double* energies3) {
  if (int rc = check_ctx(c, true)) return rc;
  if (want_grad)
    if (int rc = flush_projection(c)) return rc;
  if (leaflet < 0 || leaflet > 2) return fail(-1, "bad leaflet index");
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.set) return fail(-4, "ms_ctx_set_leaflet has not been called for this leaflet (or the topology changed)");
  if (modules & ~uint32_t(MS_MOD_TILT | MS_MOD_BENDING_TILT | MS_MOD_TILT_SMOOTHNESS))
    return fail(-1, "leaflet modules are MS_MOD_TILT, MS_MOD_BENDING_TILT and MS_MOD_TILT_SMOOTHNESS");
  const int which_t = leaflet == 0 ? MS_ARR_TILTS_IN : (leaflet == 1 ? MS_ARR_TILTS_OUT : MS_ARR_TILTS_FIELD);
  const int which_g = leaflet == 0 ? MS_ARR_TILT_GRAD_IN : (leaflet == 1 ? MS_ARR_TILT_GRAD_OUT : MS_ARR_TILT_GRAD_FIELD);
  if (!L.tilts.p && c->nv > 0) return fail(-4, "the leaflet's tilt field has not been uploaded (MS_ARR_TILTS_IN / _OUT)");
  if (use_trial && !c->d_trial.p) return fail(-4, "use_trial set but no trial positions exist (ms_ctx_make_trial)");
  (void)which_t;
  if (want_tilt_grad)
    if (int rc = ensure_array(c, which_g)) return rc;
  ms::BtMesh bm;  // triangle rows + corner CSR are shared with the single-field coupling stage
  if (int rc = bt_prepare(c, bm)) return rc;
  const size_t nv = size_t(c->nv), nf = size_t(c->nf);
  if (int rc = c->d_lf_corner.ensure(3 * ms::kLfCornerA * nf + 1)) return rc;
  if (int rc = c->d_lf_vbuf.ensure(ms::kLfVertex * nv + 1)) return rc;
  if (int rc = c->d_lf_shape.ensure(9 * nf + 1)) return rc;
  if (int rc = c->d_lf_tilt.ensure(9 * nf + 1)) return rc;
  if (int rc = c->d_lf_facet_e.ensure(3 * nf + 1)) return rc;
  if (int rc = ensure_leaflet_results(c)) return rc;
  double* lf_e = c->d_lf_e.p + 5 * size_t(leaflet);         // result row of this leaflet: 3 energies, |g|^2, r.z
  double* lf_scratch = c->d_lf_e.p + 16;                     // reduction scratch behind the 15 results
  ms::LeafletMesh m;
  fill_leaflet_mesh(c, L, use_trial != 0, m);
  static const bool fused_off = std::getenv("MS_LEAFLET_NO_FUSE") != nullptr;
  if (!fused_off && c->lf_fused_ok && c->nf <= ms::kLfFusedMaxItems && c->nv <= ms::kLfFusedMaxItems && c->nf > 0) {
    // a mesh this small is launch-latency bound: all phases in one cooperative launch
    if (!c->d_lf_ticket.p) {
      if (int rc = c->d_lf_ticket.ensure(1)) return rc;
      CU(cudaMemset(c->d_lf_ticket.p, 0, sizeof(unsigned long long)));
      c->lf_ticket_base = 0;
      if (int rc = c->d_lf_block_e.ensure(6 * ms::kLfFusedMaxBlocks)) return rc;
    }
    cudaError_t e = ms::launch_leaflet_fused(
        m, (modules & MS_MOD_BENDING_TILT) != 0, (modules & MS_MOD_TILT) != 0, (modules & MS_MOD_TILT_SMOOTHNESS) != 0,
        c->d_lf_corner.p, c->d_lf_vbuf.p, c->d_lf_shape.p, c->d_lf_tilt.p, c->d_lf_block_e.p, ms::kLfFusedMaxBlocks, lf_e,
        want_grad ? c->d_grad.p : nullptr, (accumulate & MS_ACC_GRAD) != 0, want_tilt_grad ? L.tilt_grad.p : nullptr,
        (accumulate & MS_ACC_TILT_GRAD) != 0, c->d_lf_ticket.p, &c->lf_ticket_base, c->stream);
    if (e == cudaSuccess) {
      if (energies3) {
        CU(cudaMemcpyAsync(energies3, lf_e, 3 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
      }
      return 0;
    }
    cudaGetLastError();       // not launchable cooperatively here: the sweeps as separate launches from now on
    c->lf_fused_ok = false;
  }
  CU(ms::launch_leaflet(m, (modules & MS_MOD_BENDING_TILT) != 0, (modules & MS_MOD_TILT) != 0,
                        (modules & MS_MOD_TILT_SMOOTHNESS) != 0, c->d_lf_corner.p,
                        c->d_lf_vbuf.p, c->d_lf_shape.p, c->d_lf_tilt.p, c->d_lf_facet_e.p, lf_e, lf_scratch,
                        want_grad ? c->d_grad.p : nullptr, (accumulate & MS_ACC_GRAD) != 0,
                        want_tilt_grad ? L.tilt_grad.p : nullptr, (accumulate & MS_ACC_TILT_GRAD) != 0, c->stream));
  if (energies3) {
    CU(cudaMemcpyAsync(energies3, lf_e, 3 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

int ms_ctx_set_leaflet_fixed(ms_ctx* c, int32_t leaflet, const uint8_t* fixed_rows) {
  if (int rc = check_ctx(c, true)) return rc;
  if (leaflet < 0 || leaflet > 2) return fail(-1, "bad leaflet index");
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  return upload_optional(c, fixed_rows, size_t(c->nv), true, L.fixed, L.has_fixed);
}

int ms_ctx_update_vertex_normals(ms_ctx* c) {
  if (int rc = check_ctx(c, true)) return rc;
  if (c->n_owned != c->nv) return fail(-5, "not available on a partitioned context");
  if (int rc = ensure_corner_csr(c)) return rc;
  if (int rc = c->d_vnormals.ensure(3 * size_t(c->nv) + 1)) return rc;
  CU(ms::launch_vertex_normals(c->nv, c->d_tri.p, c->d_csr_ptr.p, c->d_csr_idx.p, c->d_pos.p, c->d_vnormals.p, c->stream));
  c->vnormals_ready = true;
  return 0;
}

static int leaflet_ready(ms_ctx* c, int32_t leaflet, bool need_normals) {
  if (int rc = check_ctx(c, true)) return rc;
  if (leaflet < 0 || leaflet > 2) return fail(-1, "bad leaflet index");
  if (!c->leaflet[leaflet].tilts.p && c->nv > 0) return fail(-4, "the leaflet's tilt field has not been uploaded");
  if (need_normals && !c->vnormals_ready) return fail(-4, "ms_ctx_update_vertex_normals has not been called for this topology");
  return 0;
}

int ms_ctx_leaflet_project_tilts(ms_ctx* c, int32_t leaflet) {
  if (int rc = leaflet_ready(c, leaflet, true)) return rc;
  CU(ms::launch_project_tangent(c->nv, c->d_vnormals.p, c->leaflet[leaflet].tilts.p, c->stream));
  return 0;
}

int ms_ctx_leaflet_gradient_norm2(ms_ctx* c, int32_t leaflet, double* norm2) {
  if (int rc = leaflet_ready(c, leaflet, false)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.tilt_grad.p && c->nv > 0) return fail(-4, "no tilt gradient exists for this leaflet (ms_ctx_eval_leaflet)");
  if (int rc = c->d_rowsq.ensure(size_t(c->nv) + 1)) return rc;
  if (int rc = ensure_leaflet_results(c)) return rc;
  double* out = c->d_lf_e.p + 5 * size_t(leaflet) + 3;
  CU(ms::launch_masked_norm2(c->nv, L.tilt_grad.p, L.has_fixed ? L.fixed.p : nullptr, c->d_rowsq.p, out,
                             c->d_lf_e.p + 16, c->stream));
  if (norm2) {
    CU(cudaMemcpyAsync(norm2, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

int ms_ctx_eval_leaflet_pair(ms_ctx* c, uint32_t modules, int32_t want_grad, int32_t want_tilt_grad, uint32_t accumulate,
                             int32_t use_trial) {
  if (int rc = check_ctx(c, true)) return rc;
  if (want_grad)
    if (int rc = flush_projection(c)) return rc;
  ms_ctx::Leaflet& A = c->leaflet[0];
  ms_ctx::Leaflet& B = c->leaflet[1];
  static const bool fused_off = std::getenv("MS_LEAFLET_NO_FUSE") != nullptr;
  const bool small = c->nf <= ms::kLfFusedMaxItems / 2 && c->nv <= ms::kLfFusedMaxItems / 2 && c->nf > 0;
  if (!fused_off && c->lf_fused_ok && small && A.set && B.set && A.tilts.p && B.tilts.p &&
      !(modules & ~uint32_t(MS_MOD_TILT | MS_MOD_BENDING_TILT | MS_MOD_TILT_SMOOTHNESS)) &&
      !(use_trial && !c->d_trial.p)) {
    if (want_tilt_grad) {
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD_IN)) return rc;
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD_OUT)) return rc;
    }
    ms::BtMesh bm;
    if (int rc = bt_prepare(c, bm)) return rc;
    const size_t nv = size_t(c->nv), nf = size_t(c->nf);
    if (int rc = c->d_lf_corner.ensure(3 * ms::kLfCornerA * nf + 1)) return rc;
    if (int rc = c->d_lf_vbuf.ensure(ms::kLfVertex * nv + 1)) return rc;
    if (int rc = c->d_lf_shape.ensure(9 * nf + 1)) return rc;
    if (int rc = c->d_lf_tilt.ensure(9 * nf + 1)) return rc;
    if (int rc = c->d_lf_corner2.ensure(3 * ms::kLfCornerA * nf + 1)) return rc;
    if (int rc = c->d_lf_vbuf2.ensure(ms::kLfVertex * nv + 1)) return rc;
    if (int rc = c->d_lf_shape2.ensure(9 * nf + 1)) return rc;
    if (int rc = c->d_lf_tilt2.ensure(9 * nf + 1)) return rc;
    if (int rc = ensure_leaflet_results(c)) return rc;
    if (!c->d_lf_ticket.p) {
      if (int rc = c->d_lf_ticket.ensure(1)) return rc;
      CU(cudaMemset(c->d_lf_ticket.p, 0, sizeof(unsigned long long)));
      c->lf_ticket_base = 0;
    }
    if (int rc = c->d_lf_block_e.ensure(6 * ms::kLfFusedMaxBlocks)) return rc;
    ms::LeafletMesh m0, m1;
    fill_leaflet_mesh(c, A, use_trial != 0, m0);
    fill_leaflet_mesh(c, B, use_trial != 0, m1);
    double* const corner[2] = {c->d_lf_corner.p, c->d_lf_corner2.p};
    double* const vbuf[2] = {c->d_lf_vbuf.p, c->d_lf_vbuf2.p};
    double* const shape[2] = {c->d_lf_shape.p, c->d_lf_shape2.p};
    double* const tilt[2] = {c->d_lf_tilt.p, c->d_lf_tilt2.p};
    double* const e_out[2] = {c->d_lf_e.p, c->d_lf_e.p + 5};
    double* const tg[2] = {want_tilt_grad ? A.tilt_grad.p : nullptr, want_tilt_grad ? B.tilt_grad.p : nullptr};
    cudaError_t e = ms::launch_leaflet_fused_pair(
        m0, m1, (modules & MS_MOD_BENDING_TILT) != 0, (modules & MS_MOD_TILT) != 0, (modules & MS_MOD_TILT_SMOOTHNESS) != 0,
        corner, vbuf, shape, tilt, e_out, tg, c->d_lf_block_e.p, ms::kLfFusedMaxBlocks, want_grad ? c->d_grad.p : nullptr,
        (accumulate & MS_ACC_GRAD) != 0, (accumulate & MS_ACC_TILT_GRAD) != 0, c->d_lf_ticket.p, &c->lf_ticket_base,
        c->stream);
    if (e == cudaSuccess) return 0;
    cudaGetLastError();
    c->lf_fused_ok = false;
  }
  // one leaflet after the other: the inner leaflet's shape gradient first, the outer one's added to it
  if (int rc = ms_ctx_eval_leaflet(c, MS_LEAFLET_IN, modules, want_grad, want_tilt_grad, accumulate, use_trial, nullptr))
    return rc;
  return ms_ctx_eval_leaflet(c, MS_LEAFLET_OUT, modules, want_grad, want_tilt_grad,
                             accumulate | (want_grad ? MS_ACC_GRAD : 0u), use_trial, nullptr);
}

int ms_ctx_leaflet_results(ms_ctx* c, double* out15) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!out15) return fail(-1, "null argument");
  if (int rc = ensure_leaflet_results(c)) return rc;
  CU(cudaMemcpyAsync(out15, c->d_lf_e.p, 15 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int ms_ctx_leaflet_make_trial(ms_ctx* c, int32_t leaflet, double step, int32_t along_direction) {
  if (int rc = leaflet_ready(c, leaflet, true)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.tilt_grad.p && c->nv > 0) return fail(-4, "no tilt gradient exists for this leaflet (ms_ctx_eval_leaflet)");
  if (along_direction && !L.dir.p && c->nv > 0) return fail(-4, "no CG direction exists (ms_ctx_leaflet_cg_direction)");
  if (int rc = L.trial.ensure(3 * size_t(c->nv) + 1)) return rc;
  // t - step * g  or  t + step * d
  CU(ms::launch_tilt_trial(c->nv, L.tilts.p, along_direction ? L.dir.p : L.tilt_grad.p, c->d_vnormals.p,
                           L.has_fixed ? L.fixed.p : nullptr, along_direction ? -step : step, L.trial.p, c->stream));
  return 0;
}

int ms_ctx_leaflet_build_preconditioner(ms_ctx* c, int32_t leaflet, double k_smooth, int32_t kept_facets_only) {
  if (int rc = leaflet_ready(c, leaflet, false)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.set) return fail(-4, "ms_ctx_set_leaflet has not been called for this leaflet");
  ms::BtMesh bm;
  if (int rc = bt_prepare(c, bm)) return rc;
  if (int rc = L.minv.ensure(size_t(c->nv) + 1)) return rc;
  ms::LeafletMesh m;
  fill_leaflet_mesh(c, L, false, m);
  CU(ms::launch_leaflet_jacobi(m, kept_facets_only != 0, k_smooth, L.has_fixed ? L.fixed.p : nullptr, L.minv.p, c->stream));
  L.has_minv = true;
  return 0;
}

static int cg_ready(ms_ctx* c, int32_t leaflet, int32_t preconditioned) {
  if (int rc = leaflet_ready(c, leaflet, false)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.tilt_grad.p && c->nv > 0) return fail(-4, "no tilt gradient exists for this leaflet (ms_ctx_eval_leaflet)");
  if (preconditioned && !L.has_minv) return fail(-4, "no preconditioner exists (ms_ctx_leaflet_build_preconditioner)");
  return 0;
}

int ms_ctx_leaflet_rz(ms_ctx* c, int32_t leaflet, int32_t preconditioned, double* rz) {
  if (int rc = cg_ready(c, leaflet, preconditioned)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (int rc = c->d_rowsq.ensure(size_t(c->nv) + 1)) return rc;
  if (int rc = ensure_leaflet_results(c)) return rc;
  double* out = c->d_lf_e.p + 5 * size_t(leaflet) + 4;
  CU(ms::launch_rz(c->nv, L.tilt_grad.p, preconditioned ? L.minv.p : nullptr, c->d_rowsq.p, out, c->d_lf_e.p + 16,
                   c->stream));
  if (rz) {
    CU(cudaMemcpyAsync(rz, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

int ms_ctx_leaflet_cg_direction(ms_ctx* c, int32_t leaflet, double beta, int32_t restart, int32_t preconditioned) {
  if (int rc = cg_ready(c, leaflet, preconditioned)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!restart && !L.dir.p && c->nv > 0) return fail(-4, "no previous CG direction: restart first");
  if (int rc = L.dir.ensure(3 * size_t(c->nv) + 1)) return rc;
  CU(ms::launch_tilt_cg_direction(c->nv, L.tilt_grad.p, preconditioned ? L.minv.p : nullptr, beta, restart != 0, L.dir.p,
                                  c->stream));
  return 0;
}

int ms_ctx_leaflet_swap_trial(ms_ctx* c, int32_t leaflet) {
  if (int rc = leaflet_ready(c, leaflet, false)) return rc;
  ms_ctx::Leaflet& L = c->leaflet[leaflet];
  if (!L.trial.p && c->nv > 0) return fail(-4, "no trial tilt field exists (ms_ctx_leaflet_make_trial)");
  std::swap(L.tilts.p, L.trial.p);  // DevBuf owns its pointer: exchange the fields, not the objects
  std::swap(L.tilts.n, L.trial.n);
  return 0;
}

// ---- halo exchange over NVLink peer memory ---------------------------------------------------------------
static int ensure_flag_words(ms_ctx* c) {
  if (c->d_flag_words.p) return 0;
  if (int rc = c->d_flag_words.ensure(ms::kFlagWords)) return rc;
  CU(cudaMemset(c->d_flag_words.p, 0, ms::kFlagWords * sizeof(unsigned long long)));
  if (int rc = c->d_halo_error.ensure(1)) return rc;
  CU(cudaMemset(c->d_halo_error.p, 0, sizeof(int)));
  return 0;
}

int ms_ctx_ipc_export(ms_ctx* c, int32_t which, uint8_t* handle64) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!handle64) return fail(-1, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == MS_IPC_HANDLE_BYTES, "IPC handle size");
  void* p = nullptr;
  if (which == MS_IPC_FLAGS) {
    if (int rc = ensure_flag_words(c)) return rc;
    p = c->d_flag_words.p;
  } else if (which == MS_ARR_POSITIONS || which == MS_ARR_TRIAL || which == MS_ARR_SEEDS) {
    if (int rc = ensure_array(c, which)) return rc;
    int64_t len = 0;
    p = array_ptr(c, which, &len);
  } else {
    return fail(-1, "only positions, trial positions, seeds and the flag words are exported");
  }
  if (!p) return fail(-1, "array is not allocated");
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, p));
  std::memcpy(handle64, &h, sizeof(h));
  return 0;
}

static int peer_register(ms_ctx* c, int32_t slot, int32_t which, void* p);

int ms_ctx_peer_close(ms_ctx* c) {
  if (int rc = check_ctx(c, false)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  for (void* p : c->peers.opened)
    if (p) cudaIpcCloseMemHandle(p);
  c->peers = ms_ctx::PeerTable();
  return 0;
}

int ms_ctx_peer_open(ms_ctx* c, int32_t slot, int32_t which, const uint8_t* handle64) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!handle64 || slot < 0 || slot >= 4096) return fail(-1, "bad peer arguments");
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, sizeof(h));
  void* p = nullptr;
  CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  c->peers.opened.push_back(p);
  return peer_register(c, slot, which, p);
}

static int peer_register(ms_ctx* c, int32_t slot, int32_t which, void* p) {
  ms_ctx::PeerTable& t = c->peers;
  const size_t need = size_t(slot) + 1;
  if (t.pos.size() < need) {
    t.pos.resize(need, nullptr);
    t.trial.resize(need, nullptr);
    t.seeds.resize(need, nullptr);
    t.flags.resize(need, nullptr);
  }
  switch (which) {
    case MS_ARR_POSITIONS: t.pos[size_t(slot)] = static_cast<const double*>(p); break;
    case MS_ARR_TRIAL: t.trial[size_t(slot)] = static_cast<const double*>(p); break;
    case MS_ARR_SEEDS: t.seeds[size_t(slot)] = static_cast<const double*>(p); break;
    case MS_IPC_FLAGS: t.flags[size_t(slot)] = static_cast<unsigned long long*>(p); break;
    default: return fail(-1, "unknown peer array");
  }
  t.tables_current = false;
  return 0;
}

int ms_ctx_peer_set_pointer(ms_ctx* c, int32_t slot, int32_t which, void* device_ptr) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!device_ptr || slot < 0 || slot >= 4096) return fail(-1, "bad peer arguments");
  return peer_register(c, slot, which, device_ptr);
}

void* ms_ctx_flag_words_ptr(ms_ctx* c) {
  if (!c || !c->have_topology || use_device(c)) return nullptr;
  if (ensure_flag_words(c)) return nullptr;
  return c->d_flag_words.p;
}

int ms_ctx_set_ghost_sources(ms_ctx* c, int32_t n_slots, const int32_t* owner_slot, const int32_t* owner_row) {
  if (int rc = check_ctx(c, true)) return rc;
  const int64_t n_ghost = int64_t(c->nv) - c->n_owned;
  if (n_slots <= 0 || (n_ghost > 0 && (!owner_slot || !owner_row))) return fail(-1, "bad ghost source arguments");
  for (int64_t g = 0; g < n_ghost; ++g)
    if (owner_slot[g] < 0 || owner_slot[g] >= n_slots || owner_row[g] < 0) return fail(-1, "ghost source out of range");
  ms_ctx::PeerTable& t = c->peers;
  if (int rc = t.d_owner.ensure(size_t(n_ghost) + 1)) return rc;
  if (int rc = t.d_row.ensure(size_t(n_ghost) + 1)) return rc;
  if (n_ghost) {
    CU(cudaMemcpy(t.d_owner.p, owner_slot, size_t(n_ghost) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(t.d_row.p, owner_row, size_t(n_ghost) * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  t.n_slots = n_slots;
  t.tables_current = false;
  return 0;
}

static int peer_tables(ms_ctx* c) {
  ms_ctx::PeerTable& t = c->peers;
  if (t.tables_current) return 0;
  const size_t n = size_t(t.n_slots);
  if (n == 0) return fail(-4, "ms_ctx_set_ghost_sources has not been called");
  t.pos.resize(n, nullptr);
  t.trial.resize(n, nullptr);
  t.seeds.resize(n, nullptr);
  t.flags.resize(n, nullptr);
  if (int rc = t.d_pos.ensure(n)) return rc;
  if (int rc = t.d_trial.ensure(n)) return rc;
  if (int rc = t.d_seeds.ensure(n)) return rc;
  if (int rc = t.d_flags.ensure(n)) return rc;
  CU(cudaMemcpy(t.d_pos.p, t.pos.data(), n * sizeof(void*), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t.d_trial.p, t.trial.data(), n * sizeof(void*), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t.d_seeds.p, t.seeds.data(), n * sizeof(void*), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t.d_flags.p, t.flags.data(), n * sizeof(void*), cudaMemcpyHostToDevice));
  t.tables_current = true;
  return 0;
}

int ms_ctx_halo_prepare(ms_ctx* c) {
  if (int rc = check_ctx(c, true)) return rc;
  if (int rc = ensure_flag_words(c)) return rc;
  if (int rc = peer_tables(c)) return rc;
  // the tickets of the fused finalisation, the push kernel and the in-kernel pulls: allocated here, not inside the
  // lock-step sequence (zeroed once only: d_ticket[2] must stay in step with the host mirror pull_arrived)
  if (!c->d_ticket.p) {
    if (int rc = c->d_ticket.ensure(4)) return rc;
    CU(cudaMemsetAsync(c->d_ticket.p, 0, 4 * sizeof(unsigned int), c->stream));
  }
  CU(ms::launch_halo_warmup(c->d_flag_words.p, c->d_scalars.p, c->d_halo_error.p, c->d_ticket.p + 1, c->stream));
  CU(cudaDeviceSynchronize());
  return 0;
}

int ms_ctx_halo_signal(ms_ctx* c, int32_t flag_index) {
  NvtxRange range("ms_b200 halo signal");
  if (int rc = check_ctx(c, true)) return rc;
  if (flag_index != MS_FLAG_POSITIONS && flag_index != MS_FLAG_SEEDS)  // words 2 / 3 belong to the all-reduce and the warm-up
    return fail(-1, "flag index must be MS_FLAG_POSITIONS or MS_FLAG_SEEDS");
  if (int rc = ensure_flag_words(c)) return rc;
  CU(ms::launch_halo_signal(c->d_flag_words.p + flag_index, ++c->flag_epoch[flag_index], c->stream));
  return 0;
}

// pull (signal == false: the flag was raised earlier, by ms_ctx_halo_signal or by the last CTA of pass A) or
// signal + pull in one launch
static int halo_launch(ms_ctx* c, int32_t which, int32_t flag_index, bool signal) {
  if (flag_index != MS_FLAG_POSITIONS && flag_index != MS_FLAG_SEEDS)  // words 2 / 3 belong to the all-reduce and the warm-up
    return fail(-1, "flag index must be MS_FLAG_POSITIONS or MS_FLAG_SEEDS");
  if (int rc = ensure_flag_words(c)) return rc;
  const int64_t n_ghost = int64_t(c->nv) - c->n_owned;
  if (n_ghost <= 0) {
    if (signal) CU(ms::launch_halo_signal(c->d_flag_words.p + flag_index, ++c->flag_epoch[flag_index], c->stream));
    return 0;
  }
  if (int rc = peer_tables(c)) return rc;
  ms_ctx::PeerTable& t = c->peers;
  const double* const* table = nullptr;
  const std::vector<const double*>* host = nullptr;
  int width = 3;
  switch (which) {
    case MS_ARR_POSITIONS: table = t.d_pos.p; host = &t.pos; break;
    case MS_ARR_TRIAL: table = t.d_trial.p; host = &t.trial; break;
    case MS_ARR_SEEDS: table = t.d_seeds.p; host = &t.seeds; width = ms::kSeedStride; break;
    default: return fail(-1, "only positions, trial positions and seeds travel through the halo");
  }
  bool any = false;
  for (const double* p : *host) any = any || p != nullptr;
  if (!any) return fail(-4, "no peer array has been opened for this exchange (ms_ctx_peer_open)");
  int64_t len = 0;
  double* dst = array_ptr(c, which, &len);
  if (!dst) return fail(-4, "the local array does not exist");
  // the epoch this rank has published is the epoch every owner must have reached (lock-step sequence)
  if (signal) {
    const unsigned long long epoch = ++c->flag_epoch[flag_index];
    CU(ms::launch_halo_exchange(c->d_flag_words.p + flag_index, int(n_ghost), width, table, t.d_flags.p, t.n_slots,
                                flag_index, epoch, t.d_owner.p, t.d_row.p, dst + size_t(c->n_owned) * width,
                                c->d_halo_error.p, c->stream));
    return 0;
  }
  CU(ms::launch_halo_pull(int(n_ghost), width, table, t.d_flags.p, t.n_slots, flag_index, c->flag_epoch[flag_index],
                          t.d_owner.p, t.d_row.p, dst + size_t(c->n_owned) * width, c->d_halo_error.p, c->stream));
  return 0;
}

int ms_ctx_halo_pull(ms_ctx* c, int32_t which, int32_t flag_index) {
  NvtxRange range("ms_b200 halo pull");
  if (int rc = check_ctx(c, true)) return rc;
  return halo_launch(c, which, flag_index, false);
}

int ms_ctx_set_rank_slot(ms_ctx* c, int32_t slot, int32_t n_slots) {
  if (int rc = check_ctx(c, true)) return rc;
  if (n_slots <= 0 || slot < 0 || slot >= n_slots) return fail(-1, "bad rank slot");
  if (int rc = ensure_flag_words(c)) return rc;
  ms_ctx::PeerTable& t = c->peers;
  const size_t need = size_t(n_slots);
  if (t.pos.size() < need) {
    t.pos.resize(need, nullptr);
    t.trial.resize(need, nullptr);
    t.seeds.resize(need, nullptr);
    t.flags.resize(need, nullptr);
  }
  t.flags[size_t(slot)] = c->d_flag_words.p;  // this rank's own block takes part in the all-reduce
  t.my_slot = slot;
  t.n_slots = n_slots;
  t.tables_current = false;
  return 0;
}

int ms_ctx_allreduce_scalars(ms_ctx* c, int32_t count) {
  NvtxRange range("ms_b200 all-reduce (peer memory)");
  if (int rc = check_ctx(c, true)) return rc;
  if (count <= 0 || count > 16) return fail(-1, "between 1 and 16 scalars");
  if (int rc = ensure_flag_words(c)) return rc;
  if (int rc = peer_tables(c)) return rc;
  ms_ctx::PeerTable& t = c->peers;
  for (int32_t s = 0; s < t.n_slots; ++s)
    if (!t.flags[size_t(s)]) return fail(-4, "the flag words of every rank must be opened (ms_ctx_peer_open, ms_ctx_set_rank_slot)");
  CU(ms::launch_allreduce_peer(c->d_scalars.p, count, c->d_flag_words.p, t.d_flags.p, t.n_slots, ++c->flag_epoch[2],
                               c->d_halo_error.p, c->stream));
  return 0;
}

int ms_ctx_halo_error(ms_ctx* c, int32_t* error) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!error) return fail(-1, "null argument");
  *error = 0;
  if (!c->d_halo_error.p) return 0;
  int e = 0;
  CU(cudaMemcpyAsync(&e, c->d_halo_error.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *error = e;
  return 0;
}

int ms_ctx_set_push_targets(ms_ctx* c, int32_t n, const int32_t* dst_slot, const int32_t* src_row, const int32_t* dst_row) {
  if (int rc = check_ctx(c, true)) return rc;
  ms_ctx::PeerTable& t = c->peers;
  if (n < 0 || (n > 0 && (!dst_slot || !src_row || !dst_row))) return fail(-1, "bad push target arguments");
  if (t.n_slots <= 0 || t.my_slot < 0) return fail(-4, "ms_ctx_set_rank_slot has not been called");
  if (t.n_slots > ms::kPushMaxRanks) return fail(-1, "the push transport holds up to 16 ranks");
  uint64_t mask = 0;
  for (int32_t i = 0; i < n; ++i) {
    if (dst_slot[i] < 0 || dst_slot[i] >= t.n_slots || dst_slot[i] == t.my_slot || src_row[i] < 0 ||
        src_row[i] >= c->n_owned || dst_row[i] < 0)
      return fail(-1, "push target out of range");
    mask |= 1ull << dst_slot[i];
  }
  if (int rc = t.d_push_slot.ensure(size_t(n) + 1)) return rc;
  if (int rc = t.d_push_src.ensure(size_t(n) + 1)) return rc;
  if (int rc = t.d_push_dst.ensure(size_t(n) + 1)) return rc;
  if (n) {
    CU(cudaMemcpy(t.d_push_slot.p, dst_slot, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(t.d_push_src.p, src_row, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(t.d_push_dst.p, dst_row, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  t.n_push = n;
  t.push_mask = mask;
  t.push_ready = true;
  return 0;
}

// push this rank's rows of `which` into the ghost slots of the ranks that list them and raise its arrival word there
static int halo_push(ms_ctx* c, int32_t which, int kind) {
  ms_ctx::PeerTable& t = c->peers;
  if (!t.push_ready) return fail(-4, "ms_ctx_set_push_targets has not been called");
  if (int rc = peer_tables(c)) return rc;
  if (!c->d_ticket.p) {
    if (int rc = c->d_ticket.ensure(4)) return rc;
    CU(cudaMemsetAsync(c->d_ticket.p, 0, 4 * sizeof(unsigned int), c->stream));
  }
  double* const* table = nullptr;
  int width = 3;
  switch (which) {
    case MS_ARR_POSITIONS: table = const_cast<double* const*>(reinterpret_cast<const double* const*>(t.d_pos.p)); break;
    case MS_ARR_TRIAL: table = const_cast<double* const*>(reinterpret_cast<const double* const*>(t.d_trial.p)); break;
    case MS_ARR_SEEDS:
      table = const_cast<double* const*>(reinterpret_cast<const double* const*>(t.d_seeds.p));
      width = ms::kSeedStride;
      break;
    default: return fail(-1, "only positions, trial positions and seeds travel through the halo");
  }
  int64_t len = 0;
  const double* src = array_ptr(c, which, &len);
  if (!src) return fail(-4, "the local array does not exist");
  const unsigned long long epoch = ++c->flag_epoch[kind];
  CU(ms::launch_halo_push(t.n_push, width, src, table, t.d_push_slot.p, t.d_push_src.p, t.d_push_dst.p, t.d_flags.p,
                          t.n_slots, t.push_mask, t.my_slot, kind, epoch, c->d_ticket.p + 1, c->stream));
  return 0;
}

int ms_ctx_halo_push(ms_ctx* c, int32_t which, int32_t flag_index) {
  NvtxRange range("ms_b200 halo push");
  if (int rc = check_ctx(c, true)) return rc;
  if (flag_index != MS_FLAG_POSITIONS && flag_index != MS_FLAG_SEEDS)
    return fail(-1, "flag index must be MS_FLAG_POSITIONS or MS_FLAG_SEEDS");
  if (int rc = ensure_flag_words(c)) return rc;
  return halo_push(c, which, flag_index);
}

// the patch kernel waits for the pushed rows of `kind` before it stages its first patch
static void attach_wait(ms_ctx* c, ms::PatchLaunch& a, int kind) {
  a.wait_flags = c->d_flag_words.p + ms::kPushFlagBase + 64 * kind;
  a.wait_epoch = c->flag_epoch[kind];
  a.wait_mask = c->peers.push_mask;
  a.wait_error = c->d_halo_error.p;
}

// in-kernel halo exchange (ms::HaloPull): the launch walks the interior patches first and pulls `which` meanwhile
static int attach_pull(ms_ctx* c, ms::PatchLaunch& a, int32_t which, int32_t flag_index, bool signal_here) {
  ms_ctx::PeerTable& t = c->peers;
  const int64_t n_ghost = int64_t(c->nv) - c->n_owned;
  const int n_patches = int(c->packed.patches.size());
  a.patch_list = c->d_patch_order.p;   // interior patches, then the patches that read ghost rows
  a.patch_begin = 0;
  a.patch_count = n_patches;
  if (signal_here) {
    a.pull.own_flag = c->d_flag_words.p + flag_index;
    ++c->flag_epoch[flag_index];
  }
  a.pull.epoch = c->flag_epoch[flag_index];
  if (n_ghost <= 0) return 0;   // still signals: other ranks may hold ghosts of this one
  int width = 3;
  const double* const* table = nullptr;
  switch (which) {
    case MS_ARR_POSITIONS: table = t.d_pos.p; break;
    case MS_ARR_TRIAL: table = t.d_trial.p; break;
    case MS_ARR_SEEDS: table = t.d_seeds.p; width = ms::kSeedStride; break;
    default: return fail(-1, "only positions, trial positions and seeds travel through the halo");
  }
  int64_t len = 0;
  double* dst = array_ptr(c, which, &len);
  if (!dst) return fail(-4, "the local array does not exist");
  if (!c->d_ticket.p) {
    if (int rc = c->d_ticket.ensure(4)) return rc;
    CU(cudaMemsetAsync(c->d_ticket.p, 0, 4 * sizeof(unsigned int), c->stream));
  }
  a.pull.n_ghost = int32_t(n_ghost);
  a.pull.width = width;
  a.pull.peer_base = table;
  a.pull.peer_flag = t.d_flags.p;
  a.pull.n_slots = t.n_slots;
  a.pull.flag_index = flag_index;
  a.pull.owner = t.d_owner.p;
  a.pull.row = t.d_row.p;
  a.pull.dst = dst + size_t(c->n_owned) * width;
  a.pull.arrived = c->d_ticket.p + 2;
  c->pull_arrived += unsigned(ms::patch_grid(a));
  a.pull.arrived_target = c->pull_arrived;
  a.pull.first_boundary = c->n_interior;
  a.pull.first_ghost_row = int32_t(c->n_owned);
  a.pull.error = c->d_halo_error.p;
  return 0;
}

// One evaluation of this rank's partition with the transport folded into the compute launches (peer memory):
//   [signal + pull positions] -> pass A (its last CTA raises the seed flag) -> [pull seeds] -> pass B (its last
//   CTA reduces the per-CTA rows and publishes the local scalars) -> gather (rank-order sum) + KKT coefficient
// = 5 launches where the unfused sequence (ms_ctx_halo_signal / _pull, passes, ms_ctx_eval_reduce,
// ms_ctx_allreduce_scalars, ms_ctx_eval_project) needs 10.  Ranks must run concurrently (one process per GPU).
int ms_ctx_eval_partition(ms_ctx* c, const ms_eval_opts* o, int32_t exchange_positions) {
  NvtxRange range("ms_b200 partition evaluation");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o) return fail(-1, "null options");
  if (o->patch_count != -1 || c->packed.patches.empty()) return fail(-1, "ms_ctx_eval_partition evaluates whole, non-empty partitions");
  if (has_bt(o)) return fail(-1, "bending_tilt evaluations use the unfused sequence");
  if (int rc = ensure_flag_words(c)) return rc;
  if (int rc = peer_tables(c)) return rc;
  ms_ctx::PeerTable& t = c->peers;
  for (int32_t s = 0; s < t.n_slots; ++s)
    if (!t.flags[size_t(s)]) return fail(-4, "the flag words of every rank must be opened (ms_ctx_peer_open, ms_ctx_set_rank_slot)");
  const bool bending = needs_bending(o);
  const bool ran_a = bending || !o->want_grad;
  const bool run_b = o->want_grad || (o->want_tilt_grad && (o->modules & MS_MOD_TILT));
  if (!o->want_grad && run_b) return fail(-1, "tilt-only evaluations use the unfused sequence");
  const bool push = t.push_ready;   // PUSH: owners store into the ghost slots, receivers poll local words only
  // bit 1 of exchange_positions: exchange INSIDE the patch kernels (ms::HaloPull), hidden behind the interior patches
  const bool overlap = (exchange_positions & 2) != 0 && !push && c->packed.params.threads >= 64;
  exchange_positions &= 1;
  bool wait_positions = false;
  bool pull_positions = false;
  if (exchange_positions) {
    if (overlap) {
      pull_positions = true;
    } else if (push) {
      if (int rc = halo_push(c, o->use_trial ? MS_ARR_TRIAL : MS_ARR_POSITIONS, MS_FLAG_POSITIONS)) return rc;
      wait_positions = true;
    } else if (int rc = halo_launch(c, o->use_trial ? MS_ARR_TRIAL : MS_ARR_POSITIONS, MS_FLAG_POSITIONS, true)) {
      return rc;
    }
  }
  const unsigned long long reduce_epoch = ++c->flag_epoch[2];
  auto publish = [&](ms::PatchLaunch& a) -> int {
    if (int rc = attach_finalize(c, o, a)) return rc;
    a.fin.constraint_mode = -2;  // the coefficient needs the GLOBAL sums: k_allreduce_gather_coef / _local_coef
    a.fin.publish_epoch = reduce_epoch;
    if (push) {
      a.fin.push_words = t.d_flags.p;
      a.fin.push_slots = t.n_slots;
      a.fin.push_my_slot = t.my_slot;
    } else {
      a.fin.publish_words = c->d_flag_words.p;
      if (overlap) {  // gather in the last CTA as well: no third launch
        a.fin.gather_words = t.d_flags.p;
        a.fin.gather_slots = t.n_slots;
        a.fin.gather_mode = o->want_grad ? o->constraint_mode : -2;
        a.fin.gather_error = c->d_halo_error.p;
      }
    }
    return 0;
  };
  if (ran_a) {
    ms::PatchLaunch a;
    if (int rc = fill_launch(c, o, a)) return rc;
    a.partials = c->d_partials_a.p;
    c->ran_pass_a = true;
    if (!o->want_grad) {
      if (int rc = publish(a)) return rc;
    } else if (bending && !push) {  // ticket without a reduction: the last CTA raises the seed flag
      if (int rc = attach_finalize(c, o, a)) return rc;
      a.fin.scalars = nullptr;
      a.fin.signal_flag = c->d_flag_words.p + MS_FLAG_SEEDS;
      a.fin.signal_epoch = ++c->flag_epoch[MS_FLAG_SEEDS];
    }
    if (wait_positions) attach_wait(c, a, MS_FLAG_POSITIONS);
    wait_positions = false;
    if (pull_positions)
      if (int rc = attach_pull(c, a, o->use_trial ? MS_ARR_TRIAL : MS_ARR_POSITIONS, MS_FLAG_POSITIONS, true)) return rc;
    pull_positions = false;
    CU(ms::launch_pass_a(a, c->stream));
  } else {
    c->ran_pass_a = false;
  }
  if (o->want_grad) {
    if (bending && !overlap) {
      if (push) {
        if (int rc = halo_push(c, MS_ARR_SEEDS, MS_FLAG_SEEDS)) return rc;
      } else if (int rc = halo_launch(c, MS_ARR_SEEDS, MS_FLAG_SEEDS, false)) {
        return rc;
      }
    }
    ms::PatchLaunch a;
    if (int rc = fill_launch(c, o, a)) return rc;
    a.partials = c->d_partials_b.p;
    c->proj.active = false;
    if (overlap && bending) {  // the seed flag was raised by the last CTA of pass A
      if (int rc = attach_pull(c, a, MS_ARR_SEEDS, MS_FLAG_SEEDS, false)) return rc;
    } else if (pull_positions) {  // surface / volume only: pass B is the first kernel
      if (int rc = attach_pull(c, a, o->use_trial ? MS_ARR_TRIAL : MS_ARR_POSITIONS, MS_FLAG_POSITIONS, true)) return rc;
    }
    if (push && bending) attach_wait(c, a, MS_FLAG_SEEDS);
    else if (wait_positions) attach_wait(c, a, MS_FLAG_POSITIONS);   // surface / volume only: pass B is the first kernel
    if ((o->modules & MS_MOD_TILT) && !a.tilt_grad) {
      if (int rc = ensure_array(c, MS_ARR_TILT_GRAD)) return rc;
      a.tilt_grad = c->d_tilt_grad.p;
    }
    if (int rc = publish(a)) return rc;
    CU(ms::launch_pass_b(a, bending, !bending, c->stream));
  }
  bool use_gc, use_fixed;
  projection_of(c, o, use_gc, use_fixed);
  if (overlap) {
    // gathered by the last CTA of the last pass
  } else if (push)
    CU(ms::launch_allreduce_local_coef(c->d_scalars.p, 12, c->d_flag_words.p, t.n_slots, reduce_epoch,
                                       o->want_grad ? o->constraint_mode : -2, use_gc ? 1 : 0, o->k_vol, o->v_target,
                                       c->d_halo_error.p, c->stream));
  else
    CU(ms::launch_allreduce_gather_coef(c->d_scalars.p, 12, t.d_flags.p, t.n_slots, reduce_epoch,
                                        o->want_grad ? o->constraint_mode : -2, use_gc ? 1 : 0, o->k_vol, o->v_target,
                                        c->d_halo_error.p, c->stream));
  if (o->want_grad) {
    c->proj.active = use_gc || use_fixed;
    c->proj.use_gc = use_gc;
    c->proj.use_fixed = use_fixed;
  }
  return 0;
}

// ---- pipelined host evaluation ---------------------------------------------------------------------
// The positions travel in chunks of rows; a patch can run pass A as soon as every row it reads has
// arrived, and pass B as soon as pass A has run for every patch that owns one of its local vertices.
static int pipe_prepare(ms_ctx* c) {
  if (c->pipe_ready) return 0;
  const ms::PackedMesh& pk = c->packed;
  const int32_t np = int32_t(pk.patches.size());
  std::vector<int32_t> need_a(size_t(np), 0), pos_a(size_t(np), 0), order_a(size_t(np), 0), order_b(size_t(np), 0),
      need_b(size_t(np), 0);
  for (int32_t p = 0; p < np; ++p) {
    const ms::PatchHeader& h = pk.patches[size_t(p)];
    int32_t m = h.v_lo + h.n_owned;
    for (int32_t j = 0; j < h.n_halo; ++j) m = std::max(m, pk.halo_ids[size_t(h.halo_off) + size_t(j)] + 1);
    need_a[size_t(p)] = m;
  }
  std::iota(order_a.begin(), order_a.end(), 0);
  std::stable_sort(order_a.begin(), order_a.end(), [&](int32_t x, int32_t y) { return need_a[size_t(x)] < need_a[size_t(y)]; });
  for (int32_t i = 0; i < np; ++i) pos_a[size_t(order_a[size_t(i)])] = i;
  for (int32_t p = 0; p < np; ++p) {
    const ms::PatchHeader& h = pk.patches[size_t(p)];
    int32_t m = pos_a[size_t(p)];
    for (int32_t j = 0; j < h.n_halo; ++j) {
      const int32_t v = pk.halo_ids[size_t(h.halo_off) + size_t(j)];
      // the patch owning vertex v: last patch with v_lo <= v
      const int32_t q = int32_t(std::upper_bound(c->v_lo.begin(), c->v_lo.begin() + np, v) - c->v_lo.begin()) - 1;
      if (q >= 0) m = std::max(m, pos_a[size_t(q)]);
    }
    need_b[size_t(p)] = m + 1;  // number of orderA patches that must have been launched
  }
  std::iota(order_b.begin(), order_b.end(), 0);
  std::stable_sort(order_b.begin(), order_b.end(), [&](int32_t x, int32_t y) { return need_b[size_t(x)] < need_b[size_t(y)]; });
  c->pipe_need_a.resize(size_t(np));
  c->pipe_need_b.resize(size_t(np));
  for (int32_t i = 0; i < np; ++i) {
    c->pipe_need_a[size_t(i)] = need_a[size_t(order_a[size_t(i)])];
    c->pipe_need_b[size_t(i)] = need_b[size_t(order_b[size_t(i)])];
  }
  if (int rc = c->d_order_a.ensure(size_t(np) + 1)) return rc;
  if (int rc = c->d_order_b.ensure(size_t(np) + 1)) return rc;
  if (np) {
    CU(cudaMemcpy(c->d_order_a.p, order_a.data(), size_t(np) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_order_b.p, order_b.data(), size_t(np) * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  if (!c->copy_stream) CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  c->pipe_ready = true;
  return 0;
}

constexpr int kPipeChunksMax = 32;

static int pipe_chunks() {
  static const int n = [] {
    const char* e = std::getenv("MS_PIPE_CHUNKS");
    const int v = e ? std::atoi(e) : 8;
    return v < 2 ? 2 : (v > kPipeChunksMax ? kPipeChunksMax : v);
  }();
  return n;
}

static bool pipe_applicable(const ms_ctx* c, const ms_eval_opts* o, const double* pos_host) {
  static const bool disabled = std::getenv("MS_NO_PIPELINE") != nullptr;
  return !disabled && pos_host && c->perm.empty() && c->n_owned == c->nv && !has_bt(o) && !(o->modules & MS_MOD_TILT) && !o->want_tilt_grad &&
         o->patch_count == -1 &&
         c->nv >= 200000 && c->packed.patches.size() >= 64;
}

// upload + pass A + pass B, overlapped; leaves the per-CTA sums in rows [0, rows_a) / [0, rows_b)
static int eval_pipelined(ms_ctx* c, const ms_eval_opts* o, const double* pos_host, int& rows_a, int& rows_b) {
  if (int rc = pipe_prepare(c)) return rc;
  if (o->use_trial)
    if (int rc = ensure_array(c, MS_ARR_TRIAL)) return rc;
  ms::PatchLaunch base;
  if (int rc = fill_launch(c, o, base)) return rc;
  const int32_t np = int32_t(c->packed.patches.size());
  const bool ran_a = needs_bending(o) || !o->want_grad;
  c->ran_pass_a = ran_a;
  double* dst = o->use_trial ? c->d_trial.p : c->d_pos.p;
  if (!o->use_trial) c->has_positions = true;
  const int kPipeChunks = pipe_chunks();
  while (c->pipe_events.size() < size_t(kPipeChunks) + 1) {
    cudaEvent_t e = nullptr;
    CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->pipe_events.push_back(e);
  }
  // the copies may start once everything queued so far (readers of the old positions) has finished
  CU(cudaEventRecord(c->pipe_events[size_t(kPipeChunks)], c->stream));
  CU(cudaStreamWaitEvent(c->copy_stream, c->pipe_events[size_t(kPipeChunks)], 0));
  const int64_t nv = c->nv;
  int64_t row_hi[kPipeChunksMax];
  // chunk boundaries: quadratic spacing (large chunks first, small ones last) keeps the kernels busy early and
  // leaves little work behind the last copy; MS_PIPE_SPACING=uniform for equal chunks
  static const bool uniform = [] {
    const char* e = std::getenv("MS_PIPE_SPACING");
    return e && std::string(e) == "uniform";
  }();
  auto boundary = [&](int k) -> int64_t {
    if (k >= kPipeChunks) return nv;
    const double x = double(k) / kPipeChunks;
    return int64_t(double(nv) * (uniform ? x : 1.0 - (1.0 - x) * (1.0 - x)));
  };
  for (int k = 0; k < kPipeChunks; ++k) {
    const int64_t r0 = boundary(k), r1 = boundary(k + 1);
    row_hi[k] = r1;
    if (r1 > r0)
      CU(cudaMemcpyAsync(dst + 3 * r0, pos_host + 3 * r0, size_t(3 * (r1 - r0)) * sizeof(double), cudaMemcpyHostToDevice,
                         c->copy_stream));
    CU(cudaEventRecord(c->pipe_events[size_t(k)], c->copy_stream));
  }
  int32_t a_done = 0, b_done = 0;
  rows_a = rows_b = 0;
  for (int k = 0; k < kPipeChunks; ++k) {
    CU(cudaStreamWaitEvent(c->stream, c->pipe_events[size_t(k)], 0));
    const int32_t a_hi = int32_t(std::upper_bound(c->pipe_need_a.begin(), c->pipe_need_a.end(), int32_t(row_hi[k])) -
                                 c->pipe_need_a.begin());
    if (a_hi > a_done) {
      ms::PatchLaunch a = base;
      a.patch_list = c->d_order_a.p;
      a.patch_begin = a_done;
      a.patch_count = a_hi - a_done;
      if (ran_a) {
        a.partials = c->d_partials_a.p;
        a.partial_row0 = rows_a;
        CU(ms::launch_pass_a(a, c->stream));
        rows_a += ms::patch_grid(a);
      } else if (o->want_grad) {
        // no pass A (surface / volume only): pass B reads positions alone and follows the same order
        a.partials = c->d_partials_b.p;
        a.partial_row0 = rows_b;
        CU(ms::launch_pass_b(a, false, true, c->stream));
        rows_b += ms::patch_grid(a);
      }
      a_done = a_hi;
    }
    if (ran_a && o->want_grad) {
      const int32_t b_hi = int32_t(std::upper_bound(c->pipe_need_b.begin(), c->pipe_need_b.end(), a_done) -
                                   c->pipe_need_b.begin());
      if (b_hi > b_done) {
        ms::PatchLaunch b = base;
        b.patch_list = c->d_order_b.p;
        b.patch_begin = b_done;
        b.patch_count = b_hi - b_done;
        b.partials = c->d_partials_b.p;
        b.partial_row0 = rows_b;
        CU(ms::launch_pass_b(b, true, false, c->stream));
        rows_b += ms::patch_grid(b);
        b_done = b_hi;
      }
    }
  }
  if (a_done != np || (ran_a && o->want_grad && b_done != np)) return fail(-9, "pipelined evaluation did not cover every patch");
  return 0;
}

int ms_ctx_eval_host(ms_ctx* c, const ms_eval_opts* o, const double* pos_host, double* scalars16,
                     double* grad_host, double* volgrad_host, double* tilt_grad_host) {
  NvtxRange range("ms_b200 eval_host (H2D, evaluation, D2H)");
  if (int rc = check_ctx(c, true)) return rc;
  if (!o || !scalars16) return fail(-1, "null argument");
  const int64_t n3 = 3 * int64_t(c->nv);
  if (pipe_applicable(c, o, pos_host)) {
    // large meshes: the upload is cut into row chunks and the patch kernels start as their rows arrive
    int rows_a = 0, rows_b = 0;
    if (int rc = eval_pipelined(c, o, pos_host, rows_a, rows_b)) return rc;
    if (int rc = reduce_rows(c, o, rows_a, rows_b)) return rc;
    if (int rc = ms_ctx_eval_project(c, o)) return rc;
  } else {
    if (pos_host)
      if (int rc = ms_ctx_upload(c, o->use_trial ? MS_ARR_TRIAL : MS_ARR_POSITIONS, pos_host, 0, n3)) return rc;
    if (int rc = ms_ctx_eval_async(c, o)) return rc;
  }
  if (o->want_grad && grad_host && n3) {
    if (int rc = flush_projection(c)) return rc;
    if (int rc = download_rows(c, c->d_grad.p, grad_host, 3)) return rc;
  }
  if (o->want_grad && volgrad_host && n3 && (o->modules & MS_MOD_VOLUME))
    if (int rc = download_rows(c, c->d_volgrad.p, volgrad_host, 3)) return rc;
  if ((o->want_grad || o->want_tilt_grad) && tilt_grad_host && n3 && c->d_tilt_grad.p)
    if (int rc = download_rows(c, c->d_tilt_grad.p, tilt_grad_host, 3)) return rc;
  return ms_ctx_read_scalars(c, scalars16);
}

int ms_ctx_set_send_rows(ms_ctx* c, const int32_t* rows, int64_t n) {
  if (int rc = check_ctx(c, true)) return rc;
  if (n < 0 || (n > 0 && !rows)) return fail(-1, "bad arguments");
  for (int64_t i = 0; i < n; ++i)
    if (rows[i] < 0 || rows[i] >= c->nv) return fail(-1, "send row out of range");
  if (int rc = c->d_send_rows.ensure(size_t(n) + 1)) return rc;
  if (n) CU(cudaMemcpy(c->d_send_rows.p, rows, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice));
  c->n_send_rows = n;
  return 0;
}

int ms_ctx_pack_send(ms_ctx* c, int which, void* out_device) {
  if (int rc = check_ctx(c, true)) return rc;
  if (which == MS_ARR_GRAD)
    if (int rc = flush_projection(c)) return rc;
  int64_t len = 0;
  const double* src = array_ptr(c, which, &len);
  if (!src || c->nv <= 0 || len % c->nv) return fail(-1, "array is not a per-vertex array");
  if (c->n_send_rows > 0 && !out_device) return fail(-1, "null output buffer");
  CU(ms::launch_gather_rows(src, int(len / c->nv), c->d_send_rows.p, c->n_send_rows,
                            static_cast<double*>(out_device), c->stream));
  return 0;
}

int ms_ctx_make_trial(ms_ctx* c, double alpha) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!c->d_dir.p) return fail(-4, "no search direction uploaded (MS_ARR_DIRECTION)");
  if (int rc = ensure_array(c, MS_ARR_TRIAL)) return rc;
  CU(ms::launch_axpy(c->d_pos.p, c->d_dir.p, alpha, c->d_trial.p, 3 * int64_t(c->nv), c->stream));
  return 0;
}

int ms_ctx_accept_trial(ms_ctx* c) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!c->d_trial.p) return fail(-4, "no trial positions exist");
  CU(cudaMemcpyAsync(c->d_pos.p, c->d_trial.p, 3 * size_t(c->nv) * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  c->has_positions = true;
  return 0;
}

int ms_ctx_vertex_average(ms_ctx* c, const int32_t* group, int32_t rounds) {
  if (int rc = check_ctx(c, true)) return rc;
  if (c->n_owned != c->nv) return fail(-5, "vertex averaging is not available on a partitioned context");
  if (rounds < 0) return fail(-1, "rounds must be >= 0");
  if (!c->has_positions) return fail(-4, "no positions have been set (MS_ARR_POSITIONS)");
  if (rounds == 0 || c->nv == 0) return 0;
  if (int rc = ensure_corner_csr(c)) return rc;
  if (int rc = ensure_array(c, MS_ARR_TRIAL)) return rc;
  const size_t nv = size_t(c->nv);
  if (group) {
    std::vector<int32_t> tmp;
    if (!c->perm.empty()) {
      tmp = permuted(group, c->perm);
      group = tmp.data();
    }
    if (int rc = c->d_va_group.ensure(nv)) return rc;
    CU(cudaMemcpyAsync(c->d_va_group.p, group, nv * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));  // tmp (or the caller's array) may go away after the return
  }
  ms::VaMesh m;
  m.nv = c->nv;
  m.tri = c->d_tri.p;
  m.csr_ptr = c->d_csr_ptr.p;
  m.csr_idx = c->d_csr_idx.p;
  m.group = group ? c->d_va_group.p : nullptr;
  m.fixed = c->has_fixed ? c->d_fixed.p : nullptr;
  // Jacobi rounds alternate between the positions and the trial buffer; an odd count ends with one copy back
  double* buf[2] = {c->d_pos.p, c->d_trial.p};
  for (int32_t r = 0; r < rounds; ++r) {
    m.pos = buf[r & 1];
    CU(ms::launch_vertex_average(m, buf[(r + 1) & 1], c->stream));
  }
  if (rounds & 1)
    CU(cudaMemcpyAsync(c->d_pos.p, c->d_trial.p, 3 * nv * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  return 0;
}

int ms_ctx_equiangulate(ms_ctx* c, int32_t max_iterations, int64_t* n_flips, int32_t* n_sweeps) {
  if (int rc = check_ctx(c, true)) return rc;
  if (c->n_owned != c->nv) return fail(-5, "equiangulation is not available on a partitioned context");
  if (max_iterations < 0) return fail(-1, "max_iterations must be >= 0");
  if (!c->has_positions) return fail(-4, "no positions have been set (MS_ARR_POSITIONS)");
  for (int32_t x : c->h_tri)
    if (x < 0 || x >= c->nv) return fail(-1, "a facet has a vertex index outside [0, nv)");
  c->eq_rounds.clear();
  std::fill(c->eq_ms, c->eq_ms + 4, 0.0);
  if (n_flips) *n_flips = 0;
  if (n_sweeps) *n_sweeps = 0;
  if (max_iterations == 0 || c->nf == 0) return 0;
  if (int rc = ensure_tri(c)) return rc;
  NvtxRange range("ms_b200 equiangulate");
  using clock = std::chrono::steady_clock;
  auto ms_since = [](clock::time_point t0) { return std::chrono::duration<double, std::milli>(clock::now() - t0).count(); };
  const size_t nh = 3 * size_t(c->nf), nc_max = nh / 2 + 1;
  constexpr int kBatch = 8;  // selection rounds between two reads of the undecided counters
  // sweep scratch, released on return: sorted half-edge keys, candidates, conflict lists, round states, counters
  DevBuf<uint64_t> key_in, keys, nkey;
  DevBuf<int32_t> h_in, order, cand_pos, h1, h2, slot, nkey_cand, nkey_pos, counters;
  DevBuf<uint8_t> flag, state0, state1, temp;
  size_t tb_edges = 0, tb_cands = 0;
  CU(ms::eq_temp_bytes(int64_t(nh), &tb_edges));
  CU(ms::eq_temp_bytes(int64_t(nc_max), &tb_cands));
  const size_t tb = std::max(tb_edges, tb_cands);
  for (int rc : {key_in.ensure(nh), keys.ensure(nh), nkey.ensure(nc_max), h_in.ensure(nh), order.ensure(nh),
                 cand_pos.ensure(nh), h1.ensure(nc_max), h2.ensure(nc_max), slot.ensure(nh), nkey_cand.ensure(nc_max),
                 nkey_pos.ensure(nc_max), counters.ensure(kBatch + 2), flag.ensure(nh), state0.ensure(nc_max),
                 state1.ensure(nc_max), temp.ensure(tb + 1)})
    if (rc) return rc;
  ms::EqMesh m{c->nv, c->nf, c->d_tri.p, c->d_pos.p, c->has_fixed ? c->d_fixed.p : nullptr,
               c->perm.empty() ? nullptr : c->d_perm.p, keys.p, order.p};
  ms::EqCands s{0, h1.p, h2.p, slot.p, nkey.p, nkey_cand.p, nkey_pos.p};
  uint8_t* state[2] = {state0.p, state1.p};
  int32_t h_counters[kBatch + 2];
  int64_t total = 0;
  int32_t sweeps = 0;
  struct Events {  // the sweeps' device time; the context's own events belong to ms_ctx_timer_*
    cudaEvent_t e[2] = {nullptr, nullptr};
    ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
  } ev;
  CU(cudaEventCreate(&ev.e[0]));
  CU(cudaEventCreate(&ev.e[1]));
  CU(cudaEventRecord(ev.e[0], c->stream));
  for (int32_t sweep = 0; sweep < max_iterations; ++sweep) {
    CU(ms::launch_eq_sort_edges(m, key_in.p, h_in.p, keys.p, order.p, temp.p, tb, c->stream));
    CU(ms::launch_eq_candidates(m, flag.p, cand_pos.p, counters.p + kBatch, temp.p, tb, c->stream));
    CU(cudaMemcpyAsync(h_counters + kBatch, counters.p + kBatch, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    s.n = h_counters[kBatch];
    if (s.n == 0) {
      c->eq_rounds.push_back(0);
      break;
    }
    // the sort inputs are free again: they hold the candidates' new-diagonal keys and ids
    CU(ms::launch_eq_conflicts(m, s.n, cand_pos.p, s, key_in.p, h_in.p, temp.p, tb, c->stream));
    CU(cudaMemsetAsync(state[0], 0, size_t(s.n), c->stream));
    int32_t done = -1;  // the round after which no candidate was undecided
    for (int32_t r0 = 0; done < 0; r0 += kBatch) {
      if (r0 > s.n) return fail(-1, "equiangulation: the selection rounds do not converge");  // cannot happen
      CU(cudaMemsetAsync(counters.p, 0, kBatch * sizeof(int32_t), c->stream));
      for (int k = 0; k < kBatch; ++k)
        CU(ms::launch_eq_round(s, state[(r0 + k) & 1], state[(r0 + k + 1) & 1], k ? counters.p + k - 1 : nullptr,
                               counters.p + k, c->stream));
      CU(cudaMemcpyAsync(h_counters, counters.p, kBatch * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      for (int k = 0; k < kBatch && done < 0; ++k)
        if (h_counters[k] == 0) done = r0 + k;
    }
    CU(cudaMemsetAsync(counters.p + kBatch + 1, 0, sizeof(int32_t), c->stream));
    CU(ms::launch_eq_apply(s, state[(done + 1) & 1], c->d_tri.p, counters.p + kBatch + 1, c->stream));
    CU(cudaMemcpyAsync(h_counters + kBatch + 1, counters.p + kBatch + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->eq_rounds.push_back(done + 1);
    total += h_counters[kBatch + 1];
    ++sweeps;
  }
  CU(cudaEventRecord(ev.e[1], c->stream));
  CU(cudaEventSynchronize(ev.e[1]));
  float sweep_ms = 0.f;
  CU(cudaEventElapsedTime(&sweep_ms, ev.e[0], ev.e[1]));
  c->eq_ms[0] = sweep_ms;
  if (total > 0) {
    // facet rows stay in place, so per-facet and per-vertex data survive; only the packing follows the new rows,
    // packed where they are
    DevBuf<uint8_t> body_dev;
    if (!c->h_body.empty()) {
      if (int rc = body_dev.ensure(size_t(c->nf))) return rc;
      CU(cudaMemcpyAsync(body_dev.p, c->h_body.data(), size_t(c->nf), cudaMemcpyHostToDevice, c->stream));
    }
    CU(cudaEventRecord(ev.e[0], c->stream));
    DevPacking packed;
    const int rc = pack_rows(c, c->nv, c->nv, c->nf, c->d_tri.p, body_dev.p, packed);
    CU(cudaEventRecord(ev.e[1], c->stream));
    CU(cudaEventSynchronize(ev.e[1]));
    float pack_ms = 0.f;
    CU(cudaEventElapsedTime(&pack_ms, ev.e[0], ev.e[1]));
    c->eq_ms[2] = pack_ms;
    if (rc) {  // the flipped rows do not pack: back to the rows and packing the context had
      const std::string why = g_err;
      CU(cudaMemcpy(c->d_tri.p, c->h_tri.data(), nh * sizeof(int32_t), cudaMemcpyHostToDevice));
      return fail(rc, "equiangulation: " + why + "; the context keeps its previous triangles");
    }
    auto t0 = clock::now();
    std::vector<int32_t> rows(nh);
    CU(cudaMemcpy(rows.data(), c->d_tri.p, nh * sizeof(int32_t), cudaMemcpyDeviceToHost));
    c->eq_ms[1] = ms_since(t0);
    t0 = clock::now();
    c->h_tri.swap(rows);
    drop_connectivity_state(c);
    c->tri_ready = true;  // d_tri holds the new rows
    if (int rc2 = upload_packing(c, std::move(packed), c->nv)) return rc2;
    if (c->has_gamma)
      if (int rc2 = upload_slot_gamma(c)) return rc2;
    c->eq_ms[3] = ms_since(t0);
  }
  if (n_flips) *n_flips = total;
  if (n_sweeps) *n_sweeps = sweeps;
  return 0;
}

int ms_ctx_equiangulate_stats(const ms_ctx* c, double* ms4, int32_t* rounds, int32_t capacity, int32_t* n_sweeps_run) {
  if (!c || !n_sweeps_run) return fail(-1, "null argument");
  *n_sweeps_run = int32_t(c->eq_rounds.size());
  if (ms4) std::copy(c->eq_ms, c->eq_ms + 4, ms4);
  if (rounds)
    for (int32_t i = 0; i < capacity && size_t(i) < c->eq_rounds.size(); ++i) rounds[i] = c->eq_rounds[size_t(i)];
  return 0;
}

int ms_ctx_get_triangles(const ms_ctx* c, int32_t* out) {
  if (!c || !out) return fail(-1, "null argument");
  if (!c->have_topology) return fail(-2, "ms_ctx_set_topology has not been called");
  for (size_t i = 0; i < c->h_tri.size(); ++i) {
    const int32_t x = c->h_tri[i];
    out[i] = (!c->perm.empty() && x >= 0 && x < c->nv) ? c->perm[size_t(x)] : x;
  }
  return 0;
}

int ms_ctx_refine(ms_ctx* c, int32_t levels, int32_t* nv_out, int32_t* nf_out) {
  if (int rc = check_ctx(c, true)) return rc;
  if (c->n_owned != c->nv) return fail(-5, "refinement is not available on a partitioned context");
  if (levels < 0) return fail(-1, "levels must be >= 0");
  if (!c->has_positions) return fail(-4, "no positions have been set (MS_ARR_POSITIONS)");
  for (int32_t x : c->h_tri)
    if (x < 0 || x >= c->nv) return fail(-1, "a facet has a vertex index outside [0, nv)");
  bool tilt_field = c->d_tilts.p != nullptr;
  for (const auto& lf : c->leaflet) tilt_field = tilt_field || lf.tilts.p != nullptr;
  if (c->has_kappa || c->has_c0 || tilt_field)
    return fail(-6, "refinement does not set per-vertex kappa / c0 or tilts at the midpoints: refine on the host "
                    "(geometry/refine.py refine_triangles), then ms_ctx_set_topology and upload them again");
  // without facets every level only renumbers the vertices: one level gives the result of any number
  const int32_t runs = c->nf == 0 ? std::min(levels, 1) : levels;
  for (int64_t l = 0, nf = c->nf; l < runs; ++l, nf *= 4) {
    if (3 * nf > INT32_MAX) return fail(-1, "refinement: more than 2^31 - 1 half-edges in a level");
    if (4 * nf > INT32_MAX) return fail(-1, "refinement: more than 2^31 - 1 facets");
  }
  std::fill(c->rf_ms, c->rf_ms + 4, 0.0);
  if (nv_out) *nv_out = c->nv;
  if (nf_out) *nf_out = c->nf;
  if (runs == 0) return 0;
  if (int rc = ensure_tri(c)) return rc;
  NvtxRange range("ms_b200 refine");
  using clock = std::chrono::steady_clock;
  auto ms_since = [](clock::time_point t0) { return std::chrono::duration<double, std::milli>(clock::now() - t0).count(); };
  struct Events {  // the device time; the context's own events belong to ms_ctx_timer_*
    cudaEvent_t e[2] = {nullptr, nullptr};
    ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
  } ev;
  CU(cudaEventCreate(&ev.e[0]));
  CU(cudaEventCreate(&ev.e[1]));
  const int32_t nf0 = c->nf;
  const bool fx = c->has_fixed, bd = c->has_boundary;
  // Scratch, released on return; the context changes only after everything is built, allocated and packed.
  // Levels run in the caller's numbering (the first reads the context's rows through key_id) into double buffers.
  DevBuf<double> lpos[2];
  DevBuf<uint8_t> lfixed[2], lbnd[2], temp;
  DevBuf<int32_t> ltri[2], h_in, order, flag, scan, edge, head;
  DevBuf<uint64_t> key_in, keys;
  ms::EqMesh m{c->nv, c->nf, c->d_tri.p, c->d_pos.p, fx ? c->d_fixed.p : nullptr,
               c->perm.empty() ? nullptr : c->d_perm.p, nullptr, nullptr};
  const uint8_t* bnd = bd ? c->d_boundary.p : nullptr;
  CU(cudaEventRecord(ev.e[0], c->stream));
  for (int32_t l = 0; l < runs; ++l) {
    const size_t nh = 3 * size_t(m.nf);
    size_t tb = 0;
    CU(ms::rf_temp_bytes(int64_t(nh), &tb));
    for (int rc : {key_in.ensure(nh), keys.ensure(nh), h_in.ensure(nh), order.ensure(nh), flag.ensure(nh),
                   scan.ensure(nh), edge.ensure(nh + 1), head.ensure(nh + 1), temp.ensure(tb + 1)})
      if (rc) return rc;
    CU(ms::launch_eq_sort_edges(m, key_in.p, h_in.p, keys.p, order.p, temp.p, tb, c->stream));
    m.keys = keys.p;
    m.order = order.p;
    CU(ms::launch_rf_edges(m, flag.p, scan.p, edge.p, head.p, temp.p, tb, c->stream));
    int32_t ne = 0;
    if (nh) {
      CU(cudaMemcpyAsync(&ne, scan.p + nh - 1, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
    }
    if (int64_t(m.nv) + ne > INT32_MAX) return fail(-1, "refinement: more than 2^31 - 1 vertices");
    const size_t nv2 = size_t(m.nv) + size_t(ne), nf2 = 4 * size_t(m.nf);
    const int i = l & 1;
    for (int rc : {lpos[i].ensure(3 * nv2), fx ? lfixed[i].ensure(nv2) : 0, bd ? lbnd[i].ensure(nv2) : 0,
                   ltri[i].ensure(3 * nf2)})
      if (rc) return rc;
    const ms::RfMesh r{m, bnd, head.p, edge.p, ne};
    const ms::RfOut o{lpos[i].p, lfixed[i].p, lbnd[i].p, ltri[i].p};
    CU(ms::launch_rf_build(r, o, c->stream));
    m = ms::EqMesh{int32_t(nv2), int32_t(nf2), ltri[i].p, lpos[i].p, fx ? lfixed[i].p : nullptr, nullptr, nullptr, nullptr};
    bnd = bd ? lbnd[i].p : nullptr;
  }
  // the internal vertex order of the refined mesh: the Morton order of its positions, as set_topology would choose it
  const size_t nv2 = size_t(m.nv), nf2 = size_t(m.nf), n3 = 3 * nv2;
  DevBuf<ms::MortonBox> boxes;
  DevBuf<int32_t> perm2, inv2, tri_int, bnd32;
  DevBuf<double> pos_int, grad, volgrad, seeds, stage;
  DevBuf<uint8_t> fixed_int, bnd_int;
  {
    size_t tb = 0;
    CU(ms::rf_temp_bytes(int64_t(nv2), &tb));
    for (int rc : {boxes.ensure(1 + ms::kRfBoxBlocks), key_in.ensure(nv2), keys.ensure(nv2), h_in.ensure(nv2),
                   perm2.ensure(nv2), inv2.ensure(nv2), temp.ensure(tb + 1), tri_int.ensure(3 * nf2 + 1),
                   pos_int.ensure(n3), grad.ensure(n3), volgrad.ensure(n3), seeds.ensure(ms::kSeedStride * nv2),
                   fx ? fixed_int.ensure(nv2) : 0, bd ? bnd_int.ensure(nv2) : 0, bd ? bnd32.ensure(nv2 + 1) : 0})
      if (rc) return rc;
    CU(ms::launch_rf_morton(m.pos, m.nv, boxes.p, key_in.p, h_in.p, keys.p, perm2.p, inv2.p, temp.p, tb, c->stream));
  }
  CU(ms::launch_gather_rows(m.pos, 3, perm2.p, int64_t(nv2), pos_int.p, c->stream));
  CU(ms::launch_rf_renumber(m.tri, int64_t(3 * nf2), inv2.p, tri_int.p, c->stream));
  if (fx) CU(ms::launch_rf_gather_flags(m.fixed, perm2.p, int64_t(nv2), fixed_int.p, nullptr, c->stream));
  if (bd) {
    CU(cudaMemsetAsync(bnd32.p, 0, (nv2 + 1) * sizeof(int32_t), c->stream));
    CU(ms::launch_rf_gather_flags(bnd, perm2.p, int64_t(nv2), bnd_int.p, bnd32.p, c->stream));
  }
  if (n3) {
    CU(cudaMemsetAsync(grad.p, 0, n3 * sizeof(double), c->stream));
    CU(cudaMemsetAsync(volgrad.p, 0, n3 * sizeof(double), c->stream));
  }
  CU(cudaEventRecord(ev.e[1], c->stream));
  CU(cudaEventSynchronize(ev.e[1]));
  float dev_ms = 0.f;
  CU(cudaEventElapsedTime(&dev_ms, ev.e[0], ev.e[1]));
  c->rf_ms[0] = dev_ms;
  // children inherit their parent's per-facet values: child j of the last level descends from facet j mod nf0
  auto t0 = clock::now();
  std::vector<uint8_t> body;
  std::vector<double> gamma;
  DevBuf<uint8_t> body_dev;
  if (!c->h_body.empty()) {
    body.resize(nf2);
    for (size_t j = 0; j < nf2; ++j) body[j] = c->h_body[j % size_t(nf0)];
    if (int rc = body_dev.ensure(nf2)) return rc;
    CU(cudaMemcpyAsync(body_dev.p, body.data(), nf2, cudaMemcpyHostToDevice, c->stream));
  }
  if (!c->h_gamma.empty()) {
    gamma.resize(nf2);
    for (size_t j = 0; j < nf2; ++j) gamma[j] = c->h_gamma[j % size_t(nf0)];
  }
  const double inherit_ms = ms_since(t0);
  // the refined rows are packed where they are
  CU(cudaEventRecord(ev.e[0], c->stream));
  DevPacking packed;
  const int prc = pack_rows(c, m.nv, m.nv, m.nf, tri_int.p, body_dev.p, packed);
  CU(cudaEventRecord(ev.e[1], c->stream));
  CU(cudaEventSynchronize(ev.e[1]));
  float pack_ms = 0.f;
  CU(cudaEventElapsedTime(&pack_ms, ev.e[0], ev.e[1]));
  c->rf_ms[2] = pack_ms;
  if (prc) return fail(prc, "refinement: " + std::string(g_err) + "; the context keeps its previous mesh");
  // only the rows (for h_tri) and the order come back
  t0 = clock::now();
  std::vector<int32_t> rows(3 * nf2), new_perm(nv2);
  if (nf2) CU(cudaMemcpy(rows.data(), tri_int.p, 3 * nf2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (nv2) CU(cudaMemcpy(new_perm.data(), perm2.p, nv2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
  c->rf_ms[1] = ms_since(t0);
  t0 = clock::now();
  bool identity = true;
  for (size_t v = 0; v < nv2 && identity; ++v) identity = new_perm[v] == int32_t(v);
  if (identity) new_perm.clear();
  if (!new_perm.empty())
    if (int rc = stage.ensure(ms::kSeedStride * nv2)) return rc;
  // commit
  c->nv = c->n_owned = m.nv;
  c->nf = m.nf;
  c->h_tri.swap(rows);
  c->perm.swap(new_perm);
  c->h_body.swap(body);
  c->h_gamma.swap(gamma);
  c->d_pos.swap(pos_int);
  c->d_grad.swap(grad);
  c->d_volgrad.swap(volgrad);
  c->d_seeds.swap(seeds);
  c->d_tri.swap(tri_int);
  if (!c->perm.empty()) {
    c->d_perm.swap(perm2);
    c->d_stage.swap(stage);
  }
  if (fx) c->d_fixed.swap(fixed_int);
  if (bd) {
    c->d_boundary.swap(bnd_int);
    c->d_boundary32.swap(bnd32);
  }
  drop_connectivity_state(c);
  c->tri_ready = true;  // d_tri holds the new rows
  // per-vertex arrays of the previous size: produced again on demand
  for (DevBuf<double>* b : {&c->d_trial, &c->d_dir, &c->d_tilt_grad, &c->d_tilt_sq, &c->d_kvecs, &c->d_avor, &c->d_aeff,
                            &c->d_evert})
    b->release();
  for (auto& lf : c->leaflet) lf.tilt_grad.release();
  if (int rc = upload_packing(c, std::move(packed), c->nv)) return rc;
  if (c->has_gamma)
    if (int rc = upload_slot_gamma(c)) return rc;
  c->rf_ms[3] = ms_since(t0) + inherit_ms;
  if (nv_out) *nv_out = c->nv;
  if (nf_out) *nf_out = c->nf;
  return 0;
}

int ms_ctx_refine_stats(const ms_ctx* c, double* ms4) {
  if (!c || !ms4) return fail(-1, "null argument");
  std::copy(c->rf_ms, c->rf_ms + 4, ms4);
  return 0;
}

int ms_ctx_dots(ms_ctx* c) {
  if (int rc = check_ctx(c, true)) return rc;
  if (int rc = flush_projection(c)) return rc;
  CU(ms::launch_dots(c->d_grad.p, c->d_volgrad.p, 3 * int64_t(c->n_owned), c->d_dot_partials.p, kDotBlocks,
                     c->d_scalars.p, c->stream));
  return 0;
}

int ms_ctx_direction_from_gradient(ms_ctx* c, double scale) {
  if (int rc = check_ctx(c, true)) return rc;
  if (int rc = ensure_array(c, MS_ARR_DIRECTION)) return rc;
  if (c->proj.active) {  // d = scale * (g + coef gC), fixed rows zero: the projection rides the pass that forms d
    if (c->n_owned < c->nv)
      CU(cudaMemsetAsync(c->d_dir.p + 3 * size_t(c->n_owned), 0, 3 * size_t(c->nv - c->n_owned) * sizeof(double), c->stream));
    CU(ms::launch_scale_projected(c->d_grad.p, c->proj.use_gc ? c->d_volgrad.p : nullptr,
                                  c->proj.use_fixed ? c->d_fixed.p : nullptr, c->n_owned, c->d_scalars.p, scale, c->d_dir.p,
                                  c->stream));
    return 0;
  }
  CU(ms::launch_scale(c->d_grad.p, scale, c->d_dir.p, 3 * int64_t(c->nv), c->stream));
  return 0;
}

int ms_ctx_axpy(ms_ctx* c, int dst, int src, double alpha, int32_t skip_fixed) {
  if (int rc = check_ctx(c, true)) return rc;
  if (dst == MS_ARR_GRAD || src == MS_ARR_GRAD || dst == MS_ARR_VOLGRAD)
    if (int rc = flush_projection(c)) return rc;
  int64_t ld = 0, ls = 0;
  double* d = array_ptr(c, dst, &ld);
  double* s = array_ptr(c, src, &ls);
  if (!d || !s || ld != ls || ld != 3 * int64_t(c->nv)) return fail(-1, "ms_ctx_axpy needs two allocated (nv,3) arrays");
  CU(ms::launch_axpy_rows(s, alpha, (skip_fixed && c->has_fixed) ? c->d_fixed.p : nullptr, c->nv, d, c->stream));
  return 0;
}

int ms_ctx_cg_direction(ms_ctx* c, int32_t restart) {
  if (int rc = check_ctx(c, true)) return rc;
  if (int rc = flush_projection(c)) return rc;
  if (int rc = ensure_array(c, MS_ARR_DIRECTION)) return rc;
  const int64_t nv = c->nv;
  if (restart || !c->d_cg_prev_g.p || c->d_cg_prev_g.n < size_t(3 * nv)) {
    CU(ms::launch_scale(c->d_grad.p, -1.0, c->d_dir.p, 3 * nv, c->stream));
    return 0;
  }
  CU(ms::launch_cg_direction(c->d_grad.p, c->d_cg_prev_g.p, c->d_cg_prev_d.p, c->has_fixed ? c->d_fixed.p : nullptr,
                             nv, c->d_dir.p, c->stream));
  return 0;
}

int ms_ctx_cg_commit(ms_ctx* c) {
  if (int rc = check_ctx(c, true)) return rc;
  if (int rc = flush_projection(c)) return rc;
  if (!c->d_dir.p) return fail(-4, "no search direction exists");
  const size_t n3 = 3 * size_t(c->nv);
  if (int rc = c->d_cg_prev_g.ensure(n3 + 1)) return rc;
  if (int rc = c->d_cg_prev_d.ensure(n3 + 1)) return rc;
  CU(cudaMemcpyAsync(c->d_cg_prev_g.p, c->d_grad.p, n3 * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_cg_prev_d.p, c->d_dir.p, n3 * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  return 0;
}

// the reductions of ms_ctx_line_search_stats, left on the device (d_ls_bits, scalars); needs d_tri and d_ls_bits
static int enqueue_line_search_stats(ms_ctx* c) {
  CU(ms::launch_ls_init(c->d_ls_bits.p, c->stream));
  CU(ms::launch_min_edge2(c->d_tri.p, c->nf, c->nv, c->d_pos.p, c->d_ls_bits.p, c->stream));
  CU(ms::launch_max_row_norm2(c->d_dir.p, c->n_owned, c->d_ls_bits.p + 1, c->stream));
  // <g,g>, <g,d>, <d,d> with the deterministic two-level sum; they land in the scalar vector
  if (c->proj.active)
    CU(ms::launch_dots_projected(c->d_grad.p, c->proj.use_gc ? c->d_volgrad.p : nullptr,
                                 c->proj.use_fixed ? c->d_fixed.p : nullptr, c->d_dir.p, c->n_owned, c->d_dot_partials.p,
                                 kDotBlocks, c->d_scalars.p, c->stream));
  else
    CU(ms::launch_dots(c->d_grad.p, c->d_dir.p, 3 * int64_t(c->n_owned), c->d_dot_partials.p, kDotBlocks,
                       c->d_scalars.p, c->stream));
  return 0;
}

int ms_ctx_line_search_stats(ms_ctx* c, double* out4) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!out4) return fail(-1, "null argument");
  if (!c->d_dir.p) return fail(-4, "no search direction exists (ms_ctx_direction_from_gradient / MS_ARR_DIRECTION)");
  if (int rc = ensure_tri(c)) return rc;
  if (int rc = c->d_ls_bits.ensure(4)) return rc;
  if (int rc = enqueue_line_search_stats(c)) return rc;
  unsigned long long bits[4];
  double sc[MS_SC_COUNT];
  CU(cudaMemcpyAsync(bits, c->d_ls_bits.p, sizeof(bits), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(sc, c->d_scalars.p, sizeof(sc), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  ms::ms_min_ls_stats(bits, sc, c->nf, out4);  // min edge length, largest row norm of d, <g,d>, <g,g>
  return 0;
}

int ms_ctx_normal_change_ok(ms_ctx* c, double limit_radians, int32_t* ok) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!ok) return fail(-1, "null argument");
  // beyond pi the cosine rule no longer orders the angles (cos(2 pi) == cos(0))
  if (!(limit_radians >= 0.0 && limit_radians <= 3.141592653589793)) return fail(-1, "limit_radians must lie in [0, pi]");
  if (!c->d_trial.p) return fail(-4, "no trial positions exist");
  if (int rc = ensure_tri(c)) return rc;
  if (int rc = c->d_ls_bits.ensure(4)) return rc;
  int* flag = reinterpret_cast<int*>(c->d_ls_bits.p + 2);
  CU(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
  CU(ms::launch_normal_change(c->d_tri.p, c->nf, c->nv, c->d_pos.p, c->d_trial.p, std::cos(limit_radians), flag,
                              c->stream));
  int host_flag = 0;
  CU(cudaMemcpyAsync(&host_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *ok = host_flag ? 0 : 1;
  return 0;
}

// ---- ms_ctx_minimize: the loop of DeviceMinimizer.minimize as one CUDA graph -------------------------------------
// Graph: WHILE(run) { k_min_control -> IF(act == k) { launches of action k } for every action k the options can
// reach }.  The control kernel reads the scalars the last action left on the device, advances the state machine of
// ms_minimize.cuh and opens the IF node of the next action; MN_DONE closes the WHILE node.  Each action's body is
// captured from the same entry points the host loop calls, so the launches (and their bits) are the same.
}  // extern "C"
namespace {

// the evaluation options DeviceMinimizer._opts / _enforce / the drift check build
ms_eval_opts min_eval_opts(const ms::MinOpts& o, bool want_grad, bool use_trial) {
  ms_eval_opts e;
  std::memset(&e, 0, sizeof(e));
  e.modules = o.modules | (o.volume_mode >= 0 ? MS_MOD_VOLUME : 0u);
  e.flags = o.flags;
  e.want_grad = want_grad;
  e.constraint_mode = o.volume_mode;
  e.k_vol = o.k_vol;
  e.v_target = o.v_target;
  e.apply_fixed = 1;
  e.use_trial = use_trial;
  e.patch_count = -1;
  return e;
}

ms_eval_opts volume_eval_opts(bool want_grad, bool use_trial) {
  ms_eval_opts e;
  std::memset(&e, 0, sizeof(e));
  e.modules = MS_MOD_VOLUME;
  e.want_grad = want_grad;
  e.constraint_mode = -1;
  e.use_trial = use_trial;
  e.patch_count = -1;
  return e;
}

// record the launches of fn() into `body` (a conditional node's graph) instead of running them
template <class F>
int capture_into(ms_ctx* c, cudaGraph_t body, F&& fn) {
  CU(cudaStreamBeginCaptureToGraph(c->mn_stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  cudaStream_t saved = c->stream;
  c->stream = c->mn_stream;
  const int rc = fn();
  c->stream = saved;
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(c->mn_stream, &g);
  if (rc) return rc;
  CU(e);
  return 0;
}

int add_conditional(cudaGraph_t graph, const cudaGraphNode_t* dep, size_t n_dep, cudaGraphConditionalHandle h,
                    cudaGraphConditionalNodeType type, cudaGraph_t* body) {
  alignas(cudaGraphNodeParams) unsigned char raw[sizeof(cudaGraphNodeParams)] = {};  // zeroed (no default constructor)
  cudaGraphNodeParams& p = *reinterpret_cast<cudaGraphNodeParams*>(raw);
  p.type = cudaGraphNodeTypeConditional;
  p.conditional.handle = h;
  p.conditional.type = type;
  p.conditional.size = 1;
  cudaGraphNode_t node;
  CU(cudaGraphAddNode(&node, graph, dep, n_dep, &p));
  *body = p.conditional.phGraph_out[0];
  return 0;
}

struct GraphHolder {
  cudaGraph_t g = nullptr;
  cudaGraphExec_t exec = nullptr;
  ~GraphHolder() {
    if (exec) cudaGraphExecDestroy(exec);
    if (g) cudaGraphDestroy(g);
  }
};

// the launches of action k (captured into its IF node)
int minimize_action(ms_ctx* c, const ms::MinOpts& o, int k, ms::MinState* st, const ms_ctx::PendingProjection& p_grad) {
  const int64_t nv = c->nv;
  switch (k) {
    case ms::MN_EVAL_GRAD: {
      const ms_eval_opts e = min_eval_opts(o, true, false);
      return ms_ctx_eval_async(c, &e);
    }
    case ms::MN_DIRECTION:
      c->proj = p_grad;  // what the gradient evaluation left
      if (o.stepper == 0) return ms_ctx_direction_from_gradient(c, -1.0);
      if (int rc = flush_projection(c)) return rc;
      CU(ms::launch_cg_direction(c->d_grad.p, c->d_cg_prev_g.p, c->d_cg_prev_d.p, c->has_fixed ? c->d_fixed.p : nullptr,
                                 nv, c->d_dir.p, c->stream, &st->cg_restart));
      return ms_ctx_cg_commit(c);
    case ms::MN_STATS:
      c->proj = p_grad;
      if (o.stepper == 1) c->proj.active = false;  // the conjugate-gradient direction applied it in place
      return enqueue_line_search_stats(c);
    case ms::MN_EVAL_ENERGY: case ms::MN_EVAL_TRIAL: {
      const ms_eval_opts e = min_eval_opts(o, false, k == ms::MN_EVAL_TRIAL);
      return ms_ctx_eval_async(c, &e);
    }
    case ms::MN_MAKE_TRIAL:
      CU(ms::launch_axpy(c->d_pos.p, c->d_dir.p, 0.0, c->d_trial.p, 3 * nv, c->stream, &st->alpha));
      return 0;
    case ms::MN_GUARD: {
      int* flag = reinterpret_cast<int*>(c->d_ls_bits.p + 2);
      CU(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
      CU(ms::launch_normal_change(c->d_tri.p, c->nf, c->nv, c->d_pos.p, c->d_trial.p, std::cos(0.5), flag, c->stream));
      return 0;
    }
    case ms::MN_ENF_EVAL_POS: case ms::MN_ENF_EVAL_TRIAL: {
      const ms_eval_opts e = volume_eval_opts(true, k == ms::MN_ENF_EVAL_TRIAL);
      return ms_ctx_eval_async(c, &e);
    }
    case ms::MN_ENF_AXPY_POS: case ms::MN_ENF_AXPY_TRIAL:
      CU(ms::launch_axpy_rows(c->d_volgrad.p, 0.0, c->has_fixed ? c->d_fixed.p : nullptr, nv,
                              k == ms::MN_ENF_AXPY_TRIAL ? c->d_trial.p : c->d_pos.p, c->stream, &st->neg_lam));
      return 0;
    case ms::MN_ACCEPT:
      CU(cudaMemcpyAsync(c->d_pos.p, c->d_trial.p, 3 * size_t(nv) * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
      return 0;
    case ms::MN_DRIFT_EVAL: {
      const ms_eval_opts e = volume_eval_opts(false, false);
      return ms_ctx_eval_async(c, &e);
    }
    default: return fail(-1, "unknown action");
  }
}

bool action_reachable(const ms::MinOpts& o, int k) {
  switch (k) {
    case ms::MN_ENF_EVAL_POS: case ms::MN_ENF_AXPY_POS: return o.enforce_volume != 0;
    case ms::MN_ENF_EVAL_TRIAL: case ms::MN_ENF_AXPY_TRIAL: return o.enforce_volume && o.projection_during;
    case ms::MN_DRIFT_EVAL: return o.enforce_volume && o.volume_mode == 0 && !o.projection_during;
    default: return true;
  }
}

// build and instantiate the graph; the host mirrors the captures touch are restored by the caller
int minimize_build(ms_ctx* c, const ms::MinOpts& o, int32_t hist_cap, const ms_ctx::PendingProjection& p_grad,
                   int32_t ran_a_grad, GraphHolder& gh) {
  CU(cudaGraphCreate(&gh.g, 0));
  ms::MinHandles h;
  std::memset(&h, 0, sizeof(h));
  CU(cudaGraphConditionalHandleCreate(&h.run, gh.g, 1, cudaGraphCondAssignDefault));
  cudaGraph_t loop;
  if (int rc = add_conditional(gh.g, nullptr, 0, h.run, cudaGraphCondTypeWhile, &loop)) return rc;
  for (int k = 0; k < ms::MN_ACTIONS; ++k)
    if (action_reachable(o, k)) {
      CU(cudaGraphConditionalHandleCreate(&h.act[k], loop, 0, 0));
      h.present |= 1u << k;
    }
  ms::MinState* st = c->d_min_state.p;
  if (int rc = capture_into(c, loop, [&] {
        CU(ms::launch_min_control(o, st, c->d_scalars.p, c->d_ls_bits.p, c->nf, c->d_min_hist.p, hist_cap,
                                  p_grad.active ? 1 : 0, ran_a_grad, h, c->stream));
        return 0;
      }))
    return rc;
  cudaGraphNode_t ctrl;
  size_t n_nodes = 1;
  CU(cudaGraphGetNodes(loop, &ctrl, &n_nodes));
  for (int k = 0; k < ms::MN_ACTIONS; ++k) {
    if (!(h.present & (1u << k))) continue;
    cudaGraph_t body;
    if (int rc = add_conditional(loop, &ctrl, 1, h.act[k], cudaGraphCondTypeIf, &body)) return rc;
    if (int rc = capture_into(c, body, [&] { return minimize_action(c, o, k, st, p_grad); })) return rc;
  }
  CU(cudaGraphInstantiate(&gh.exec, gh.g, 0));
  return 0;
}

}  // namespace
extern "C" {

int ms_ctx_minimize(ms_ctx* c, const ms_minimize_opts* opts, int32_t n_steps, ms_minimize_result* io, double* history,
                    int32_t capacity) {
  if (int rc = check_ctx(c, true)) return rc;
  if (!opts || !io) return fail(-1, "null argument");
  if (c->n_owned != c->nv) return fail(-6, "ms_ctx_minimize runs on single-context meshes (not on a partition)");
  if (n_steps < 0) return fail(-1, "n_steps must be >= 0");
  if (capacity < 0 || (capacity > 0 && !history)) return fail(-1, "history capacity without a history buffer");
  if (!ms::ms_min_valid(*opts)) return fail(-1, "ms_minimize_opts outside the supported bounds");
  if (!c->has_positions) return fail(-4, "no positions uploaded");
  if (c->packed.patches.empty()) return fail(-2, "the mesh has no patches");
  const ms::MinOpts o = *opts;
  const size_t n3 = 3 * size_t(c->nv);
  // a committed conjugate-gradient pair exists (ms_ctx_cg_direction restarts without one); the buffers allocated below
  // for the captured launches do not hold one
  const bool cg_valid = c->d_cg_prev_g.p && c->d_cg_prev_g.n >= n3;
  int64_t host_syncs = c->tri_ready ? 1 : 2;  // the final synchronise, and the blocking row upload of ensure_tri
  // every allocation before anything is enqueued: the captured launches must find their buffers in place
  for (int w : {MS_ARR_TRIAL, MS_ARR_DIRECTION})
    if (int rc = ensure_array(c, w)) return rc;
  if (o.modules & MS_MOD_TILT) {
    if (!c->d_tilts.p) return fail(-5, "tilt module requested but no tilts were uploaded");
    if (int rc = c->d_tilt_sq.ensure(size_t(c->nv) + 1)) return rc;
    if (int rc = ensure_array(c, MS_ARR_TILT_GRAD)) return rc;
  }
  if (o.stepper == 1) {
    if (int rc = c->d_cg_prev_g.ensure(n3 + 1)) return rc;
    if (int rc = c->d_cg_prev_d.ensure(n3 + 1)) return rc;
  }
  if (int rc = ensure_tri(c)) return rc;
  if (int rc = c->d_ls_bits.ensure(4)) return rc;
  if (!c->d_ticket.p) {
    if (int rc = c->d_ticket.ensure(4)) return rc;
    CU(cudaMemsetAsync(c->d_ticket.p, 0, 4 * sizeof(unsigned int), c->stream));
  }
  if (int rc = c->d_min_state.ensure(1)) return rc;
  const int32_t hist_rows = std::max<int32_t>(n_steps, 1);
  if (int rc = c->d_min_hist.ensure(4 * size_t(hist_rows))) return rc;
  const size_t rows_back = size_t(std::min(capacity, hist_rows));
  if (!c->h_min_state) CU(cudaMallocHost(reinterpret_cast<void**>(&c->h_min_state), sizeof(ms::MinState)));
  if (rows_back > c->h_min_hist_n) {
    if (c->h_min_hist) cudaFreeHost(c->h_min_hist);
    c->h_min_hist = nullptr;
    c->h_min_hist_n = 0;
    CU(cudaMallocHost(reinterpret_cast<void**>(&c->h_min_hist), 4 * rows_back * sizeof(double)));
    c->h_min_hist_n = rows_back;
  }
  if (!c->mn_stream) CU(cudaStreamCreateWithFlags(&c->mn_stream, cudaStreamNonBlocking));
  for (cudaEvent_t& e : c->mn_ev)
    if (!e) CU(cudaEventCreate(&e));

  // the projection an MN_EVAL_GRAD leaves pending, and whether it runs pass A
  const ms_eval_opts eg = min_eval_opts(o, true, false);
  ms_ctx::PendingProjection p_grad;
  projection_of(c, &eg, p_grad.use_gc, p_grad.use_fixed);
  p_grad.active = p_grad.use_gc || p_grad.use_fixed;
  const int32_t ran_a_grad = needs_bending(&eg) ? 1 : 0;

  const auto t0 = std::chrono::steady_clock::now();
  const ms_ctx::PendingProjection proj0 = c->proj;
  const bool ran_a0 = c->ran_pass_a;
  GraphHolder gh;
  const int brc = minimize_build(c, o, hist_rows, p_grad, ran_a_grad, gh);
  c->proj = proj0;  // the captures ran nothing: the host mirrors stay as they were
  c->ran_pass_a = ran_a0;
  if (brc) return brc;
  c->mn_ms[1] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();

  ms::MinState& s = *c->h_min_state;
  std::memset(&s, 0, sizeof(s));
  s.step_size = io->step_size;
  s.cg_iter = io->cg_iter;
  s.cg_have_history = io->cg_have_history ? 1 : 0;
  s.cg_valid = cg_valid ? 1 : 0;
  s.n_steps = n_steps;
  s.pc = ms::PC_START;
  s.proj_active = -1;  // unchanged until an action changes it
  s.last_ran_a = -1;
  CU(cudaMemcpyAsync(c->d_min_state.p, &s, sizeof(s), cudaMemcpyHostToDevice, c->stream));
  CU(cudaEventRecord(c->mn_ev[0], c->stream));
  CU(cudaGraphLaunch(gh.exec, c->stream));
  CU(cudaEventRecord(c->mn_ev[1], c->stream));
  CU(cudaMemcpyAsync(&s, c->d_min_state.p, sizeof(s), cudaMemcpyDeviceToHost, c->stream));
  if (rows_back)
    CU(cudaMemcpyAsync(c->h_min_hist, c->d_min_hist.p, 4 * rows_back * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // the one host synchronisation of the call
  if (rows_back) std::memcpy(history, c->h_min_hist, 4 * rows_back * sizeof(double));
  float dev_ms = 0.0f;
  CU(cudaEventElapsedTime(&dev_ms, c->mn_ev[0], c->mn_ev[1]));

  if (s.proj_active == 0) c->proj = ms_ctx::PendingProjection();
  if (s.proj_active == 1) c->proj = p_grad;
  if (s.last_ran_a >= 0) c->ran_pass_a = s.last_ran_a != 0;
  if (s.n_accepted > 0) c->has_positions = true;
  io->step_size = s.step_size;
  io->cg_iter = s.cg_iter;
  io->cg_have_history = s.cg_have_history;
  io->energy = s.res_energy;
  io->grad_norm = s.res_has_grad_norm ? s.res_grad_norm : 0.0;
  io->iterations = s.res_iterations;
  io->terminated_early = s.res_terminated_early;
  io->step_success = s.res_step_success;
  io->has_grad_norm = s.res_has_grad_norm;
  io->n_history = s.n_hist;
  c->mn_counts[0] = s.n_hist;
  c->mn_counts[1] = s.n_trials;
  c->mn_counts[2] = s.n_evals;
  c->mn_counts[3] = host_syncs;
  c->mn_counts[4] = s.n_actions;
  c->mn_counts[5] = s.n_guards;
  c->mn_counts[6] = s.n_guard_rejects;
  c->mn_ms[0] = dev_ms;
  return 0;
}

int ms_ctx_minimize_stats(const ms_ctx* c, int64_t* counts7, double* ms2) {
  if (!c) return fail(-1, "null context");
  if (counts7) std::copy(c->mn_counts, c->mn_counts + 7, counts7);
  if (ms2) std::copy(c->mn_ms, c->mn_ms + 2, ms2);
  return 0;
}

int ms_ctx_timer_start(ms_ctx* c) {
  if (int rc = check_ctx(c, false)) return rc;
  CU(cudaEventRecord(c->ev0, c->stream));
  return 0;
}

int ms_ctx_timer_stop(ms_ctx* c, float* ms_out) {
  if (int rc = check_ctx(c, false)) return rc;
  if (!ms_out) return fail(-1, "null argument");
  CU(cudaEventRecord(c->ev1, c->stream));
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaEventElapsedTime(ms_out, c->ev0, c->ev1));
  return 0;
}

int ms_ctx_sync(ms_ctx* c) {
  if (int rc = check_ctx(c, false)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

int ms_ctx_event_record(ms_ctx* c, int32_t index) {
  if (int rc = check_ctx(c, false)) return rc;
  if (index < 0 || index >= (1 << 16)) return fail(-1, "event index out of range");
  if (size_t(index) >= c->events.size()) c->events.resize(size_t(index) + 1, nullptr);
  if (!c->events[size_t(index)]) CU(cudaEventCreate(&c->events[size_t(index)]));
  CU(cudaEventRecord(c->events[size_t(index)], c->stream));
  return 0;
}

int ms_ctx_event_elapsed(ms_ctx* c, int32_t from, int32_t to, float* ms_out) {
  if (int rc = check_ctx(c, false)) return rc;
  if (!ms_out || from < 0 || to < 0 || size_t(from) >= c->events.size() || size_t(to) >= c->events.size() ||
      !c->events[size_t(from)] || !c->events[size_t(to)])
    return fail(-1, "event was never recorded");
  CU(cudaEventSynchronize(c->events[size_t(to)]));
  CU(cudaEventElapsedTime(ms_out, c->events[size_t(from)], c->events[size_t(to)]));
  return 0;
}

int ms_ctx_flush_l2(ms_ctx* c, int64_t bytes) {
  if (int rc = check_ctx(c, false)) return rc;
  if (bytes <= 0) return 0;
  if (int rc = c->d_flush.ensure(size_t(bytes))) return rc;
  CU(cudaMemsetAsync(c->d_flush.p, 1, size_t(bytes), c->stream));
  return 0;
}

int ms_host_register(void* ptr, int64_t bytes) {
  CU(cudaHostRegister(ptr, size_t(bytes), cudaHostRegisterDefault));
  return 0;
}

int ms_host_unregister(void* ptr) {
  CU(cudaHostUnregister(ptr));
  return 0;
}

// --------------------------------------------------------------------------
// Stateless shims.  Each call: copy in, build the corner CSR on the host, run
// the facet kernel + deterministic gather, copy out.  No state is kept.
// --------------------------------------------------------------------------
namespace {

struct SoupDev {
  DevBuf<double> pos;
  DevBuf<int32_t> tri, ptr, idx;
  ms::SoupArgs args;
};

int soup_setup(int32_t nv, int32_t nf, const double* pos, const int32_t* tri, int32_t zero_based,
               bool need_csr, SoupDev& d) {
  int n = 0;
  if (int rc = ms_device_count(&n)) return rc;
  if (n <= 0) return fail(-7, "no CUDA device: the B200 path has no CPU fallback");
  if (nv < 0 || nf < 0 || (nv > 0 && !pos) || (nf > 0 && !tri)) return fail(-1, "bad arguments");
  if (int rc = d.pos.ensure(3 * size_t(nv) + 1)) return rc;
  if (int rc = d.tri.ensure(3 * size_t(nf) + 1)) return rc;
  if (nv) CU(cudaMemcpy(d.pos.p, pos, 3 * size_t(nv) * sizeof(double), cudaMemcpyHostToDevice));
  if (nf) CU(cudaMemcpy(d.tri.p, tri, 3 * size_t(nf) * sizeof(int32_t), cudaMemcpyHostToDevice));
  const int32_t shift = zero_based ? 0 : -1;
  if (need_csr) {
    std::vector<int32_t> t;
    const int32_t* tz = tri;
    if (shift) {
      t.assign(tri, tri + 3 * size_t(nf));
      for (auto& x : t) x += shift;
      tz = t.data();
    }
    std::vector<int32_t> ptr, idx;
    ms::build_corner_csr(nv, nf, tz, ptr, idx);
    if (int rc = d.ptr.ensure(ptr.size())) return rc;
    if (int rc = d.idx.ensure(idx.size() + 1)) return rc;
    CU(cudaMemcpy(d.ptr.p, ptr.data(), ptr.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (!idx.empty()) CU(cudaMemcpy(d.idx.p, idx.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  d.args.nv = nv;
  d.args.nf = nf;
  d.args.pos = d.pos.p;
  d.args.tri = d.tri.p;
  d.args.csr_ptr = d.ptr.p;
  d.args.csr_idx = d.idx.p;
  d.args.shift = shift;
  return 0;
}

int to_dev(DevBuf<double>& b, const double* host, size_t n) {
  if (int rc = b.ensure(n + 1)) return rc;
  if (n) CU(cudaMemcpy(b.p, host, n * sizeof(double), cudaMemcpyHostToDevice));
  return 0;
}

int to_host(double* host, const DevBuf<double>& b, size_t n) {
  if (n && host) CU(cudaMemcpy(host, b.p, n * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace

int ms_surface_energy_and_gradient(int32_t nv, int32_t nf, const double* pos, const int32_t* tri,
                                   const double* gamma, double* grad, double* energy,
                                   int32_t zero_based) {
  if (!energy || (nv > 0 && !grad) || (nf > 0 && !gamma)) return fail(-1, "null argument");
  SoupDev d;
  if (int rc = soup_setup(nv, nf, pos, tri, zero_based, true, d)) return rc;
  DevBuf<double> d_gamma, d_corner, d_fe, d_grad, d_e;
  if (int rc = to_dev(d_gamma, gamma, size_t(nf))) return rc;
  if (int rc = to_dev(d_grad, grad, 3 * size_t(nv))) return rc;
  if (int rc = d_corner.ensure(9 * size_t(nf) + 1)) return rc;
  if (int rc = d_fe.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_e.ensure(1)) return rc;
  CU(ms::launch_soup_surface(d.args, d_gamma.p, d_corner.p, d_fe.p, d_grad.p, d_e.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (int rc = to_host(grad, d_grad, 3 * size_t(nv))) return rc;
  return to_host(energy, d_e, 1);
}

int ms_volume_and_gradient(int32_t nv, int32_t nf, const double* pos, const int32_t* tri,
                           double factor, double* grad, double* volume) {
  if (!volume) return fail(-1, "null argument");
  SoupDev d;
  if (int rc = soup_setup(nv, nf, pos, tri, 1, true, d)) return rc;
  DevBuf<double> d_corner, d_fv, d_grad, d_v;
  if (grad)
    if (int rc = to_dev(d_grad, grad, 3 * size_t(nv))) return rc;
  if (int rc = d_corner.ensure(9 * size_t(nf) + 1)) return rc;
  if (int rc = d_fv.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_v.ensure(1)) return rc;
  CU(ms::launch_soup_volume(d.args, factor, d_corner.p, d_fv.p, grad ? d_grad.p : nullptr, d_v.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (grad)
    if (int rc = to_host(grad, d_grad, 3 * size_t(nv))) return rc;
  return to_host(volume, d_v, 1);
}

int ms_grad_cotan_batch(int32_t n, const double* u, const double* v, double* gu, double* gv) {
  int nd = 0;
  if (int rc = ms_device_count(&nd)) return rc;
  if (nd <= 0) return fail(-7, "no CUDA device: the B200 path has no CPU fallback");
  if (n < 0 || (n > 0 && (!u || !v || !gu || !gv))) return fail(-1, "bad arguments");
  DevBuf<double> du, dv, dgu, dgv;
  if (int rc = to_dev(du, u, 3 * size_t(n))) return rc;
  if (int rc = to_dev(dv, v, 3 * size_t(n))) return rc;
  if (int rc = dgu.ensure(3 * size_t(n) + 1)) return rc;
  if (int rc = dgv.ensure(3 * size_t(n) + 1)) return rc;
  CU(ms::launch_grad_cotan(n, du.p, dv.p, dgu.p, dgv.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (int rc = to_host(gu, dgu, 3 * size_t(n))) return rc;
  return to_host(gv, dgv, 3 * size_t(n));
}

int ms_apply_beltrami_laplacian(int32_t dim, int32_t nv, int32_t nf, const double* weights,
                                const int32_t* tri, const double* field, double* out,
                                int32_t zero_based) {
  if (dim < 1 || (nf > 0 && !weights) || (nv > 0 && (!field || !out))) return fail(-1, "bad arguments");
  SoupDev d;
  DevBuf<double> dummy;
  if (int rc = dummy.ensure(4)) return rc;
  // positions are not used by this kernel; pass the field buffer shape-compatibly
  std::vector<double> zero_pos(3 * size_t(nv), 0.0);
  if (int rc = soup_setup(nv, nf, zero_pos.data(), tri, zero_based, true, d)) return rc;
  DevBuf<double> d_w, d_f, d_corner, d_out;
  if (int rc = to_dev(d_w, weights, 3 * size_t(nf))) return rc;
  if (int rc = to_dev(d_f, field, size_t(dim) * size_t(nv))) return rc;
  if (int rc = d_corner.ensure(3 * size_t(dim) * size_t(nf) + 1)) return rc;
  if (int rc = d_out.ensure(size_t(dim) * size_t(nv) + 1)) return rc;
  CU(ms::launch_soup_laplacian(d.args, dim, d_w.p, d_f.p, d_corner.p, d_out.p, nullptr));
  CU(cudaDeviceSynchronize());
  return to_host(out, d_out, size_t(dim) * size_t(nv));
}

int ms_p1_triangle_divergence(int32_t nv, int32_t nf, const double* pos, const double* tilts,
                              const int32_t* tri, double* div_tri, double* area, double* g0,
                              double* g1, double* g2, int32_t zero_based) {
  if ((nv > 0 && !tilts) || (nf > 0 && (!div_tri || !area || !g0 || !g1 || !g2))) return fail(-1, "null argument");
  SoupDev d;
  if (int rc = soup_setup(nv, nf, pos, tri, zero_based, false, d)) return rc;
  DevBuf<double> d_t, d_div, d_area, d_g0, d_g1, d_g2;
  if (int rc = to_dev(d_t, tilts, 3 * size_t(nv))) return rc;
  if (int rc = d_div.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_area.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_g0.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_g1.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_g2.ensure(3 * size_t(nf) + 1)) return rc;
  CU(ms::launch_p1_divergence(d.args, d_t.p, d_div.p, d_area.p, d_g0.p, d_g1.p, d_g2.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (int rc = to_host(div_tri, d_div, size_t(nf))) return rc;
  if (int rc = to_host(area, d_area, size_t(nf))) return rc;
  if (int rc = to_host(g0, d_g0, 3 * size_t(nf))) return rc;
  if (int rc = to_host(g1, d_g1, 3 * size_t(nf))) return rc;
  return to_host(g2, d_g2, 3 * size_t(nf));
}

int ms_p1_vertex_divergence(int32_t nv, int32_t nf, const double* pos, const double* tilts, const int32_t* tri,
                            double* div_v, double* area_v, int32_t zero_based) {
  if ((nv > 0 && (!tilts || !div_v || !area_v))) return fail(-1, "null argument");
  SoupDev d;
  if (int rc = soup_setup(nv, nf, pos, tri, zero_based, true, d)) return rc;
  DevBuf<double> d_t, d_div, d_area, d_g0, d_g1, d_g2, d_dv, d_av;
  if (int rc = to_dev(d_t, tilts, 3 * size_t(nv))) return rc;
  if (int rc = d_div.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_area.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_g0.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_g1.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_g2.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_dv.ensure(size_t(nv) + 1)) return rc;
  if (int rc = d_av.ensure(size_t(nv) + 1)) return rc;
  CU(ms::launch_p1_divergence(d.args, d_t.p, d_div.p, d_area.p, d_g0.p, d_g1.p, d_g2.p, nullptr));
  CU(ms::launch_p1_vertex_divergence(d.args, d_div.p, d_area.p, d_dv.p, d_av.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (int rc = to_host(div_v, d_dv, size_t(nv))) return rc;
  return to_host(area_v, d_av, size_t(nv));
}

int ms_compute_curvature_data(int32_t nv, int32_t nf, const double* pos, const int32_t* tri,
                              double* k_vecs, double* vertex_areas, double* weights,
                              int32_t zero_based, double* va0, double* va1, double* va2) {
  if ((nv > 0 && (!k_vecs || !vertex_areas)) || (nf > 0 && !weights)) return fail(-1, "null argument");
  SoupDev d;
  if (int rc = soup_setup(nv, nf, pos, tri, zero_based, true, d)) return rc;
  DevBuf<double> d_corner, d_k, d_a, d_w, d_va0, d_va1, d_va2;
  if (int rc = d_corner.ensure(12 * size_t(nf) + 1)) return rc;
  if (int rc = d_k.ensure(3 * size_t(nv) + 1)) return rc;
  if (int rc = d_a.ensure(size_t(nv) + 1)) return rc;
  if (int rc = d_w.ensure(3 * size_t(nf) + 1)) return rc;
  if (int rc = d_va0.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_va1.ensure(size_t(nf) + 1)) return rc;
  if (int rc = d_va2.ensure(size_t(nf) + 1)) return rc;
  CU(ms::launch_soup_curvature(d.args, d_corner.p, d_k.p, d_a.p, d_w.p, d_va0.p, d_va1.p, d_va2.p, nullptr));
  CU(cudaDeviceSynchronize());
  if (int rc = to_host(k_vecs, d_k, 3 * size_t(nv))) return rc;
  if (int rc = to_host(vertex_areas, d_a, size_t(nv))) return rc;
  if (int rc = to_host(weights, d_w, 3 * size_t(nf))) return rc;
  if (int rc = to_host(va0, d_va0, size_t(nf))) return rc;
  if (int rc = to_host(va1, d_va1, size_t(nf))) return rc;
  return to_host(va2, d_va2, size_t(nf));
}

}  // extern "C"
