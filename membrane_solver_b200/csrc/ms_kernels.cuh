// Kernel launch interface between the C-ABI layer (ms_capi.cu) and the kernels
// (ms_kernels.cu).  Plain structs of device pointers; no torch types.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ms_b200.h"
#include "ms_bt.cuh"
#include "ms_leaflet.cuh"
#include "ms_math.cuh"
#include "ms_pack.h"
#include "ms_equiangulate.cuh"
#include "ms_minimize.cuh"
#include "ms_pack_device.cuh"
#include "ms_refine.cuh"
#include "ms_vertex_average.cuh"

namespace ms {

// Slots of the per-evaluation scalar vector (device, 16 doubles).
enum ScalarSlot : int {
  SC_E_SURFACE = 0,
  SC_AREA = 1,
  SC_VOLUME = 2,       // body volume (already divided by 6)
  SC_E_BENDING = 3,
  SC_E_TILT = 4,
  SC_E_BENDING_TILT = 5,
  SC_G_G = 8,          // <g,g>
  SC_G_GC = 9,         // <g,gC>
  SC_GC_GC = 10,       // <gC,gC>
  SC_LAMBDA = 11,      // KKT multiplier applied
  SC_COEF = 12,        // projected gradient = g + SC_COEF * gC (then fixed rows zeroed); 0 without a constraint
  SC_COUNT = 16,
};
constexpr int kPartialStride = 12;  // per-patch partial sums: slots 0..11 above

constexpr int kSeedStride = 5;  // per-vertex pass-A output: fK(3), fA_eff, fA_vor

// Compile-time capacities of a patch in shared memory (strides of the structure-of-arrays
// staging buffers).  The run-time pack parameters must not exceed them.
constexpr int kPatchOwnedCap = 512;   // owned vertices per patch
constexpr int kPatchLocalCap = 896;   // owned + halo vertices per patch
constexpr int kPatchSlotCap = 1536;   // record slots per patch (rounds x threads)
#ifndef MS_CONSUMER_THREADS
#define MS_CONSUMER_THREADS 448
#endif
constexpr int kConsumerThreads = MS_CONSUMER_THREADS;  // + one epilogue warp + one producer warp per CTA
constexpr int kMaxConsumerWarps = kConsumerThreads / 32;
constexpr int kMaxGroups = 14;        // thread groups taking turns (named barriers 1..14)

// Fused finalisation of an evaluation: the LAST persistent CTA of a pass to finish (ticket) adds up the per-CTA
// rows of both passes in fixed order, writes the scalar vector and the KKT coefficient -- no reduce / project launches.
struct PatchFinalize {
  unsigned int* ticket;       // zeroed counter; nullptr: this launch does not finalise
  const double* partials_a;   // per-CTA rows of pass A (rows_a of them; 0: pass A did not run)
  const double* partials_b;   // per-CTA rows of pass B
  int32_t rows_a, rows_b;
  uint32_t b_mask;            // slot k comes from pass B's rows when bit k is set, else from pass A's
  int32_t constraint_mode;    // -2 leave the coefficient alone (energy-only evaluation); -1 none; 0 lagrange;
                              // 1 penalty (constraint_manager.py:294-301, body.py:223-238)
  int32_t has_gc;             // the volume gradient takes part in the projection
  double k_vol, v_target;
  double* scalars;            // nullptr: no reduction (the ticket only raises signal_flag)
  // partitioned evaluations over peer memory (see k_halo_pull / k_allreduce_gather): the last CTA can also
  unsigned long long* signal_flag;    // raise this rank's "owned rows are written" flag (pass A: the seeds) ...
  unsigned long long signal_epoch;
  unsigned long long* publish_words;  // ... and publish the local scalars into the all-reduce slot of this epoch
  unsigned long long publish_epoch;
  // push transport: the local scalars go into the slot of this rank in EVERY rank's block (remote stores), then the
  // arrival word of this rank there is raised
  unsigned long long* const* push_words;   // flag blocks of all ranks (device table, own block included)
  int32_t push_slots, push_my_slot;
  // gather in the same CTA: after publishing, wait for every rank's publish flag, add the slots in rank order and
  // write the KKT coefficient from the GLOBAL sums (mode gather_mode) -- the evaluation of a partition is then two
  // launches, like the evaluation of a whole mesh
  unsigned long long* const* gather_words;  // non-null: flag blocks of all ranks
  int32_t gather_slots, gather_mode;
  int* gather_error;
};

// Halo exchange INSIDE a patch kernel (partitioned meshes, peer memory).  The launch walks the interior patches first
// (patch_list); meanwhile the epilogue warps of every CTA wait for the owners' flags and copy a slice of the ghost rows
// out of the owners' arrays; the producer warp of a CTA waits for `arrived` to reach `arrived_target` (every CTA has
// copied its slice) only before it stages its first patch that reads ghost rows.  The exchange, the skew between the
// ranks included, hides behind the interior patches, and no separate signal / pull launch is needed.
struct HaloPull {
  int32_t n_ghost, width;            // n_ghost == 0: nothing to pull
  const double* const* peer_base;    // array of every owner slot
  unsigned long long* const* peer_flag;
  int32_t n_slots, flag_index;
  unsigned long long epoch;          // what every owner's flag must have reached
  const int32_t* owner;              // per ghost row: owner slot, row in the owner's array
  const int32_t* row;
  double* dst;                       // first ghost row of the local array
  unsigned long long* own_flag;      // non-null: block 0 raises it (epoch) when the kernel starts -- the rows this rank
                                     // owns were written by the previous kernel of the stream
  unsigned int* arrived;             // monotonically increasing counter (one increment per CTA and launch)
  unsigned int arrived_target;
  int32_t first_boundary;            // position in the patch sequence of the first patch that reads ghost rows
  int32_t first_ghost_row;           // local rows >= this are ghost rows (read around L1: see stage_row)
  int* error;
};

struct PatchLaunch {
  // packed topology (device)
  const PatchHeader* patches;  // n_patches + 1 entries: a sentinel closes the slot ranges
  const int32_t* halo_ids;
  const FacetRec* recs;
  const double* slot_gamma;   // per-slot surface tension, or nullptr -> gamma_u
  int32_t patch_begin, patch_count;
  const int32_t* patch_list;  // optional indirection: the launch walks patch_list[patch_begin + i], i < patch_count
  int32_t partial_row0;       // first row of `partials` this launch writes (one row per CTA)
  int32_t max_ctas;           // > 0: launch at most this many persistent CTAs (leave SMs to NCCL kernels)
  int32_t threads;            // record slots per round = lanes of one consumer group
  int32_t max_owned, max_local;
  int32_t max_slots, max_rounds;  // largest record count / round count of any patch
  // mesh state (device)
  const double* pos;          // (nv,3)
  const double* tilts;        // (nv,3) or nullptr
  const uint8_t* is_boundary; // nv or nullptr
  const int32_t* boundary32;  // the same flags as int32 (cp.async staging), nullptr with is_boundary
  const double* tilt_sq;      // nv: |t|^2 per vertex (tilt magnitude module), nullptr without tilts
  const double* kappa;        // nv or nullptr -> kappa_u
  const double* c0;           // nv or nullptr -> c0_u
  double gamma_u, kappa_u, c0_u, k_tilt;
  uint32_t modules, flags;
  // outputs (device)
  double* seeds;      // (nv,kSeedStride)  pass A -> pass B
  double* partials;   // (grid, kPartialStride): one row of running sums per persistent CTA
  double* grad;       // (nv,3)   pass B
  double* volgrad;    // (nv,3)   pass B, when MS_MOD_VOLUME
  double* tilt_grad;  // (nv,3)   pass B, when tilt modules with tilt gradients requested
  // optional diagnostics written by pass A when non-null
  double* k_vecs;     // (nv,3)
  double* a_vor;      // nv
  double* a_eff;      // nv
  double* e_vertex;   // nv   per-vertex bending energy (bending.compute_energy_array)
  PatchFinalize fin;
  // push transport: before the first patch is staged the CTA waits until the arrival words of every source rank in
  // wait_mask (LOCAL memory, written by the peers) have reached wait_epoch: the ghost rows are then in place
  HaloPull pull;
  const unsigned long long* wait_flags;
  unsigned long long wait_epoch;
  uint64_t wait_mask;
  int* wait_error;
  int32_t debug;      // timing experiments only (MS_DEBUG_VARIANT; results are wrong): 1 no token ring, 2 no
                      // accumulation, 4 no per-facet compute
  int* self_check;    // -DMS_SELF_CHECK builds: three violation counters (device), else unused
};

size_t pass_a_smem_bytes(const PatchLaunch& a);
size_t pass_b_smem_bytes(const PatchLaunch& a);
int patch_grid(const PatchLaunch& a);  // persistent CTAs launched for this patch range (= partial rows)

// scalars_here: also sum the per-facet scalars (surface energy, area, volume).
cudaError_t launch_pass_a(const PatchLaunch& a, cudaStream_t st);
cudaError_t launch_pass_b(const PatchLaunch& a, bool bending, bool scalars_here, cudaStream_t st);
// scalars[0..11] = fixed-order sums of the per-CTA rows: slot k from pb when bit k of b_mask is set,
// else from pa; volume slot / 6.
cudaError_t launch_reduce_partials(const double* pa, int rows_a, const double* pb, int rows_b, unsigned b_mask,
                                   double* scalars, cudaStream_t st);
cudaError_t configure_kernels();  // SM count + opt-in to large dynamic shared memory (once per device)

// --- dense vector helpers on (n) doubles: KKT projection of the volume constraint ---
// scalars[SC_G_G, SC_G_GC, SC_GC_GC] <- deterministic dot products.
cudaError_t launch_dots(const double* g, const double* gc, int64_t n, double* block_partials,
                        int n_blocks, double* scalars, cudaStream_t st);
// mode 0: lagrange  g -= (<g,gC>/<gC,gC>) gC if <gC,gC> > 1e-18 (constraint_manager.py:294-301)
// mode 1: penalty   g += k (V - V0) gC (body.py:223-238); then g[fixed] = 0 in both modes.
cudaError_t launch_project(double* g, const double* gc, const uint8_t* fixed, int64_t nv,
                           double* scalars, int mode, double k_vol, double v_target,
                           cudaStream_t st);
// scalars[SC_COEF], scalars[SC_LAMBDA] from the dot products / the volume (one thread): the projection itself is
// applied by whoever consumes the gradient (launch_apply_projection, launch_scale_projected, launch_dots_projected)
cudaError_t launch_kkt_coefficient(double* scalars, int mode, int has_gc, double k_vol, double v_target, cudaStream_t st);
// g <- (g + scalars[SC_COEF] * gc) with fixed rows zeroed, in place (gc / fixed may be null)
cudaError_t launch_apply_projection(double* g, const double* gc, const uint8_t* fixed, int64_t nv, const double* scalars,
                                    cudaStream_t st);
// out <- scale * projected(g) without touching g
cudaError_t launch_scale_projected(const double* g, const double* gc, const uint8_t* fixed, int64_t nv,
                                   const double* scalars, double scale, double* out, cudaStream_t st);
// scalars[SC_G_G, SC_G_GC, SC_GC_GC] <- <p,p>, <p,d>, <d,d> with p = projected(g) formed on the fly
cudaError_t launch_dots_projected(const double* g, const double* gc, const uint8_t* fixed, const double* d, int64_t nv,
                                  double* block_partials, int n_blocks, double* scalars, cudaStream_t st);
// out[i*width + c] = src[rows[i]*width + c]: packs the rows a neighbouring partition needs
cudaError_t launch_gather_rows(const double* src, int width, const int32_t* rows, int64_t n,
                               double* out, cudaStream_t st);
// out[rows[i]*width + c] = src[i*width + c]: internal vertex order -> caller's order
cudaError_t launch_scatter_rows(const double* src, int width, const int32_t* rows, int64_t n,
                                double* out, cudaStream_t st);
// x_out = x + alpha * d  (trial positions of the line search, line_search.py:358-382); alpha_dev (device, may be
// null) replaces alpha
cudaError_t launch_axpy(const double* x, const double* d, double alpha, double* out, int64_t n,
                        cudaStream_t st, const double* alpha_dev = nullptr);

// --- generic (any triangle soup) kernels behind the stateless KernelSpec shims ---
struct SoupArgs {
  int32_t nv, nf;
  const double* pos;
  const int32_t* tri;
  const int32_t* csr_ptr;  // vertex -> corners
  const int32_t* csr_idx;
  int32_t shift;           // 0 for zero-based indices, -1 for one-based
};
cudaError_t launch_soup_surface(const SoupArgs& s, const double* gamma, double* corner /*nf*9*/,
                                double* facet_e /*nf*/, double* grad /*nv*3, +=*/,
                                double* energy_out, cudaStream_t st);
cudaError_t launch_soup_volume(const SoupArgs& s, double factor, double* corner, double* facet_v,
                               double* grad /*+=*/, double* volume_out, cudaStream_t st);
cudaError_t launch_soup_curvature(const SoupArgs& s, double* corner /*nf*12*/, double* k_vecs,
                                  double* vertex_areas, double* weights, double* va0, double* va1,
                                  double* va2, cudaStream_t st);
cudaError_t launch_soup_laplacian(const SoupArgs& s, int32_t dim, const double* weights,
                                  const double* field, double* corner /*nf*3*dim*/, double* out,
                                  cudaStream_t st);
cudaError_t launch_grad_cotan(int32_t n, const double* u, const double* v, double* gu, double* gv,
                              cudaStream_t st);
cudaError_t launch_p1_divergence(const SoupArgs& s, const double* tilts, double* div, double* area,
                                 double* g0, double* g1, double* g2, cudaStream_t st);
cudaError_t launch_p1_vertex_divergence(const SoupArgs& s, const double* div, const double* area, double* div_v,
                                       double* area_v, cudaStream_t st);
cudaError_t launch_sum(const double* x, int64_t n, double scale, double* out, cudaStream_t st);
// out[v] = |rows[v,:]|^2 of an (n,3) array (tilt magnitude staging)
cudaError_t launch_row_norm2(const double* rows, int64_t n, double* out, cudaStream_t st);

// --- line-search helpers of the device-resident loop ---
cudaError_t launch_min_edge2(const int32_t* tri, int32_t nf, int32_t nv, const double* pos,
                             unsigned long long* out, cudaStream_t st);
cudaError_t launch_max_row_norm2(const double* rows, int64_t n, unsigned long long* out, cudaStream_t st);
cudaError_t launch_normal_change(const int32_t* tri, int32_t nf, int32_t nv, const double* old_pos,
                                 const double* new_pos, double cos_limit, int* flag, cudaStream_t st);
cudaError_t launch_scale(const double* x, double scale, double* out, int64_t n, cudaStream_t st);
cudaError_t launch_axpy_rows(const double* x, double alpha, const uint8_t* fixed, int64_t nv, double* y,
                             cudaStream_t st, const double* alpha_dev = nullptr);
// restart_dev (device, may be null): when it holds a non-zero value, d = -1 * g (launch_scale) instead
cudaError_t launch_cg_direction(const double* g, const double* pg, const double* pd, const uint8_t* fixed,
                                int64_t nv, double* d, cudaStream_t st, const int32_t* restart_dev = nullptr);
// the initial words of launch_min_edge2 / launch_max_row_norm2 / launch_normal_change (4 words)
cudaError_t launch_ls_init(unsigned long long* bits, cudaStream_t st);

// --- loop control of ms_ctx_minimize (ms_minimize.cuh): condition handles of the graph's WHILE node and of the IF
// node of every action present (bit k of `present`) ---
struct MinHandles {
  cudaGraphConditionalHandle run;
  cudaGraphConditionalHandle act[MN_ACTIONS];
  uint32_t present;
};
// one thread: ms_min_step on the device state, then the condition values of the next action
cudaError_t launch_min_control(const MinOpts& o, MinState* s, const double* scalars, const unsigned long long* ls_bits,
                               int32_t nf, double* hist, int32_t hist_cap, int32_t proj_grad, int32_t ran_a_grad,
                               const MinHandles& h, cudaStream_t st);

constexpr int kSumBlocks = 592;  // partial sums of the two-stage fixed-order reductions (4 CTAs per SM)
// --- bending-tilt coupling on the resident mesh (ms_bt.cuh); corner holds 12*nf doubles, e_out 1 + kSumBlocks ---
// stage: divergence / effective areas -> vertex seeds (into `seeds`, read by pass B) and base term ->
// per-facet energy (sum into e_out) and, when tilt_grads, corner contributions of the tilt gradient
cudaError_t launch_bt_stage(const BtMesh& m, double sign, const double* k_vecs, const double* a_vor,
                            const double* a_eff, double* corner, double* seeds, double* base, double* facet_e,
                            double* e_out, bool tilt_grads, cudaStream_t st);
cudaError_t launch_bt_tilt_gather(const BtMesh& m, const double* corner3, double* tilt_grad, bool accumulate,
                                  cudaStream_t st);
cudaError_t launch_bt_finalize(const double* e_bt, double* scalars, cudaStream_t st);

// --- leaflet tilt modules (ms_leaflet.cuh).  corner: 27*nf doubles, vbuf: 5*nv, corner_shape / corner_tilt:
// 9*nf each, facet_e: 3*nf, e_out3: {E_bending_tilt, E_tilt, E_tilt_smoothness}, sum_scratch: 3*kSumBlocks doubles.  grad / tilt_grad may be null. ---
cudaError_t launch_leaflet(const LeafletMesh& m, bool with_bt, bool with_tilt, bool with_smooth, double* corner,
                           double* vbuf, double* corner_shape, double* corner_tilt, double* facet_e, double* e_out3,
                           double* sum_scratch, double* grad,
                           bool accumulate_grad, double* tilt_grad, bool accumulate_tilt_grad, cudaStream_t st);

// small meshes: the same evaluation as ONE cooperative launch (block_e: 3 * max_blocks doubles; ticket: one zeroed
// 64-bit word that is never reset; *ticket_base mirrors it on the host)
cudaError_t launch_leaflet_fused(const LeafletMesh& m, bool with_bt, bool with_tilt, bool with_smooth, double* corner,
                                 double* vbuf, double* corner_shape, double* corner_tilt, double* block_e, int max_blocks,
                                 double* e_out3, double* grad, bool accumulate_grad, double* tilt_grad,
                                 bool accumulate_tilt_grad, unsigned long long* ticket, unsigned long long* ticket_base,
                                 cudaStream_t st);
cudaError_t launch_leaflet_fused_pair(const LeafletMesh& m0, const LeafletMesh& m1, bool with_bt, bool with_tilt,
                                      bool with_smooth, double* const corner[2], double* const vbuf[2],
                                      double* const shape[2], double* const tilt[2], double* const e_out3[2],
                                      double* const tilt_grad[2], double* block_e /* 6 * max_blocks */, int max_blocks,
                                      double* grad, bool accumulate_grad, bool accumulate_tilt_grad,
                                      unsigned long long* ticket, unsigned long long* ticket_base, cudaStream_t st);
constexpr int kLfFusedMaxBlocks = 512;
constexpr int kLfFusedMaxItems = 1 << 16;  // facets / vertices up to which the single-launch variant is used

// --- halo exchange over NVLink peer memory (flag wait + peer loads in one kernel) ---
cudaError_t launch_halo_signal(unsigned long long* flag, unsigned long long epoch, cudaStream_t st);
cudaError_t launch_halo_pull(int n_ghost, int width, const double* const* peer_base, unsigned long long* const* peer_flag,
                             int n_slots, int flag_index, unsigned long long epoch, const int32_t* owner,
                             const int32_t* row, double* dst, int* error, cudaStream_t st);
cudaError_t launch_allreduce_peer(double* scalars, int n, unsigned long long* own_words, unsigned long long* const* peer_words,
                                  int n_slots, unsigned long long epoch, int* error, cudaStream_t st);
// signal + pull in one launch (multi-process only: the kernel waits for peers that run concurrently)
cudaError_t launch_halo_exchange(unsigned long long* own_flag, int n_ghost, int width, const double* const* peer_base,
                                 unsigned long long* const* peer_flag, int n_slots, int flag_index,
                                 unsigned long long epoch, const int32_t* owner, const int32_t* row, double* dst,
                                 int* error, cudaStream_t st);
// gather half of the all-reduce (the publish half ran in the last CTA of the pass) + KKT coefficient
cudaError_t launch_allreduce_gather_coef(double* scalars, int n, unsigned long long* const* peer_words, int n_slots,
                                         unsigned long long epoch, int mode, int has_gc, double k_vol, double v_target,
                                         int* error, cudaStream_t st);
cudaError_t launch_halo_warmup(unsigned long long* words, double* scalars, int* error, unsigned int* push_ticket,
                               cudaStream_t st);
constexpr int kFlagWords = 1024;  // exported block (words): [0..3] epoch flags of the pull transport, [8..39] 2 x 16 scalar
                                  // slots of the pull all-reduce; push transport: [64 + 64 kind + src] arrival epochs of
                                  // the halo rows (kind 0 positions, 1 seeds) and [192 + src] of the scalars pushed by
                                  // rank src, [256 + (16 parity + src) 16 + k] those scalars (world <= 16)
constexpr int kPushFlagBase = 64, kPushScalarFlagBase = 192, kPushScalarBase = 256, kPushMaxRanks = 16;
// PUSH transport: the owner stores its rows straight into the ghost slots of the ranks that list them (posted NVLink
// writes: nobody waits for a round trip) and then raises, in each of those ranks' flag blocks, the word that belongs to
// it; the receiver polls LOCAL memory only.  One launch; the last block to finish raises the flags.
cudaError_t launch_halo_push(int n_rows, int width, const double* src, double* const* peer_base, const int32_t* dst_slot,
                             const int32_t* src_row, const int32_t* dst_row, unsigned long long* const* peer_flags,
                             int n_slots, uint64_t dst_mask, int my_slot, int kind, unsigned long long epoch,
                             unsigned int* ticket, cudaStream_t st);
// gather of scalars that were PUSHED into this rank's block (k_patch's last CTA, PatchFinalize::push_*): local polls,
// rank-order sum, KKT coefficient
cudaError_t launch_allreduce_local_coef(double* scalars, int n, unsigned long long* own_words, int n_slots,
                                        unsigned long long epoch, int mode, int has_gc, double k_vol, double v_target,
                                        int* error, cudaStream_t st);

// --- leaflet tilt relaxation helpers ---
cudaError_t launch_vertex_normals(int32_t nv, const int32_t* tri, const int32_t* csr_ptr, const int32_t* csr_idx,
                                  const double* pos, double* normals, cudaStream_t st);
cudaError_t launch_project_tangent(int64_t nv, const double* normals, double* t, cudaStream_t st);
cudaError_t launch_tilt_trial(int64_t nv, const double* t, const double* g, const double* normals, const uint8_t* fixed,
                              double step, double* trial, cudaStream_t st);
cudaError_t launch_leaflet_jacobi(const LeafletMesh& m, bool use_keep, double k_smooth, const uint8_t* fixed, double* minv,
                                  cudaStream_t st);
cudaError_t launch_rz(int64_t nv, const double* g, const double* minv, double* rows, double* out, double* sum_scratch,
                      cudaStream_t st);
cudaError_t launch_tilt_cg_direction(int64_t nv, const double* g, const double* minv, double beta, bool restart, double* dir,
                                     cudaStream_t st);
cudaError_t launch_masked_norm2(int64_t nv, double* g, const uint8_t* fixed, double* rowsq, double* out,
                                double* sum_scratch, cudaStream_t st);

// --- vertex averaging (the `V` command): one thread per vertex, m.pos -> out (a different buffer) ---
cudaError_t launch_vertex_average(const VaMesh& m, double* out, cudaStream_t st);

// --- equiangulation (the `u` command), one sweep in four steps (ms_equiangulate.cuh) ---
// scratch of the sorts and the candidate selection for up to n_half_edges items
cudaError_t eq_temp_bytes(int64_t n_half_edges, size_t* bytes);
// half-edge keys (caller numbering) sorted stably with their half-edge ids into keys / order (= m.keys / m.order)
cudaError_t launch_eq_sort_edges(const EqMesh& m, uint64_t* key_in, int32_t* h_in, uint64_t* keys, int32_t* order,
                                 void* temp, size_t temp_bytes, cudaStream_t st);
// sorted positions of the interior edges that pass eq_should_flip, in ascending key; their count to *n_cand (device)
cudaError_t launch_eq_candidates(const EqMesh& m, uint8_t* flag, int32_t* cand_pos, int32_t* n_cand, void* temp,
                                 size_t temp_bytes, cudaStream_t st);
// fills s.h1 / s.h2 / s.slot_cand / s.nkey / s.nkey_cand / s.nkey_pos of the nc candidates
cudaError_t launch_eq_conflicts(const EqMesh& m, int32_t nc, const int32_t* cand_pos, const EqCands& s,
                                uint64_t* nkey_in, int32_t* id_in, void* temp, size_t temp_bytes, cudaStream_t st);
// one selection round in -> out; adds the candidates it leaves undecided to *undecided; does nothing when
// *prev_undecided (the previous round's count, may be null) is 0
cudaError_t launch_eq_round(const EqCands& s, const uint8_t* in, uint8_t* out, const int32_t* prev_undecided,
                            int32_t* undecided, cudaStream_t st);
// rewrites the rows of the selected candidates; adds their number to *flips
cudaError_t launch_eq_apply(const EqCands& s, const uint8_t* state, int32_t* tri, int32_t* flips, cudaStream_t st);


// --- refinement (the `r` command), one level in three steps, then the Morton order (ms_refine.cuh) ---
constexpr int kRfBoxBlocks = 296;  // blocks of the bounding-box reduction; boxes holds 1 + kRfBoxBlocks entries
// scratch of the key sorts and the scan for up to n items (half-edges of a level, or vertex rows)
cudaError_t rf_temp_bytes(int64_t n, size_t* bytes);
// from the sorted keys (m.keys / m.order, launch_eq_sort_edges): edge[h] = edge of half-edge h, head[e] = sorted
// position where the run of edge e starts and head[n_edges] = 3 nf; scan[3 nf - 1] = n_edges (device)
cudaError_t launch_rf_edges(const EqMesh& m, int32_t* flag, int32_t* scan, int32_t* edge, int32_t* head, void* temp,
                            size_t temp_bytes, cudaStream_t st);
// the refined vertex rows, flags and facet rows of one level into o
cudaError_t launch_rf_build(const RfMesh& r, const RfOut& o, cudaStream_t st);
// perm (new -> old) = morton_permutation of the n positions, before dropping an identity; inv = its inverse
cudaError_t launch_rf_morton(const double* pos, int32_t n, MortonBox* boxes, uint64_t* key_in, int32_t* id_in,
                             uint64_t* key_out, int32_t* perm, int32_t* inv, void* temp, size_t temp_bytes,
                             cudaStream_t st);
// out[i] = inv[rows[i]]
cudaError_t launch_rf_renumber(const int32_t* rows, int64_t n, const int32_t* inv, int32_t* out, cudaStream_t st);
// out[i] = src[perm[i]], and out32[i] = out[i] != 0 when out32 is set
cudaError_t launch_rf_gather_flags(const uint8_t* src, const int32_t* perm, int64_t n, uint8_t* out, int32_t* out32,
                                   cudaStream_t st);

// --- patch packing on the device (ms_pack_device.cuh): the layout of ms::pack_patches, byte for byte ---
// scratch of the corner sort for n_corners = 3 nf items
cudaError_t pk_temp_bytes(int64_t n_corners, size_t* bytes);
// corner CSR (corner ids 3 f + k by vertex, facet-major; the facets with an index out of range left out): csr_ptr
// gets nv + 1 offsets, csr_idx 3 nf entries of which the first csr_ptr[nv] are the CSR
cudaError_t launch_pk_corner_csr(const int32_t* tri, int32_t nv, int32_t nf, int32_t* key_in, int32_t* id_in,
                                 int32_t* key_out, int32_t* csr_idx, int32_t* csr_ptr, void* temp, size_t temp_bytes,
                                 cudaStream_t st);
// per chunk (3 n_chunks + 1 words, zeroed here): the pk_plan bounds; bounds[3 n_chunks] = facets with all indices in range
cudaError_t launch_pk_bounds(const PackParams& p, const int32_t* csr_ptr, int32_t n_owned, const int32_t* tri,
                             int32_t nv, int32_t nf, unsigned long long* bounds, int64_t n_chunks,
                             unsigned long long* n_valid, cudaStream_t st);
// one warp per chunk: pk_chunk into the staging
cudaError_t launch_pk_chunks(const PkMesh& m, int32_t* scratch, const PkStage& stage, PkChunk* chunks, int64_t n_chunks,
                             cudaStream_t st);
// concatenation in chunk order; bases = (first patch, first halo id, first slot) of every chunk
cudaError_t launch_pk_concat(const PkStage& stage, const PkChunk* chunks, const int64_t* bases, int64_t n_chunks,
                             PatchHeader* hdr, int32_t* halo, FacetRec* recs, int32_t* slot_facet, int64_t n_slots,
                             cudaStream_t st);
// out[0] = n_hw_groups, out[1] = n_hw_excess of the packing
cudaError_t launch_pk_hw_excess(const PatchHeader* hdr, int32_t n_patches, const FacetRec* recs, int32_t threads,
                                unsigned long long* out, cudaStream_t st);
// out[s] = gamma[slot_facet[s]], 0 for an empty slot
cudaError_t launch_pk_slot_gamma(const int32_t* slot_facet, int64_t n, const double* gamma, double* out, cudaStream_t st);
// self-check negative control: slot 1 of every patch's first round repeats slot 0
cudaError_t launch_pk_inject(const PatchHeader* hdr, int32_t n_patches, FacetRec* recs, cudaStream_t st);

}  // namespace ms
