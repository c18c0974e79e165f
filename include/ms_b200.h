/*
 * membrane_solver_b200 -- C ABI of the B200 (sm_100a) energy+gradient path.
 *
 * This is the drop-in boundary: everything the reference binds through
 * fortran_kernels/loader.py (KernelSpec getters, loader.py:15-20,30,85,139,193,247)
 * for the per-iteration energy/gradient evaluation is exported here as plain C:
 * `extern "C"`, raw pointers and sizes, caller-owned memory, int return codes.
 * 0 = success; any other value is an error and ms_last_error() describes it.
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Array conventions (identical to the reference's dense caches, SURVEY.md section 8):
 *   positions / gradients / tilts   (nv,3) C-order float64  (== Fortran (3,nv))
 *   triangle rows                   (nf,3) C-order int32
 *   per-facet / per-vertex params   float64; masks uint8 (0/1)
 * The callee never retains host pointers past the call.
 */
#ifndef MS_B200_H
#define MS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MS_API __attribute__((visibility("default")))

/* ---- module / flag bits for ms_eval_opts ------------------------------------ */
#define MS_MOD_SURFACE       (1u << 0) /* modules/energy/surface.py:100-239 */
#define MS_MOD_VOLUME        (1u << 1) /* geometry/body.py:150-252: V and dV/dx of the body */
#define MS_MOD_BENDING       (1u << 2) /* modules/energy/bending.py:90-181 */
#define MS_MOD_TILT          (1u << 3) /* modules/energy/tilt.py:99-172 */
#define MS_MOD_BENDING_TILT  (1u << 4) /* modules/energy/bending_tilt.py:151-482 (single field; not with MS_MOD_BENDING) */
#define MS_MOD_TILT_SMOOTHNESS (1u << 5) /* modules/energy/tilt_smoothness*.py (leaflet evaluation only: ms_ctx_eval_leaflet) */

#define MS_FLAG_WILLMORE     (1u << 0) /* bending_energy_model = willmore (bending_params.py:18-21) */
#define MS_FLAG_APPROX       (1u << 1) /* bending_gradient_mode = approx (bending_params.py:24-31) */

/* ---- scalar slots returned by the evaluation calls (16 doubles) --------------- */
#define MS_SC_E_SURFACE      0
#define MS_SC_AREA           1
#define MS_SC_VOLUME         2
#define MS_SC_E_BENDING      3
#define MS_SC_E_TILT         4
#define MS_SC_E_BENDING_TILT 5
#define MS_SC_G_G            8
#define MS_SC_G_GC           9
#define MS_SC_GC_GC          10
#define MS_SC_LAMBDA         11
#define MS_SC_COEF           12 /* projected gradient = g + MS_SC_COEF * gC */
#define MS_SC_COUNT          16

/* ---- device arrays addressable through ms_ctx_device_ptr / ms_ctx_get_array --- */
#define MS_ARR_POSITIONS     0  /* (nv,3) */
#define MS_ARR_GRAD          1  /* (nv,3) shape gradient of the enabled modules */
#define MS_ARR_VOLGRAD       2  /* (nv,3) dV/dx of the body */
#define MS_ARR_SEEDS         3  /* (nv,5) pass-A vertex results: fK(3), fA_eff, fA_vor */
#define MS_ARR_TILTS         4  /* (nv,3) */
#define MS_ARR_TILT_GRAD     5  /* (nv,3) */
#define MS_ARR_SCALARS       6  /* 16 */
#define MS_ARR_K_VECS        7  /* (nv,3) integrated curvature vectors (diagnostic) */
#define MS_ARR_A_VOR         8  /* nv */
#define MS_ARR_A_EFF         9  /* nv */
#define MS_ARR_E_VERTEX      10 /* nv  per-vertex bending energy (bending.compute_energy_array) */
#define MS_ARR_TRIAL         11 /* (nv,3) trial positions x + alpha d */
#define MS_ARR_DIRECTION     12 /* (nv,3) search direction d */
#define MS_ARR_TILTS_IN      13 /* (nv,3) inner-leaflet tilt field  (Mesh.tilts_in_view, geometry/mesh.py:425-460) */
#define MS_ARR_TILTS_OUT     14 /* (nv,3) outer-leaflet tilt field  (Mesh.tilts_out_view, geometry/mesh.py:462-499) */
#define MS_ARR_TILT_GRAD_IN  15 /* (nv,3) dE/dt_in  of the leaflet modules */
#define MS_ARR_TILT_GRAD_OUT 16 /* (nv,3) dE/dt_out of the leaflet modules */
#define MS_ARR_TILTS_FIELD   17 /* (nv,3) single tilt field evaluated through the leaflet sweeps (MS_LEAFLET_FIELD) */
#define MS_ARR_TILT_GRAD_FIELD 18 /* (nv,3) its tilt gradient */

#define MS_PATCHES_ALL       (-1)
#define MS_PATCHES_INTERIOR  (-2)
#define MS_PATCHES_BOUNDARY  (-3)

typedef struct ms_ctx ms_ctx;

typedef struct ms_eval_opts {
  uint32_t modules;        /* MS_MOD_* */
  uint32_t flags;          /* MS_FLAG_* */
  int32_t want_grad;       /* 0: energies only (line-search trial evaluation) */
  int32_t constraint_mode; /* -1 none; 0 lagrange KKT projection (constraint_manager.py:294-301);
                              1 penalty  g += k (V-V0) dV/dx (body.py:223-238) */
  double k_vol;            /* volume_stiffness (penalty mode) */
  double v_target;         /* body target volume */
  int32_t apply_fixed;     /* zero the gradient rows of fixed vertices (minimizer.py:988-990) */
  int32_t use_trial;       /* evaluate at MS_ARR_TRIAL instead of MS_ARR_POSITIONS */
  int32_t patch_begin;     /* range of patches to evaluate;  patch_count == -1: all patches */
  int32_t patch_count;     /* MS_PATCHES_INTERIOR / MS_PATCHES_BOUNDARY: the two halves of a partitioned
                              evaluation (patches without / with ghost rows in their halo) */
  int32_t diagnostics;     /* also write K_VECS / A_VOR / A_EFF / E_VERTEX */
  int32_t want_tilt_grad;  /* with want_grad == 0: still produce MS_ARR_TILT_GRAD (tilt-only evaluation,
                              evaluation_manager.py:693-698).  With MS_MOD_TILT this runs pass B, which overwrites
                              MS_ARR_GRAD and MS_ARR_VOLGRAD with the raw gradients of the modules and drops a
                              pending projection: evaluate with want_grad again before using the gradient */
} ms_eval_opts;

typedef struct ms_pack_info {
  int32_t nv, nf;
  int32_t n_patches, threads;
  int32_t max_owned, max_local, max_rounds;
  int32_t max_slots; /* largest record count of a patch */
  int64_t n_slots;   /* record slots streamed per pass */
  int64_t n_listed;  /* facet listings over all patches (ring facets counted per patch) */
  int64_t n_valid;   /* facets with all indices in range */
  int64_t n_halo;    /* halo vertex references over all patches */
  int64_t n_round_slots; /* sum over patches of rounds x threads (= n_slots) */
  int64_t n_lane_conflicts; /* facets sharing a bank residue with another facet of their half-warp */
  int64_t n_hw_groups;      /* (round, half-warp, corner) gather groups holding at least one facet */
  int64_t n_hw_excess;      /* extra shared-memory wavefronts over those groups (0 = conflict free) */
} ms_pack_info;

/* ---- library ------------------------------------------------------------------ */
MS_API const char* ms_last_error(void);
MS_API int ms_version(void);
MS_API int ms_device_count(int* count);

/* ---- stateful context: device-resident mesh (replaces the host caches of
 *      runtime/energy_context.py:63-276 and Mesh.positions_view/triangle_row_cache) - */
MS_API int ms_ctx_create(int device, ms_ctx** out);
MS_API int ms_ctx_destroy(ms_ctx* ctx);
/* patch geometry used by the next ms_ctx_set_topology (defaults 128 / 512 / 896; these are
 * also the compiled shared-memory capacities, so values may only be lowered) */
MS_API int ms_ctx_set_pack_params(ms_ctx* ctx, int32_t threads, int32_t max_owned, int32_t max_local);
/* packer tuning for the next ms_ctx_set_topology: target share (percent) of record slots that
 * hold a facet (default 87; lower = more free lanes = fewer shared-memory bank clashes) and
 * the number of lane-placement repair passes (default 1) */
MS_API int ms_ctx_set_pack_tuning(ms_ctx* ctx, int32_t fill_pct, int32_t repair_sweeps);
/* launch at most max_ctas persistent CTAs per pass (0 = one per SM): a partitioned evaluation leaves a
 * few SMs to the NCCL kernels of the halo exchange that runs concurrently */
MS_API int ms_ctx_set_max_ctas(ms_ctx* ctx, int32_t max_ctas);
/* Optional: positions (nv,3) used ONLY to choose the internal vertex order of the next
 * ms_ctx_set_topology (Morton curve), so that meshes in arbitrary vertex order -- e.g. the
 * refinement order of runtime/refinement.py -- still pack into compact patches.  Transparent to
 * the caller: every host-side upload / download of a per-vertex array is in the caller's order;
 * only ms_ctx_device_ptr exposes internal rows (ms_ctx_get_permutation: internal row -> caller row).
 * Not used for partitions (n_owned < nv), which arrive ordered. */
MS_API int ms_ctx_set_vertex_order_hint(ms_ctx* ctx, int32_t nv, const double* pos);
MS_API int ms_ctx_get_permutation(const ms_ctx* ctx, int32_t* perm_new_to_old);
/* Re-called only after refine / equiangulate / vertex-average changed the topology
 * (commands/mesh_ops.py:21-78).  is_boundary, body_mask, fixed_mask may be NULL. */
MS_API int ms_ctx_set_topology(ms_ctx* ctx, int32_t nv, int32_t nf, const int32_t* tri,
                               const uint8_t* is_boundary, const uint8_t* body_mask,
                               const uint8_t* fixed_mask);
/* Multi-GPU partition: vertex rows [0, n_owned) are owned by this context, rows
 * [n_owned, nv) are ghost copies of vertices owned by other partitions (one ring around the
 * owned range).  Only owned rows get results; ghost rows of MS_ARR_POSITIONS (before an
 * evaluation) and MS_ARR_SEEDS (between pass A and pass B) are filled by the halo exchange. */
MS_API int ms_ctx_set_topology_partition(ms_ctx* ctx, int32_t nv, int32_t n_owned, int32_t nf,
                                         const int32_t* tri, const uint8_t* is_boundary,
                                         const uint8_t* body_mask, const uint8_t* fixed_mask);
/* rows of this partition that other partitions hold as ghosts (concatenated per destination) */
MS_API int ms_ctx_set_send_rows(ms_ctx* ctx, const int32_t* rows, int64_t n);
/* out_device[i, :] = array[send_rows[i], :] on the context stream (out is a DEVICE pointer) */
MS_API int ms_ctx_pack_send(ms_ctx* ctx, int which, void* out_device);
/* Replace the fixed-vertex mask (nv bytes, or NULL: no fixed vertex) without touching the packed topology: the
 * reference invalidates its fixed mask on its own counter (Mesh._fixed_flags_version, geometry/mesh.py:211-231),
 * independently of the topology versions. */
MS_API int ms_ctx_set_fixed_mask(ms_ctx* ctx, const uint8_t* fixed_mask);
MS_API int ms_ctx_pack_info(const ms_ctx* ctx, ms_pack_info* info);
/* patch p owns vertex rows [v_lo[p], v_lo[p+1]); v_lo has n_patches+1 entries */
MS_API int ms_ctx_patch_ranges(const ms_ctx* ctx, int32_t* v_lo);
/* halo vertex rows referenced by patches [patch_begin, patch_begin+patch_count) that lie
 * outside [own_lo, own_hi): sorted unique; returns the count through n (out may be NULL) */
MS_API int ms_ctx_halo_rows(const ms_ctx* ctx, int32_t patch_begin, int32_t patch_count,
                            int32_t own_lo, int32_t own_hi, int32_t* out, int64_t* n);
/* gamma == NULL: uniform surface tension (Mesh.get_facet_parameter_array, mesh.py:234-265) */
MS_API int ms_ctx_set_surface_tension(ms_ctx* ctx, const double* gamma, double gamma_uniform);
/* kappa / c0 == NULL: uniform (bending_params.py:41-115) */
MS_API int ms_ctx_set_bending_params(ms_ctx* ctx, const double* kappa, const double* c0,
                                     double kappa_uniform, double c0_uniform);
MS_API int ms_ctx_set_tilt_rigidity(ms_ctx* ctx, double k_tilt);
MS_API int ms_ctx_set_positions(ms_ctx* ctx, const double* pos_host);
MS_API int ms_ctx_set_tilts(ms_ctx* ctx, const double* tilts_host);
/* generic host<->device copies of a named array (count doubles from element offset).  Uploading MS_ARR_GRAD
 * replaces the gradient and drops a pending projection (ms_ctx_eval_async); uploading MS_ARR_VOLGRAD first applies a
 * pending projection with the gC the evaluation produced, so the gradient stays the one of that evaluation. */
MS_API int ms_ctx_upload(ms_ctx* ctx, int which, const double* host, int64_t offset, int64_t count);
MS_API int ms_ctx_get_array(ms_ctx* ctx, int which, double* host, int64_t offset, int64_t count);
/* Device pointer of a named array (internal row order).  For MS_ARR_GRAD and MS_ARR_VOLGRAD a pending projection is
 * applied first: the caller reads the projected gradient and may write gC without changing it.  ms_ctx_axpy with
 * dst == MS_ARR_VOLGRAD does the same. */
MS_API void* ms_ctx_device_ptr(ms_ctx* ctx, int which);
MS_API int64_t ms_ctx_array_len(const ms_ctx* ctx, int which);
MS_API int ms_ctx_set_stream(ms_ctx* ctx, void* cuda_stream);

/* ---- leaflet tilt modules: tilt_in / tilt_out, bending_tilt_in / bending_tilt_out ---------------
 * Replaces modules/energy/tilt_leaflet.py:26-169 (through tilt_in.py:34-61, tilt_out.py) and
 * modules/energy/bending_tilt_leaflet.py:231-758 (through bending_tilt_in.py, bending_tilt_out.py;
 * bt_payload.py:40-298, bt_gradient.py:20-64,89-389, bt_divergence.py:49-93), default numerical path:
 * ambient_v1 transport, analytic gradient mode.  The selections the reference derives from mesh options
 * arrive as masks in the CALLER's vertex / facet order; NULL means "none":
 *   facet_keep       nf   facets of the leaflet (leaflet_presence.py:34-170); NULL = all
 *   interior         nv   rows carrying a base term (bt_selection.py:289-330); NULL = not is_boundary
 *   base_zero        nv   rows whose base term is forced to 0 (assume-J0 presets, region rows)
 *   kappa, c0        nv   per-vertex leaflet parameters (bt_params.py:233-318); NULL = the defaults
 *   tilt_row_weight  nv   active-row weights of the tilt magnitude module (tilt_utils._active_row_weights)
 *   facet_consistent nf   mass mode per facet (1 = consistent, 0 = lumped); NULL = consistent_default
 * The geometric boundary mask is the one given to ms_ctx_set_topology.  Must be called again after
 * ms_ctx_set_topology. */
typedef struct ms_leaflet_desc {
  const uint8_t* facet_keep;
  const uint8_t* interior;
  const uint8_t* base_zero;
  const double* kappa;
  const double* c0;
  const double* tilt_row_weight;
  const uint8_t* facet_consistent;
  double kappa_default;     /* bending_modulus_in / _out */
  double c0_default;        /* spontaneous_curvature_in / _out */
  double k_tilt;            /* tilt_modulus_in / _out */
  double k_smooth;          /* tilt smoothness rigidity: bending_modulus_in / _out (tilt_smoothness_utils.py:77-84) */
  double div_sign;          /* -1 inner leaflet, +1 outer (bending_tilt_in.py:46, bending_tilt_out.py:46) */
  int32_t consistent_default;
  int32_t reserved;
} ms_leaflet_desc;

#define MS_LEAFLET_IN  0
#define MS_LEAFLET_OUT 1
#define MS_LEAFLET_FIELD 2  /* the single tilt field (modules/energy/tilt_smoothness.py:219-262): same sweeps, own arrays */
#define MS_ACC_GRAD      1u  /* add the shape gradient to MS_ARR_GRAD instead of overwriting it */
#define MS_ACC_TILT_GRAD 2u  /* add to MS_ARR_TILT_GRAD_IN / _OUT instead of overwriting */

MS_API int ms_ctx_set_leaflet(ms_ctx* ctx, int32_t leaflet, const ms_leaflet_desc* desc);
/* Evaluate the leaflet's modules (any of MS_MOD_TILT, MS_MOD_BENDING_TILT, MS_MOD_TILT_SMOOTHNESS) at MS_ARR_POSITIONS (or
 * MS_ARR_TRIAL) with the tilt field MS_ARR_TILTS_IN / _OUT.  want_grad: shape gradient into MS_ARR_GRAD;
 * want_tilt_grad: tilt gradient into MS_ARR_TILT_GRAD_IN / _OUT (want_grad == 0 is the tilt-only
 * evaluation of the inner relaxation loop, evaluation_manager.py:693-698).  MS_MOD_TILT_SMOOTHNESS
 * (modules/energy/tilt_smoothness_leaflet.py:17-79, cotangent Dirichlet energy of the tilt field) has a tilt
 * gradient only.  energies3, when not NULL,
 * receives {E_bending_tilt, E_tilt, E_tilt_smoothness} (synchronises the stream). */
MS_API int ms_ctx_eval_leaflet(ms_ctx* ctx, int32_t leaflet, uint32_t modules, int32_t want_grad,
                               int32_t want_tilt_grad, uint32_t accumulate, int32_t use_trial,
                               double* energies3);

/* --- leaflet tilt relaxation at frozen geometry (runtime/steppers/tilt_relaxation.py:426-1057, gradient-descent
 * solver; the host keeps the loop control, only scalars cross PCIe) ---
 * rows whose tilt is fixed (vertex flags tilt_fixed_in / tilt_fixed_out); NULL = none */
MS_API int ms_ctx_set_leaflet_fixed(ms_ctx* ctx, int32_t leaflet, const uint8_t* fixed_rows);
/* unit area-weighted vertex normals of MS_ARR_POSITIONS (Mesh.vertex_normals, geometry/triangle_ops.py:55-72),
 * kept on the device for the projections below */
MS_API int ms_ctx_update_vertex_normals(ms_ctx* ctx);
/* t -= (t.n) n on the leaflet's tilt field (runtime/projections/tilt.py:8-14) */
MS_API int ms_ctx_leaflet_project_tilts(ms_ctx* ctx, int32_t leaflet);
/* zero the fixed rows of MS_ARR_TILT_GRAD_IN / _OUT and return the sum of squares of the rest (:856-871);
 * norm2 may be NULL (result read later through ms_ctx_leaflet_results) */
MS_API int ms_ctx_leaflet_gradient_norm2(ms_ctx* ctx, int32_t leaflet, double* norm2);
/* Inner AND outer leaflet in one call (on meshes up to 32 768 facets: one cooperative launch for both); results
 * stay on the device (ms_ctx_leaflet_results).  The shape gradient is the inner leaflet's plus the outer one's,
 * bitwise what two ms_ctx_eval_leaflet calls (the second with MS_ACC_GRAD) leave. */
MS_API int ms_ctx_eval_leaflet_pair(ms_ctx* ctx, uint32_t modules, int32_t want_grad, int32_t want_tilt_grad,
                                    uint32_t accumulate, int32_t use_trial);
/* Batched read-back for loops that evaluate several leaflets per iteration: ms_ctx_eval_leaflet (energies3 ==
 * NULL), ms_ctx_leaflet_gradient_norm2 (norm2 == NULL) and ms_ctx_leaflet_rz (rz == NULL) leave their results on the
 * device; this call synchronises ONCE and returns, per leaflet slot l = 0..2, out15[5 l + {0,1,2}] = the three
 * energies of the last evaluation, [5 l + 3] = |g|^2, [5 l + 4] = r.z */
MS_API int ms_ctx_leaflet_results(ms_ctx* ctx, double* out15);
/* trial = P(t - step * tilt gradient) or, with along_direction, P(t + step * CG direction); fixed rows keep t
 * (build_leaflet_trial_tilts, projections/tilt.py:99-138) */
MS_API int ms_ctx_leaflet_make_trial(ms_ctx* ctx, int32_t leaflet, double step, int32_t along_direction);
/* preconditioned CG solver of the same loop (tilt_relaxation.py:1057-1440, runtime/preconditioners.py:64-146):
 * Jacobi inverse diagonal 1 / (k_tilt * barycentric area + k_smooth/2 * opposite cotangents); the area runs over the
 * leaflet's facets when kept_facets_only, else over every facet */
MS_API int ms_ctx_leaflet_build_preconditioner(ms_ctx* ctx, int32_t leaflet, double k_smooth, int32_t kept_facets_only);
/* rz = sum_v g_v . (M^-1 g_v) over the leaflet's tilt gradient (fixed rows were zeroed by ..._gradient_norm2) */
MS_API int ms_ctx_leaflet_rz(ms_ctx* ctx, int32_t leaflet, int32_t preconditioned, double* rz);
/* direction = -M^-1 g + beta * direction  (restart != 0: direction = -M^-1 g) */
MS_API int ms_ctx_leaflet_cg_direction(ms_ctx* ctx, int32_t leaflet, double beta, int32_t restart,
                                       int32_t preconditioned);
/* exchange the tilt field and the trial field: evaluate at the trial, swap back to reject */
MS_API int ms_ctx_leaflet_swap_trial(ms_ctx* ctx, int32_t leaflet);

/* ---- halo exchange over NVLink peer memory (multi-GPU, one process per GPU) --------------------------
 * Each rank exports CUDA IPC handles of its position / trial / seed arrays and of its flag words; the ranks that
 * hold ghosts of it open them.  ms_ctx_halo_signal publishes "my owned rows of the arrays guarded by this flag are
 * written" (stream-ordered); ms_ctx_halo_pull waits inside ONE kernel until every owner has published the same
 * epoch and copies the ghost rows straight out of the owners' memory (no staging buffer, no host round trip).
 * Every rank must call signal / pull in the same sequence.  The next overwrite of an exported array must be
 * ordered after a collective that all ranks enter after their pulls (the scalar all-reduce of an evaluation is). */
#define MS_IPC_FLAGS        100   /* pseudo array id: the flag words */
#define MS_IPC_HANDLE_BYTES 64
#define MS_FLAG_POSITIONS   0     /* guards MS_ARR_POSITIONS and MS_ARR_TRIAL */
#define MS_FLAG_SEEDS       1     /* guards MS_ARR_SEEDS */
/* close every peer array this context has opened (before ANY rank frees its arrays: every rank calls this, the ranks
 * meet at a barrier, then the contexts may be destroyed) */
MS_API int ms_ctx_peer_close(ms_ctx* ctx);
/* guards MS_ARR_SEEDS */
MS_API int ms_ctx_ipc_export(ms_ctx* ctx, int32_t which, uint8_t* handle64);
MS_API int ms_ctx_peer_open(ms_ctx* ctx, int32_t slot, int32_t which, const uint8_t* handle64);
/* peers living in THIS process (several contexts driven by one host thread or several threads): register the
 * owner's device pointers directly (ms_ctx_device_ptr / ms_ctx_flag_words_ptr) instead of IPC handles */
MS_API int ms_ctx_peer_set_pointer(ms_ctx* ctx, int32_t slot, int32_t which, void* device_ptr);
MS_API void* ms_ctx_flag_words_ptr(ms_ctx* ctx);
/* owner slot and owner-local row of every ghost row [n_owned, nv), in ghost order */
MS_API int ms_ctx_set_ghost_sources(ms_ctx* ctx, int32_t n_slots, const int32_t* owner_slot, const int32_t* owner_row);
/* upload the pointer tables now (allocations and NULL-stream copies serialise streams of one process: keep them
 * out of the exchange sequence when several contexts of one process wait for each other) */
MS_API int ms_ctx_halo_prepare(ms_ctx* ctx);
MS_API int ms_ctx_halo_signal(ms_ctx* ctx, int32_t flag_index);
MS_API int ms_ctx_halo_pull(ms_ctx* ctx, int32_t which, int32_t flag_index);
/* this rank's slot among n_slots ranks (its own flag block takes part in the all-reduce) */
MS_API int ms_ctx_set_rank_slot(ms_ctx* ctx, int32_t slot, int32_t n_slots);
/* sum of MS_ARR_SCALARS[0..count) over all ranks through peer memory, in rank order (bitwise the same on every
 * rank); needs the flag words of EVERY rank opened.  Replaces the NCCL all-reduce of an evaluation and, like it,
 * is entered by every rank after its pulls. */
MS_API int ms_ctx_allreduce_scalars(ms_ctx* ctx, int32_t count);
/* 0 while every pull found its flags in time; 1 after a pull gave up waiting (~10 s) */
MS_API int ms_ctx_halo_error(ms_ctx* ctx, int32_t* error);
/* One evaluation of this rank's partition with the transport folded into the compute launches: signal + pull of the
 * (trial) positions in one kernel when exchange_positions != 0, pass A whose last CTA raises the seed flag, the seed
 * pull, pass B whose last CTA reduces the per-CTA sums and publishes the local scalars, and one kernel that gathers
 * the scalars of all ranks in rank order and writes the KKT coefficient: 5 launches for the sequence
 * halo_signal / halo_pull / eval_pass_a / halo_signal / halo_pull / eval_pass_b / eval_reduce / allreduce_scalars /
 * eval_project (10 launches); results agree to rounding (the local sums are added by the last CTA in 32 row
 * groups instead of the reduce kernel's 64) and are run-to-run repeatable.  Replaces the per-evaluation halo exchange + scalar
 * all-reduce of the partitioned sweep (BASELINE.json north_star; no counterpart in the single-process reference).
 * The kernels wait for flags of peers, so the ranks must run concurrently: one process per GPU. */
/* exchange_positions: bit 0 = exchange the (trial) positions for this evaluation; bit 1 = carry the exchanges out INSIDE
 * the patch kernels (interior patches first; the epilogue warps pull the ghost rows meanwhile; the producer warps wait
 * before their first patch that reads ghost rows; the last CTA of the last pass publishes AND gathers the scalars):
 * 2 launches, the exchanges hide behind the interior patches.  Needs
 * rounds of at least 64 lanes (the default packing). */
MS_API int ms_ctx_eval_partition(ms_ctx* ctx, const ms_eval_opts* opts, int32_t exchange_positions);
/* PUSH form of the same transport (optional; ms_ctx_eval_partition uses it once the targets are set; measured no faster
 * than the pull form on 2 x B200, PartitionedMesh enables it with MS_HALO_PUSH=1): for each of the n rows of
 * this rank that another rank lists as a ghost -- that rank's slot, the row here (owned), the row in that rank's
 * arrays.  The owner then STORES its rows into the peers' ghost slots (posted NVLink writes) and raises its arrival
 * word in their flag blocks; receivers poll local memory only (inside the patch kernel, before its first patch), and
 * the 12 evaluation scalars travel the same way from the last CTA of the last pass.  Needs every peer array and flag
 * block opened (ms_ctx_peer_open) and ms_ctx_set_rank_slot; at most 16 ranks. */
MS_API int ms_ctx_set_push_targets(ms_ctx* ctx, int32_t n, const int32_t* dst_slot, const int32_t* src_row,
                                   const int32_t* dst_row);
/* one push of MS_ARR_POSITIONS / MS_ARR_TRIAL (flag_index MS_FLAG_POSITIONS) or MS_ARR_SEEDS (MS_FLAG_SEEDS) */
MS_API int ms_ctx_halo_push(ms_ctx* ctx, int32_t which, int32_t flag_index);

/* One evaluation with everything resident: pass A (+ pass B when want_grad); the last CTA of the last pass adds
 * up the per-CTA sums in fixed order and writes the scalars and the KKT / penalty coefficient (no reduce or
 * project launch).  The constraint projection g + MS_SC_COEF * gC and the fixed-row mask are DEFERRED: they are
 * applied by the consumer of the gradient (ms_ctx_direction_from_gradient, ms_ctx_line_search_stats) or, in
 * place, by the first call that exposes MS_ARR_GRAD (ms_ctx_get_array, ms_ctx_device_ptr, ms_ctx_eval_host, ...),
 * so every caller of the ABI sees the projected gradient of runtime/constraint_manager.py:294-301.
 * Asynchronous on the context stream; results stay on the device. */
MS_API int ms_ctx_eval_async(ms_ctx* ctx, const ms_eval_opts* opts);
/* the same in two calls (timing, overlap): stage 0 = pass A, stage 1 = pass B + finalisation */
MS_API int ms_ctx_eval_stage(ms_ctx* ctx, const ms_eval_opts* opts, int32_t stage);
/* the two halves, for the multi-GPU path (seed halo exchange happens between them) */
MS_API int ms_ctx_eval_pass_a(ms_ctx* ctx, const ms_eval_opts* opts);
MS_API int ms_ctx_eval_pass_b(ms_ctx* ctx, const ms_eval_opts* opts);
MS_API int ms_ctx_eval_finish(ms_ctx* ctx, const ms_eval_opts* opts);
/* ms_ctx_eval_finish = reduce (per-CTA running sums -> 12 scalars on the device) followed by
 * project (KKT / penalty coefficient from the scalars; the projection itself is deferred, see
 * ms_ctx_eval_async).  Multi-GPU: all-reduce MS_ARR_SCALARS[0..11] between. */
MS_API int ms_ctx_eval_reduce(ms_ctx* ctx, const ms_eval_opts* opts);
MS_API int ms_ctx_eval_project(ms_ctx* ctx, const ms_eval_opts* opts);
/* Self-check builds only (libms_b200_checked.so, -DMS_SELF_CHECK): violation counters of the patch kernels'
 * hand-over protocol since the context was created -- [0] an accumulator row taken by two lanes at once, [1] a
 * patch-local index out of range, [2] a row still locked when the epilogue reads it.  Other builds return -10. */
MS_API int ms_ctx_self_check(ms_ctx* ctx, int32_t* counters3);
/* synchronise and copy the 16 scalars to the host */
MS_API int ms_ctx_read_scalars(ms_ctx* ctx, double* scalars16);
/* ms_ctx_eval_async + ms_ctx_read_scalars */
MS_API int ms_ctx_eval(ms_ctx* ctx, const ms_eval_opts* opts, double* scalars16);
/* End-to-end call with HOST buffers (what a plugin module does): H2D positions, evaluate,
 * D2H scalars and, when non-NULL, the gradient / volume gradient / tilt gradient. */
MS_API int ms_ctx_eval_host(ms_ctx* ctx, const ms_eval_opts* opts, const double* pos_host,
                            double* scalars16, double* grad_host, double* volgrad_host,
                            double* tilt_grad_host);
/* trial = positions + alpha * direction (line_search.py:358-382), on the device */
MS_API int ms_ctx_make_trial(ms_ctx* ctx, double alpha);
/* positions <- trial (accept the step) */
MS_API int ms_ctx_accept_trial(ms_ctx* ctx);
/* --- device-resident line search (runtime/steppers/line_search.py:267-541, fast path) ---
 * direction = scale * gradient (gradient descent: scale = -1) */
MS_API int ms_ctx_direction_from_gradient(ms_ctx* ctx, double scale);
/* dst += alpha * src for two (nv,3) arrays, optionally leaving fixed rows untouched: the position update
 * of the hard volume projection x -= lambda dV/dx (modules/constraints/volume.py:116-149) */
MS_API int ms_ctx_axpy(ms_ctx* ctx, int dst, int src, double alpha, int32_t skip_fixed);
/* Evolver-style vertex averaging of MS_ARR_POSITIONS, `rounds` times (the `V[n]` command; runtime/vertex_average.py:28-120,
 * geometry/vertex_average.py::vertex_average_arrays).  Every edge is weighted by the summed area of the facets that list
 * it, areas taken from the positions before each round; a vertex that is not fixed (ms_ctx_set_topology /
 * ms_ctx_set_fixed_mask), has more than one edge and more than one usable edge (weight > 0) and a weight sum
 * sum w^2 >= 1e-15 moves by 1/4 sum w^2 (x_u - x_v) / sum w^2.  group: nv pin groups in the caller's vertex order,
 * -1 = none; a grouped vertex uses only edges to vertices of its own group (NULL: no pin groups).  Asynchronous on the
 * context stream (with a group array the call waits for its upload); no atomics, so repeated calls give identical
 * bits.  MS_ARR_TRIAL is the double buffer of the rounds: its contents are overwritten; every other array is left
 * alone.  Single-context meshes only: a partition context (n_owned < nv), rounds < 0, or a context without topology or
 * positions returns an error; rounds == 0 does nothing. */
MS_API int ms_ctx_vertex_average(ms_ctx* ctx, const int32_t* group, int32_t rounds);
/* Equiangulation (the `u` command; geometry/equiangulate.py::equiangulate_triangles, criterion of
 * runtime/equiangulation.py:151-233): sweeps of Delaunay edge flips over the resident triangle rows, at most
 * max_iterations of them, stopping after the first sweep without a flip.  An interior edge a-b (exactly two facets,
 * opposite directions) flips to c-d when the angles at c and d, measured in the tangent plane, add up to more than
 * pi + 1e-3, not both a and b are fixed, c != d, c-d is not an edge yet and the new facets (a, d, c) and (b, c, d) are
 * not degenerate and turn their normals by less than 120 degrees.  Candidates are taken in ascending edge key
 * min*nv + max of the CALLER's vertex numbering; one is skipped when an earlier flip of the same sweep touched one of
 * its facets or made its new diagonal.  The rows, flip count and sweep count (sweeps that flipped) are those of the
 * host twin, except where an angle sum lies within a few ulp of the threshold (acos is the platform's).  No atomics
 * on floating-point data: repeated calls give identical rows.  Facets keep their rows, so positions, the fixed and
 * boundary masks, kappa / c0, tilts, per-facet surface tension and body membership stay.  After a call that flipped,
 * the rows are packed again and everything derived from the connectivity is dropped as ms_ctx_set_topology drops it:
 * leaflet selections (call ms_ctx_set_leaflet again), vertex normals, the conjugate-gradient history, a pending
 * projection.  If the new rows do not pack (a vertex of more than 48 facets, max_local), the call returns that error
 * and the context keeps its previous rows and packing.  Synchronous.  Single-context meshes only: a partition context
 * (n_owned < nv), max_iterations < 0, a context without topology or positions, or a vertex index outside [0, nv)
 * returns an error.  n_flips / n_sweeps may be NULL. */
MS_API int ms_ctx_equiangulate(ms_ctx* ctx, int32_t max_iterations, int64_t* n_flips, int32_t* n_sweeps);
/* Diagnostics of the last ms_ctx_equiangulate: *n_sweeps_run = sweeps run (including a last one without flips);
 * rounds[i] = selection rounds of sweep i (0 for a sweep without candidates), at most `capacity` entries;
 * ms4 = device time of all sweeps (CUDA events), then host-clock times of the row download, the host packing and the
 * upload of the new packing.  rounds / ms4 may be NULL. */
MS_API int ms_ctx_equiangulate_stats(const ms_ctx* ctx, double* ms4, int32_t* rounds, int32_t capacity,
                                     int32_t* n_sweeps_run);
/* the current (nf,3) triangle rows in the caller's vertex numbering */
MS_API int ms_ctx_get_triangles(const ms_ctx* ctx, int32_t* out);
/* per-vertex Polak-Ribiere direction (runtime/steppers/conjugate_gradient.py:63-119); restart != 0 or no
 * committed history: direction = -gradient.  ms_ctx_cg_commit stores gradient and direction of an
 * accepted step as the history of the next one. */
MS_API int ms_ctx_cg_direction(ms_ctx* ctx, int32_t restart);
MS_API int ms_ctx_cg_commit(ms_ctx* ctx);
/* out4 = { minimum edge length (runtime/topology.py:174-199), largest row norm of the direction,
 *          <gradient, direction>, <gradient, gradient> } */
MS_API int ms_ctx_line_search_stats(ms_ctx* ctx, double* out4);
/* ok = 1 unless a facet normal turns by more than limit_radians between the positions and the trial
 * positions or a facet collapses (runtime/topology.py:13-48).  Only facets with |n0| > 1e-12 at the positions are
 * judged; such a facet fails when |n1| < 1e-12, when cos(angle) < cos(limit_radians), or when a trial coordinate
 * of it is NaN.  limit_radians must lie in [0, pi] (else -1). */
MS_API int ms_ctx_normal_change_ok(ms_ctx* ctx, double limit_radians, int32_t* ok);
/* deterministic <g,g>, <g,gC>, <gC,gC> into the scalar vector */
MS_API int ms_ctx_dots(ms_ctx* ctx);

/* timing on the context stream (CUDA events) and an L2 flush for benchmarks */
MS_API int ms_ctx_timer_start(ms_ctx* ctx);
MS_API int ms_ctx_timer_stop(ms_ctx* ctx, float* milliseconds);
MS_API int ms_ctx_sync(ms_ctx* ctx);
/* a pool of CUDA events recorded on the context stream, for per-kernel timing */
MS_API int ms_ctx_event_record(ms_ctx* ctx, int32_t index);
MS_API int ms_ctx_event_elapsed(ms_ctx* ctx, int32_t from_index, int32_t to_index, float* milliseconds);
/* write `bytes` of scratch device memory (evicts L2 between timed iterations) */
MS_API int ms_ctx_flush_l2(ms_ctx* ctx, int64_t bytes);
MS_API int ms_host_register(void* ptr, int64_t bytes);
MS_API int ms_host_unregister(void* ptr);

/* geometry/tilt_operators.py:414-465 p1_vertex_divergence (ambient_v1): triangle divergences averaged onto the
 * vertices with barycentric area weights; area_v receives the accumulated weights. */
MS_API int ms_p1_vertex_divergence(int32_t nv, int32_t nf, const double* pos, const double* tilts,
                                   const int32_t* tri, double* div_v, double* area_v, int32_t zero_based);

/* ---- stateless shims: one per reference kernel, host pointers in and out ------ */
/* fortran_kernels/surface_energy.f90:27-99 -- grad is accumulated (+=), E returned */
MS_API int ms_surface_energy_and_gradient(int32_t nv, int32_t nf, const double* pos,
                                          const int32_t* tri, const double* gamma, double* grad,
                                          double* energy, int32_t zero_based);
/* fortran_kernels/bending_kernels.f90:32-74 */
MS_API int ms_grad_cotan_batch(int32_t n, const double* u, const double* v, double* grad_u,
                               double* grad_v);
/* fortran_kernels/bending_kernels.f90:87-131 -- out is overwritten */
MS_API int ms_apply_beltrami_laplacian(int32_t dim, int32_t nv, int32_t nf, const double* weights,
                                       const int32_t* tri, const double* field, double* out,
                                       int32_t zero_based);
/* fortran_kernels/tilt_kernels.f90:26-86 */
MS_API int ms_p1_triangle_divergence(int32_t nv, int32_t nf, const double* pos,
                                     const double* tilts, const int32_t* tri, double* div_tri,
                                     double* area, double* g0, double* g1, double* g2,
                                     int32_t zero_based);
/* fortran_kernels/tilt_kernels.f90:88-190 -- va0/va1/va2 may be NULL */
MS_API int ms_compute_curvature_data(int32_t nv, int32_t nf, const double* pos, const int32_t* tri,
                                     double* k_vecs, double* vertex_areas, double* weights,
                                     int32_t zero_based, double* va0, double* va1, double* va2);
/* geometry/body.py:150-252 -- volume of the facets given; grad (may be NULL) += factor*dV/dx */
MS_API int ms_volume_and_gradient(int32_t nv, int32_t nf, const double* pos, const int32_t* tri,
                                  double factor, double* grad, double* volume);

#ifdef __cplusplus
}
#endif
#endif /* MS_B200_H */
