/*
 * gapro_b200 — C ABI of the B200-native GaPro pseudo-label generator hot path.
 *
 * The reference (VinAIResearch/GaPro) has no FFI layer: its hot path is two
 * Python functions,
 *     gen_pseudo_label_gaussian_process   gapro/gen_ps_utils.py:293-482
 *     fit_gp_spp                          gapro/gaussian_process_utils.py:382-445
 * whose arithmetic runs inside torch / torch_scatter / gpytorch.  This header
 * declares the stage-level entry points a ctypes (or any C) caller binds to
 * replace that arithmetic; each one cites the reference lines it replaces.
 * The Python mirror of the two reference functions lives in
 * gapro_b200/gen_ps_utils.py and gapro_b200/gaussian_process_utils.py and is
 * the only caller in this repository (see INTEGRATION.md for the binding a
 * GaPro maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; "dev" = CUDA device pointer, "host" = host
 *     pointer.  The caller owns every buffer, including workspaces (query the
 *     size with the matching *_workspace_bytes function).
 *   - a batch is a concatenation of scenes: points of scene s are rows
 *     pt_off[s] .. pt_off[s+1]-1, its boxes box_off[s] .. box_off[s+1]-1 (the
 *     LAST box of every scene is the floor slab), its superpoints
 *     spp_off[s] .. spp_off[s+1]-1 ("global" superpoint ids).  One scene is a
 *     batch of one.
 *   - every entry point enqueues its work on `stream` (a cudaStream_t) and
 *     returns immediately unless documented as synchronising.
 *   - return value 0 = ok, < 0 = error; gapro_last_error() gives the message
 *     (thread-local).  The library never exits the process and keeps no global
 *     mutable state besides that message.
 *   - there is no CPU fallback: without a CUDA device every compute entry point
 *     fails with GAPRO_ERR_CUDA.
 */
#ifndef GAPRO_B200_H
#define GAPRO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GAPRO_OK 0
#define GAPRO_ERR_INVALID (-1)
#define GAPRO_ERR_CUDA (-2)
#define GAPRO_ERR_WORKSPACE (-3)
#define GAPRO_ERR_CAPACITY (-4)

/* event kinds produced by gapro_enumerate_events */
#define GAPRO_EV_NEST_B1 0 /* b1 inside b2: intersection -> b1 (gen_ps_utils.py:411-416) */
#define GAPRO_EV_NEST_B2 1 /* b2 inside b1: intersection -> b2 (gen_ps_utils.py:418-423) */
#define GAPRO_EV_GP 2      /* GP region (gen_ps_utils.py:428-446)                         */

/* per-region status bits written by gapro_gp_fit_batch */
#define GAPRO_GP_NOT_PSD 1 /* non-positive Cholesky pivot (gpytorch would raise NotPSDError) */
#define GAPRO_GP_NAN 2     /* non-finite posterior                                           */
/* bits 8..23: how many Cholesky attempts needed extra diagonal jitter (+1e-8 * 10^k, k < 3) - the retry ladder of
 * gpytorch's psd_safe_cholesky behind gaussian_process_utils.py:417; GAPRO_GP_NOT_PSD is set only when the ladder
 * was exhausted, which is where gpytorch raises NotPSDError */
#define GAPRO_GP_RETRY_SHIFT 8

int gapro_version(void);
const char* gapro_last_error(void);

/* ---------------------------------------------------------------------------
 * U — superpoint id densification.  Replaces
 *     unique_spps, spp = torch.unique(spp, return_inverse=True)   gen_ps_utils.py:312
 * and additionally returns the points grouped by superpoint (stable, i.e. in
 * increasing point index inside every superpoint — the accumulation order of
 * torch_scatter's CPU kernels).
 *   spp_raw   dev  int64[n]    raw ids, any values with (max-min) < 2^40 per scene
 *   pt_off    host int64[n_scenes+1]
 *   spp_gid   dev  int32[n]    out: global dense id of every point (scene-local id
 *                              = spp_gid - spp_off[scene]); ids are ranks of the
 *                              sorted unique raw ids, as torch.unique returns them
 *   perm      dev  int32[n]    out: point indices sorted by (scene, id, index)
 *   seg_off   dev  int32[n+1]  out: CSR offsets into perm per global superpoint
 *                              (entries 0..S_total are valid)
 *   spp_off   host int32[n_scenes+1]  out
 * SYNCHRONISES the stream (the superpoint counts size every later buffer).
 */
size_t gapro_densify_workspace_bytes(int64_t n_points, int32_t n_scenes);
int gapro_densify_spp(const int64_t* spp_raw, const int64_t* pt_off, int32_t n_scenes, int32_t* spp_gid,
                      int32_t* perm, int32_t* seg_off, int32_t* spp_off, void* ws, size_t ws_bytes,
                      void* stream);

/* ---------------------------------------------------------------------------
 * F — floor slab.  Replaces gen_ps_utils.py:317-326: per-scene min/max of the
 * float64 coordinates, box [minx,miny,minz,maxx,maxy,minz+ground_h] and its
 * volume prod(clamp(hi-lo, min=0.001)), written into the LAST box slot of every
 * scene.
 *   xyz        dev double[n,3]
 *   boxes      dev double[n_boxes,6]  in/out (instance + wall boxes pre-filled,
 *                                     float32 values widened: gen_ps_utils.py:329)
 *   boxes_vol  dev double[n_boxes]    in/out
 *   pt_off_dev dev int64[n_scenes+1], box_off_dev dev int32[n_scenes+1]
 *   scratch    dev uint64[n_scenes*6] workspace
 */
int gapro_floor_boxes(const double* xyz, const int64_t* pt_off_dev, const int32_t* box_off_dev,
                      int32_t n_scenes, int64_t n_points, double ground_h, double* boxes, double* boxes_vol,
                      uint64_t* scratch, void* stream);

/* ---------------------------------------------------------------------------
 * A + A' — containment and superpoint occupancy.  Replaces
 *     bb_occupancy = is_within_bb_torch(p, lo-0.005, hi+0.005)    gen_ps_utils.py:349-351 (:79-80)
 *     bb_occupancy_spp = scatter_mean(bb_occupancy.float()) >= t  gen_ps_utils.py:359-362
 *     n_bbs_per_spp = bb_occupancy_spp.sum(1)                     gen_ps_utils.py:363
 * fused: one warp per superpoint walks its points (perm/seg_off), tests every
 * point against the scene's boxes in float64 and counts with warp ballots; the
 * N x B boolean matrix is never materialised.  The threshold test is
 * __fdiv_rn((float)count_in, (float)count) >= thresh (bit-exact float32 mean).
 * Also accumulates what the pair loop (gen_ps_utils.py:388-432) needs:
 *   excl_cnt[b]            #superpoints lying in box b only
 *   inter_cnt[s][b1][b2]   #superpoints lying in both b1 and b2 (b1 < b2, scene-local)
 *   occ_bits  dev uint32[S_total, words]   out: bit b of row g = superpoint g is in scene-local box b
 *   n_bbs     dev int32[S_total]           out
 *   cnt_in    dev int32[S_total, 32*words] out, optional (NULL to skip): raw counts, for tests
 *   excl_cnt  dev int32[n_boxes]           out (zeroed here)
 *   inter_cnt dev int32[n_scenes, 32*words, 32*words]  out (zeroed here)
 *   words = ceil(max boxes per scene / 32)
 */
int gapro_occupancy(const double* xyz, const int32_t* perm, const int32_t* seg_off, const int32_t* spp_off_dev,
                    const int32_t* box_off_dev, const double* boxes, int32_t n_scenes, int32_t s_total,
                    int32_t n_boxes, int32_t words, double margin, float thresh, uint32_t* occ_bits,
                    int32_t* n_bbs, int32_t* cnt_in, int32_t* excl_cnt, int32_t* inter_cnt, void* stream);

/* ---------------------------------------------------------------------------
 * Heuristic labelers (SURVEY.md section 8f, the commented alternative at gen_ps.py:112-114).
 * Replaces the arithmetic of gen_pseudo_label_box2mask (gen_ps_utils.py:242-290), gen_pseudo_label
 * (:485-569) and spp_align_label (:99-129): per-point containment in the INSTANCE boxes (margins
 * evaluated in float32, as there), rule for points in several boxes, majority vote per superpoint.
 *   boxes      dev float[n_boxes,6], boxes_vol dev float[n_boxes]  (instance boxes only; box_off_dev
 *              indexes them per scene)
 *   rule       0 = smallest volume, 1 = nearest box centre, 2 = none (such points vote background)
 *   dist_src   dev int32[n], required for rule 1, NULL otherwise: the point whose coordinates the distance
 *              to the box centres is measured from (gapro_multibox_sources below)
 *   spp_align  1: majority vote per superpoint -> inst_spp[S_total] (box index or -1);
 *              0: per-point result -> inst_pt[n] (box index, -1 background, -2 undecided)
 *   occ_thresh >= 0: only boxes holding >= occ_thresh of the superpoint may win the vote (0.7 in
 *              gen_pseudo_label); < 0: no restriction (gen_pseudo_label_box2mask)
 */
int gapro_heuristic_labels(const double* xyz, const int32_t* perm, const int32_t* seg_off, const int32_t* spp_off_dev,
                           const int32_t* box_off_dev, const float* boxes, const float* boxes_vol,
                           const int32_t* dist_src, int32_t n_scenes, int32_t s_total, int32_t words, int32_t rule,
                           int32_t spp_align, float occ_thresh, int32_t* inst_spp, int32_t* inst_pt, void* stream);

/* Source points of the "dist" rule.  gen_ps_utils.py:516 takes point_inds from nonzero() of the COMPACTED
 * matrix bb_occupancy[num_BBs_per_point > 1] and :526 indexes coords_float with them, so the k-th multi-box
 * point of a scene is measured from the coordinates of point k of that scene.  dist_src[p] = scene base + k
 * for the k-th multi-box point, p for every other point (found by executing the reference, see
 * tests/golden/make_ref_golden.py).
 *   pt_off_dev dev int64[n_scenes+1]; ws >= gapro_multibox_workspace_bytes(n_points)
 */
size_t gapro_multibox_workspace_bytes(int64_t n_points);
int gapro_multibox_sources(const double* xyz, const int64_t* pt_off_dev, const int32_t* box_off_dev,
                           const float* boxes, int32_t n_scenes, int64_t n_points, int32_t* dist_src, void* ws,
                           size_t ws_bytes, void* stream);

/* Final labels of the heuristic labelers for a whole batch (gen_ps_utils.py:283-288 / :559-564), one launch.
 * Reads the scene-local results of gapro_heuristic_labels: box index b >= 0 -> sem = boxes_cls[box_off[scene] + b],
 * inst = b; -1 (background) -> sem = instance_classes, inst = -100; -2 (undecided, rule "none") -> both -100.
 *   box_off_dev dev int32[n_scenes+1]; boxes_cls dev int64[box_off[n_scenes]] (the scenes' instance classes)
 *   spp_align  1: inst_spp dev int32[s_total], spp_off_dev dev int32[n_scenes+1] -> packed_spp dev int32[s_total,4]
 *              (16-byte aligned) receives the records (sem, inst, 1.0f bits, 0) of gapro_broadcast_labels;
 *              inst_pt, pt_off_dev, sem, inst unused
 *              0: inst_pt dev int32[n_points], pt_off_dev dev int64[n_scenes+1] -> sem, inst dev int32[n_points];
 *              inst_spp, spp_off_dev, packed_spp unused
 */
int gapro_heuristic_finalize(const int32_t* inst_spp, const int32_t* inst_pt, const int32_t* spp_off_dev,
                             const int64_t* pt_off_dev, const int32_t* box_off_dev, const int64_t* boxes_cls,
                             int32_t instance_classes, int32_t n_scenes, int32_t s_total, int64_t n_points,
                             int32_t spp_align, void* packed_spp, int32_t* sem, int32_t* inst, void* stream);

/* ---------------------------------------------------------------------------
 * B — superpoint feature pooling.  Replaces
 *     gp_feats_spp = torch_scatter.scatter(gp_feats, spp, dim=0, reduce="mean")   gen_ps_utils.py:357
 * float32 sum in increasing point index (torch_scatter CPU order, hence
 * deterministic and bit-exact against the oracle), divided by float32 count.
 * (coords_float_spp, gen_ps_utils.py:354-356, is dead in the reference and not computed.)
 *   feats dev float[n,D]; out dev float[S_total,D]
 */
int gapro_pool_feats(const float* feats, const int32_t* perm, const int32_t* seg_off, int32_t s_total,
                     int32_t D, float* out, void* stream);

/* ---------------------------------------------------------------------------
 * IoU + P — pair state machine (HOST code, no device work).  Replaces
 * gen_ps_utils.py:385-432 (batch_giou_cross :33-50, is_box1_in_box2 :75-76) for
 * ONE scene: walks (b1, b2) in the reference's order with its gates (IoU > 1e-4,
 * visited, non-empty intersection, nesting with offset 0.1 incl. the `break`,
 * IoU >= 0.6 skip, non-empty exclusive sets) and emits the ordered event list.
 * All gates depend on boxes and occupancy only, never on GP results, so the
 * list is final before any GP runs.
 *   boxes     host double[B,6]; excl_cnt host int32[B]; inter_cnt host int32[stride,stride]
 *   ev_kind/ev_b1/ev_b2 host int32[capacity] out; returns the event count or < 0
 */
int gapro_enumerate_events(const double* boxes, int32_t B, const int32_t* excl_cnt, const int32_t* inter_cnt,
                           int32_t stride, int32_t* ev_kind, int32_t* ev_b1, int32_t* ev_b2, int32_t capacity);
/* the float64 IoU matrix alone (diagonal zeroed), for tests: iou host double[B,B] */
int gapro_box_iou(const double* boxes, int32_t B, double* iou);

/* ---------------------------------------------------------------------------
 * Index lists by warp-ballot compaction.  Replaces the torch.nonzero calls of
 * gen_ps_utils.py:405 (intersection) and :428-429 (exclusive sets).  List l of
 * scene list_scene[l] is, in increasing superpoint id,
 *     b2 <  0 : { g : n_bbs[g]==1 and g in box b1 }
 *     b2 >= 0 : { g : g in box b1 and g in box b2 }
 * written (as global superpoint ids) to out_idx[list_off[l] ...]; the caller
 * sizes list_off from excl_cnt / inter_cnt.
 *   list_scene, list_b1, list_b2, list_off : dev int32[n_lists]
 */
int gapro_compact_lists(const uint32_t* occ_bits, const int32_t* n_bbs, const int32_t* spp_off_dev, int32_t words,
                        const int32_t* list_scene, const int32_t* list_b1, const int32_t* list_b2,
                        const int32_t* list_off, int32_t n_lists, int32_t* out_idx, void* stream);

/* ---------------------------------------------------------------------------
 * C — batched GP regions.  Replaces fit_gp_spp (gaussian_process_utils.py:382-445)
 * and the gpytorch machinery behind GPClassificationModel (:11-25): whitened
 * sparse variational GP classifier, inducing points = training rows (trainable),
 * Adam(lr) on -ELBO for `iters` steps, posterior at the test rows.  All
 * arithmetic is float64 (see DESIGN.md: precision policy).
 * Region r trains on feats_spp[train_idx[train_off[r] .. train_off[r+1])] — the
 * first n_b1[r] rows carry label -1, the rest +1 — and predicts at
 * feats_spp[test_idx[test_off[r] .. test_off[r+1])].
 *   feats_spp  dev float[S_total,D]
 *   train_off/test_off host int32[n_regions+1]; n_b1 host int32[n_regions]
 *   train_idx/test_idx dev int32[...]; init_noise dev float[train_off[n_regions]]
 *                      (standard-normal draws; variational mean starts at 1e-3*noise)
 *   out_prob/out_conf/out_mu/out_var dev float[test_off[n_regions]]; out_label dev uint8[...]
 *   out_mu64/out_var64 dev double[...] optional (NULL to skip)
 *   status     dev int32[n_regions]  out: GAPRO_GP_* bits
 * The workspace may be smaller than gapro_gp_workspace_bytes(); regions are
 * then processed in as many chunks as needed (minimum: the largest region).
 * Asynchronous on `stream`, except that the host tile tables of every workspace chunk are uploaded and the
 * stream is synchronised once per chunk before its kernels are enqueued (one chunk unless ws_bytes is smaller than
 * gapro_gp_workspace_bytes).
 */
size_t gapro_gp_workspace_bytes(int32_t n_regions, const int32_t* train_off, const int32_t* test_off, int32_t D);
size_t gapro_gp_min_workspace_bytes(int32_t n_regions, const int32_t* train_off, const int32_t* test_off,
                                    int32_t D);
/* host-only replay of the workspace layout for `groups` stream groups: reserved table bytes minus the bytes the
 * groups' tables take (>= 0 unless the tables would overrun the workspace); no CUDA call, used by the CPU tests */
int64_t gapro_gp_debug_aux_slack(int32_t n_regions, const int32_t* train_off, const int32_t* test_off, int32_t groups);
int gapro_gp_fit_batch(const float* feats_spp, int32_t D, int32_t n_regions, const int32_t* train_off,
                       const int32_t* n_b1, const int32_t* test_off, const int32_t* train_idx,
                       const int32_t* test_idx, const float* init_noise, int32_t iters, double lr,
                       double jitter_zz, double jitter_xx, float* out_prob, float* out_conf, uint8_t* out_label,
                       float* out_mu, float* out_var, double* out_mu64, double* out_var64, int32_t* status,
                       void* ws, size_t ws_bytes, void* stream);
/* number of kernel launches the last gapro_gp_fit_batch call on this thread enqueued */
int64_t gapro_gp_last_launch_count(void);

/* Opt-in profiling of gapro_gp_fit_batch (thread-local): CUDA events are recorded on the launching
 * stream around every phase; gapro_gp_get_profile SYNCHRONISES on them and returns, per phase slot
 * (names: gapro_gp_phase_names(), comma separated), the elapsed milliseconds, the algorithmic flops
 * (unpadded sizes, FMA = 2; SURVEY.md section 8a-C) and the flops the tile kernels issued. */
int gapro_gp_set_profiling(int enable);
const char* gapro_gp_phase_names(void);
int gapro_gp_get_profile(double* ms, double* flops_alg, double* flops_exe, int32_t cap);

/* FP64 pipe microbenchmark: sustained TFLOP/s of a register-resident DMMA (use_dmma=1) or DFMA
 * (use_dmma=0) loop on the current device - the measured roofline denominator of the GP kernels
 * (MEASURED_PEAKS.json has no FP64 figure).  scratch_dev: dev double[1].  SYNCHRONISES. */
int gapro_fp64_peak(int use_dmma, int iters, double* tflops, double* scratch_dev, void* stream);

/* Random-gather microbenchmark (the roofline of the gather-bound stages A/A' and B): one launch reads
 * idx[0..n_records) coalesced and gathers the 24-byte record table[3*idx[i] .. +3) for each; nothing is
 * written.  The caller times the launch (bench.py: CUDA events, L2 flushed) and reports
 * n_records * 28 bytes / time next to the copy bandwidth.  idx dev int32[n_records], table dev double[>= 3*(max idx+1)]. */
int gapro_gather_peak(const int32_t* idx, const double* table, int64_t n_records, double* sink, void* stream);

/* Debug/test hook: run ONE region for `iters` full steps plus the first
 * `stop_phase` phases of the next step, no prediction, and leave the workspace
 * as is.  layout receives the offsets (in doubles) of the region's buffers in
 * ws: see gapro_gp_debug_layout_names(). */
int gapro_gp_debug_run(const float* feats_spp, int32_t D, int32_t M, int32_t n_b1, int32_t N,
                       const int32_t* train_idx, const int32_t* test_idx, const float* init_noise, int32_t iters,
                       int32_t stop_phase, double lr, double jitter_zz, double jitter_xx, void* ws,
                       size_t ws_bytes, int64_t* layout, int32_t layout_cap, void* stream);
const char* gapro_gp_debug_layout_names(void);

/* ---------------------------------------------------------------------------
 * S0 + M + D + label finalisation — per-superpoint resolution.  Replaces
 * gen_ps_utils.py:365-383 (trivial assignment), the in-loop assignments/merges
 * :412-414, :419-421, :438-446 applied in event order (strict `<` on float32
 * confidences), the smallest-volume fallback :450-464 (first minimal box wins
 * ties) and the per-superpoint labels :467-476 (class of the chosen box, 18 for
 * background, wall/floor boxes -> instance -100).
 * One CTA per scene replays that scene's events sequentially.
 *   ev_off dev int32[n_scenes+1]; ev_kind/ev_b1/ev_b2 dev int32[n_events]
 *   ev_list_off/ev_list_len dev int32[n_events]: the event's intersection list in lists_idx
 *   ev_gp_off   dev int32[n_events]: offset of the event's rows in the GP outputs (-1 for nest)
 *   boxes_cls dev int64[n_boxes]; n_fg dev int32[n_scenes] (#instance boxes per scene)
 *   out per superpoint: sem_spp/inst_spp int32, prob/mu/var float; packed_spp (optional, dev
 *   int32[S_total,4], 16-byte aligned) receives the records (sem, inst, prob bits, 0) that
 *   gapro_broadcast_labels gathers with one 128-bit load per point
 */
int gapro_resolve_spp(const uint32_t* occ_bits, const int32_t* n_bbs, int32_t words, const int32_t* spp_off_dev,
                      const int32_t* box_off_dev, const double* boxes_vol, const int64_t* boxes_cls,
                      const int32_t* n_fg, int32_t instance_classes, int32_t n_scenes, const int32_t* ev_off,
                      const int32_t* ev_kind, const int32_t* ev_b1, const int32_t* ev_b2,
                      const int32_t* ev_list_off, const int32_t* ev_list_len, const int32_t* ev_gp_off,
                      const int32_t* lists_idx, const float* gp_conf, const uint8_t* gp_label, const float* gp_mu,
                      const float* gp_var, int32_t* sem_spp, int32_t* inst_spp, float* prob_spp, float* mu_spp,
                      float* var_spp, void* packed_spp, void* stream);

/* ---------------------------------------------------------------------------
 * E — broadcast to points.  Replaces gen_ps_utils.py:478-480
 * (sem[spp], inst[spp], prob[spp]; mu/var stay per superpoint, :482).
 *   packed_spp: the per-superpoint records written by gapro_resolve_spp; sem/inst dev int32[n],
 *   prob dev float[n]; all point arrays 16-byte aligned
 */
int gapro_broadcast_labels(const int32_t* spp_gid, int64_t n_points, const void* packed_spp, int32_t* sem,
                           int32_t* inst, float* prob, void* stream);

/* ---------------------------------------------------------------------------
 * A + A' in point order (the default path).  Same results as gapro_occupancy - containment
 * gen_ps_utils.py:349-351 (float64 compares on the float64 boxes, margin 0.005), occupancy pooling :359-363
 * (integer counts, one float32 divide, >= thresh), n_bbs :363 - but xyz and the dense ids are streamed in point
 * order instead of being gathered by superpoint: a per-scene 32x32x8 grid of box masks decides most boxes per
 * cell, the exact test runs only for boxes whose boundary crosses the point's cell, counts go to `cnt_table` with
 * integer reductions.
 *   spp_gid dev int32[n_points] (gapro_densify_spp); extent_keys: the scratch gapro_floor_boxes filled
 *   (per scene min xyz, max xyz as order-preserving uint64 keys); cnt_table dev int32[S_total, 32*words]
 *   (points of superpoint s inside box b, kept as an output); the other outputs as gapro_occupancy.
 */
size_t gapro_occupancy_points_workspace_bytes(int32_t n_scenes, int32_t words);
int gapro_occupancy_points(const double* xyz, const int32_t* spp_gid, const int32_t* seg_off, const int64_t* pt_off_dev,
                           const int32_t* spp_off_dev, const int32_t* box_off_dev, const double* boxes,
                           const uint64_t* extent_keys, int32_t n_scenes, int64_t n_points, int32_t s_total,
                           int32_t n_boxes, int32_t words, double margin, float thresh, uint32_t* occ_bits,
                           int32_t* n_bbs, int32_t* cnt_table, int32_t* excl_cnt, int32_t* inter_cnt, void* ws,
                           size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * Float64 products on tcgen05 by int8 digit planes ("Ozaki scheme"; csrc/ozaki.cu).  C[M,N] = op(A) op(B)^T:
 * trans = 0 - the operand is stored [vectors, K] row-major, trans = 1 - [K, vectors] row-major; kscale (optional,
 * dev double[K]) multiplies the A operand along k (A diag(kscale) B^T, the dT product of the GP step).  S digits per
 * operand (2..8; 6 gives ~1e-12 of the row-norm bound), S(S+1)/2 int8 products.  ws 1024-byte aligned.  The last of
 * `reps` runs is timed with CUDA events: ms_slice (scaling + digit planes), ms_gemm (the tcgen05 kernel).
 */
size_t gapro_ozaki_workspace_bytes(int32_t M, int32_t N, int32_t K, int32_t S);
int gapro_ozaki_gemm(const double* A, int32_t lda, int32_t transA, const double* kscale, const double* B, int32_t ldb,
                     int32_t transB, int32_t M, int32_t N, int32_t K, int32_t S, double* C, int32_t ldc, void* ws,
                     size_t ws_bytes, int32_t reps, float* ms_slice, float* ms_gemm, void* stream);

/* ---------------------------------------------------------------------------
 * Ev — pseudo-label quality (`--eval_pslabel`, gen_ps.py:116-124).  Replaces
 * get_miou_scene (eval_ps_labels.py:100-147): for every ground-truth instance id g in [0, n_gt) the best IoU
 * with a pseudo instance of the same class (class of an instance = semantic label of its first point; IoU in
 * float32 with the 1e-4 of cal_iou, :36-43).  One pass over the points fills the (n_gt+1) x (n_ps+1)
 * contingency table with integer atomics; max_iou[g] float, valid[g] = 1 when id g is in use and its class
 * is >= 0 (the rows the reference keeps, :139).  All label arrays dev int32[n_points]; n_gt / n_ps = max id + 1.
 */
size_t gapro_eval_workspace_bytes(int32_t n_gt, int32_t n_ps);
int gapro_eval_miou_scene(const int32_t* gt_sem, const int32_t* gt_inst, const int32_t* ps_sem, const int32_t* ps_inst,
                          int64_t n_points, int32_t n_gt, int32_t n_ps, float* max_iou, int32_t* valid, void* ws,
                          size_t ws_bytes, void* stream);
/* get_scene_sem_conf (eval_ps_labels.py:152-172): conf dev int64[num_classes^2], row = ground truth */
int gapro_eval_sem_conf(const int32_t* gt_sem, const int32_t* ps_sem, int64_t n_points, int32_t num_classes,
                        int64_t* conf, void* stream);

/* ---------------------------------------------------------------------------
 * G - boxes from labelled points on the device.  Replaces getInstanceInfo (gen_ps_utils.py:195-239) for the
 * values gen_ps.py uses (:72-74): instances in increasing ground-truth id with unused ids skipped (:209-210),
 * per instance min / max of the (axis-aligned) xyz in float64, class = semantic label of its first point
 * (minus 2 for scannetv2 unless -100, :236-237), volume = prod(clip(max - min, 0)) (:227).
 *   instance_label / semantic_label dev double[n_points] as loaded from the scene file; n_ids = max id + 1;
 *   boxes dev double[n_ids, 6], volumes / classes dev double[n_ids] - the first *n_used_dev rows are filled.
 *   (`corners_label`, which gen_ps.py never reads, is not produced.)
 */
size_t gapro_instance_info_workspace_bytes(int32_t n_ids);
int gapro_instance_info(const double* xyz, const double* instance_label, const double* semantic_label,
                        int64_t n_points, int32_t n_ids, int32_t scannet, double* boxes, double* volumes,
                        double* classes, int32_t* n_used_dev, void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GAPRO_B200_H */
