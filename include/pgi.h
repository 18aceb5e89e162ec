/*
 * pgi.h — C-ABI of the B200-native hypothesis-verification engine ("pgi" = pose-graph initialisation).
 *
 * This is the drop-in boundary of SURVEY §8(b).  The reference has no FFI/plugin API; the seam is the
 * pair of C++ call sites its host already has (all citations into
 * /root/reference/src/pyposegraphbuilder/include/):
 *
 *   bool PoseGraphBuilder::estimatePose(...)                    pose_graph_builder.h:153-164, :940-1078
 *        called once per pair from processImages                pose_graph_builder.h:616-627
 *   bool InTraversalPoseTester<EssentialMatrixEvaluator>::test  graph_traversal.h:194-233
 *        called from inside A*                                  graph_traversal.h:790
 *   void PoseGraphBuilder::createCorrespondenceMatrix(...)      pose_graph_builder.h:864-938
 *
 * Every entry point is plain C: caller-owned host buffers, context-owned device memory, integer status
 * codes, no exceptions, no torch types.  One context per (host thread, GPU); calls on a context are
 * serialised by the caller.  Device work is asynchronous between pgi_submit_wave and pgi_wait_wave.
 *
 * There is NO CPU fallback: every compute entry point fails with PGI_ERR_CUDA if no sm_100 device is
 * usable.
 */
#ifndef PGI_H_
#define PGI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pgi_ctx pgi_ctx;
typedef int32_t pgi_status;

enum {
    PGI_OK = 0,
    PGI_ERR_INVALID = -1, /* bad argument (null pointer, out-of-range id, N too large, ...) */
    PGI_ERR_CUDA = -2,    /* CUDA runtime error / no usable device; see pgi_last_error */
    PGI_ERR_NOMEM = -3,   /* host or device allocation failed */
    PGI_ERR_STATE = -4    /* call order violated (e.g. wait without submit) */
};

/* Wave flags (pgi_submit_wave). */
enum {
    PGI_WAVE_PATH = 1u,     /* verify the supplied path hypotheses: test + getInliers + five-point (a3-a7) */
    PGI_WAVE_FALLBACK = 2u, /* run the robust fallback (a8) for pairs whose path branch did not succeed     */
    PGI_WAVE_MASKS = 4u,    /* also produce the per-correspondence inlier masks (PGB:1000-1009, :1034-1044)  */
    PGI_WAVE_NO_TEST = 8u,  /* hypotheses are estimatePose guesses: skip the InTraversalPoseTester gate      */
    PGI_WAVE_EXTRA = 16u    /* pair ids index the pairs of pgi_register_extra_pairs, not the scene's         */
};

typedef struct pgi_config {
    int32_t device;               /* CUDA device ordinal                                              */
    uint32_t min_inliers;         /* minimum_inlier_number, cpp_example.cpp:44 (default 20)            */
    uint32_t test_min_inliers;    /* InTraversalPoseTester minimum, pose_graph_builder.h:809 (5)       */
    uint32_t fallback_max_iters;  /* cv::findEssentialMat USAC default maxIters (1000)                 */
    double threshold_multiplier;  /* 3/2, pose_graph_builder.h:798 and :963                            */
    uint32_t max_wave;            /* capacity hint: pairs per wave (grown on demand)                   */
    uint32_t flags;               /* bit 0: background context (lowest stream priority); other bits 0  */
} pgi_config;

/* Fixed 160-byte verdict record — also the element of the per-wave all-gather (SURVEY §8e). */
typedef struct pgi_verdict {
    uint32_t pair_id;        /* registered pair id                                                        */
    uint8_t branch;          /* 0 = none (rejected), 1 = path hypothesis accepted, 2 = fallback accepted  */
    uint8_t accepted;        /* estimatePose return value (PGB:1077 / :1054 / :1070)                      */
    uint8_t test_passed;     /* InTraversalPoseTester::test verdict of the (last) hypothesis (GT:194-233) */
    uint8_t n_hypotheses;    /* hypotheses supplied for the pair in this wave                             */
    uint32_t test_count;     /* inlierNumber_ out-param of test(): min(#inliers, test_min_inliers)        */
    uint32_t inlier_count;   /* inlierNumber_ of estimatePose (PGB:1022 / :1047)                          */
    uint32_t n_corr;         /* N                                                                         */
    uint32_t path_inliers;   /* |getInliers| of the last hypothesis (GT:136-168), 0 if none               */
    double E[9];             /* E handed to the decomposition, row-major (PGB:1057)                       */
    double q[4];             /* T_dst_src rotation, Eigen order (x,y,z,w) (PGB:1073-1075)                 */
    double t[3];             /* T_dst_src translation                                                     */
    uint32_t iters;          /* fallback iterations executed (0 if the fallback did not run)              */
    uint32_t status;         /* bit0: fallback ran, bit1: five-point produced no model, bit2: NaN pose    */
} pgi_verdict;

/* Per-stage device timings (CUDA events on the context stream) accumulated since the last reset. */
typedef struct pgi_stats {
    double ms_correspondences;  /* K0 build_correspondences (a1)                     */
    double ms_score;            /* K1 score_hypotheses (a2-a6)                        */
    double ms_fivept;           /* K2 fivept_first_solution (a7)                      */
    double ms_fallback_solve;   /* K4 fallback minimal solver                         */
    double ms_fallback_score;   /* K5 fallback scoring / LO / termination             */
    double ms_decompose;        /* K3 decompose_vote + pose (a9-a11)                  */
    double ms_total;            /* submit -> last kernel of the wave                  */
    uint64_t launches;          /* kernels launched                                   */
    uint64_t pairs;             /* pairs processed                                    */
    uint64_t corr_evals;        /* hypothesis x correspondence Sampson evaluations    */
    uint64_t fallback_pairs;    /* pairs that ran the fallback                        */
    uint64_t fallback_models;   /* minimal + LO models scored by the fallback         */
    uint64_t h2d_bytes;         /* bytes copied host->device                          */
    uint64_t d2h_bytes;         /* bytes copied device->host                          */
    double ms_match;            /* K9 batched descriptor matching (all chunks)        */
    uint64_t dist_evals;        /* K9 descriptor distances (each pair's n_src x n_dst once) */
    uint64_t match_pairs;       /* pairs matched by K9                                */
    uint64_t match_rows;        /* matches K9 produced                                */
    double ms_guided;           /* single-pair guided matching (K10: pgi_guided_match, pgi_guided_match_views) */
    uint64_t guided_calls;      /* single-pair calls timed in ms_guided               */
    double ms_guided_pairs;     /* K10 batched guided matching (pgi_guided_match_pairs, all chunks) */
    uint64_t guided_pairs;      /* pairs matched by K10                               */
    uint64_t guided_dist_evals; /* K10 descriptor distances computed                  */
    uint64_t guided_chunks;     /* K10 chunks run (scratch is bounded per chunk)      */
} pgi_stats;

const char *pgi_version(void);
/* Number of usable sm_100 devices (0 if none / no driver). Never fails. */
int32_t pgi_device_count(void);

pgi_status pgi_create(const pgi_config *cfg, pgi_ctx **out);
pgi_status pgi_destroy(pgi_ctx *ctx);
const char *pgi_last_error(pgi_ctx *ctx);

/* Register pairs from already normalised correspondences (the cv::Mat N x 4 CV_64F of
 * createCorrespondenceMatrix, pose_graph_builder.h:553-565).  corr_xy4 has corr_offset[n_pairs] rows
 * [x1 y1 x2 y2]; thr_norm[k] is normalizedThreshold of pair k.  Replaces any previous registration.
 * Pair ids are 0..n_pairs-1. */
pgi_status pgi_register_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint64_t *corr_offset, const double *corr_xy4,
                              const double *thr_norm);

/* Register pairs in the compact layout and build the N x 4 FP64 matrices ON THE DEVICE
 * (createCorrespondenceMatrix, pose_graph_builder.h:864-938: FP32 pixel keypoints, source-camera intrinsics for
 * both images, thr_norm = thr_px / f_src).  focal[V]; size_wh[V][2]; kp_offset[V+1]; kp_xy[sum K][2] float;
 * pair_views[n_pairs][2] (src,dst); m_offset[n_pairs+1]; matches[sum N][2] (srcIdx,dstIdx). */
pgi_status pgi_register_scene(pgi_ctx *ctx, uint64_t n_views, const double *focal, const double *size_wh,
                              const uint64_t *kp_offset, const float *kp_xy, uint64_t n_pairs,
                              const uint32_t *pair_views, const uint64_t *m_offset, const uint32_t *matches,
                              double thr_px);

/* matchFeatures (feature_utils.h:103-210) for every pair on the device (K9), then createCorrespondenceMatrix (K0) from the
 * device-resident matches: pgi_register_scene with descriptors in place of matches.  desc[sum K][dim] float (dim 64 or
 * 128, every value finite), row-aligned with kp_xy; at most 16384 keypoints per view (PGI_ERR_INVALID beyond).  Each
 * pair's matches are the rows pgi_match_features returns for it, in the same order.  m_offset_out[n_pairs + 1] receives
 * the match counts as offsets.  Device scratch is bounded by a chunk of pairs; the match list itself stays on the device. */
pgi_status pgi_register_scene_descriptors(pgi_ctx *ctx, uint64_t n_views, const double *focal, const double *size_wh,
                                          const uint64_t *kp_offset, const float *kp_xy, const float *desc, uint32_t dim,
                                          uint64_t n_pairs, const uint32_t *pair_views, double thr_px,
                                          uint64_t *m_offset_out);
/* Copy the (srcIdx, dstIdx) rows and, if non-null, the ratios of the last pgi_register_scene_descriptors on this context
 * (the correspondences.h5 cache): m_offset_out[n_pairs] rows.  PGI_ERR_STATE if a pgi_register_scene came after it. */
pgi_status pgi_read_scene_matches(pgi_ctx *ctx, uint32_t *matches_out, double *ratios_or_null, uint64_t capacity_rows);

/* Descriptors for a scene registered with pgi_register_scene (which keeps none): desc[sum K][dim] float, row-aligned with
 * that registration's kp_xy, dim 64 or 128, every value finite, at most 16384 keypoints per view (PGI_ERR_INVALID
 * otherwise).  They stay resident for pgi_guided_match_views.  PGI_ERR_STATE before any scene registration. */
pgi_status pgi_set_scene_descriptors(pgi_ctx *ctx, const float *desc, uint32_t dim);

/* Pairs whose matches the caller supplies (the quick matches the Tracklets hand out, pose_graph_builder.h:492-520), built
 * into normalised correspondences on the device by K0 from the keypoints, focal lengths, image sizes and thr_px of the last
 * scene registration.  pair_views[n_pairs][2]; m_offset[n_pairs + 1] (m_offset[0] = 0); matches[m_offset[n_pairs]][2]
 * (srcIdx, dstIdx), each index below its view's keypoint count.  The rows go into a second registration of the context,
 * replaced by the next call; waves address it with PGI_WAVE_EXTRA (pair id = row of this call).  The scene's own
 * registration is neither copied nor changed.  PGI_ERR_STATE before any scene registration. */
pgi_status pgi_register_extra_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint32_t *pair_views, const uint64_t *m_offset,
                                    const uint32_t *matches);
/* pgi_read_pair for the pairs of pgi_register_extra_pairs (testing). */
pgi_status pgi_read_extra_pair(pgi_ctx *ctx, uint32_t pair_id, double *corr_xy4, uint64_t capacity_rows, uint64_t *n_rows,
                               double *thr_norm);

/* Make `ctx` use the pairs registered in `owner` (same device) without copying them: a second context — its
 * own stream, wave buffers and statistics — can then verify waves concurrently with the first (used to overlap
 * the hypothesis-independent fallback with the sequential graph commit).  `owner` must outlive `ctx`'s use and
 * must not re-register while shared. */
pgi_status pgi_share_pairs(pgi_ctx *ctx, pgi_ctx *owner);

/* Copy the device-built normalised correspondences / thresholds of one pair back (testing a1). */
pgi_status pgi_read_pair(pgi_ctx *ctx, uint32_t pair_id, double *corr_xy4, uint64_t capacity_rows, uint64_t *n_rows,
                         double *thr_norm);

/* Submit a wave of n pairs.  hyp_offset[n+1] indexes hyp_q_t (7 doubles per hypothesis: qx qy qz qw tx ty tz,
 * the Sophus::SE3d the A* search composed, graph_traversal.h:341-344).  With several hypotheses the semantics
 * are those of the loop at pose_graph_builder.h:974-1029 (the last one decides).  Asynchronous. */
pgi_status pgi_submit_wave(pgi_ctx *ctx, uint32_t n, const uint32_t *pair_id, const uint32_t *hyp_offset,
                           const double *hyp_q_t, uint32_t flags);

/* Block until the wave is done and copy the n verdicts (wave order) to host memory.  masks_or_null receives
 * the concatenated N_k-byte inlier masks in wave order if PGI_WAVE_MASKS was set. */
pgi_status pgi_wait_wave(pgi_ctx *ctx, pgi_verdict *out, uint8_t *masks_or_null);

/* Same, but leave the verdicts on the device: copies them (device-to-device, stream-ordered, then
 * synchronised) into caller-provided DEVICE memory, e.g. the send buffer of an NCCL all-gather. */
pgi_status pgi_wait_wave_device(pgi_ctx *ctx, void *verdicts_device);

/* Synchronous single-pair wrappers with the reference's argument meaning (wave of 1). */
/* = PoseGraphBuilder::estimatePose, pose_graph_builder.h:940-1078. Returns 1/0 (accepted), <0 on error. */
int32_t pgi_estimate_pose(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, double thr_norm, const double *guesses_q_t,
                          uint32_t n_guesses, double *pose_q_t_out, uint8_t *mask_out, uint64_t *inlier_number_out,
                          pgi_verdict *verdict_or_null);
/* = InTraversalPoseTester::test, graph_traversal.h:194-233.  thr is the tester's threshold (1.5*thr_norm at
 * pose_graph_builder.h:807-811), used as given whatever its value: a row counts when its squared Sampson residual is
 * below thr*thr, so a negative thr tests like -thr and a NaN thr counts no row.  Returns 1/0, <0 on error. */
int32_t pgi_test_pose(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, double thr, uint64_t min_inliers,
                      const double *pose_q_t, uint64_t *inlier_number_out);

/* ---- A* path search on the device (K6) ---------------------------------------------------------------------
 * AStarTraversal<ImageSimilarityHeuristics>::getPath, graph_traversal.h:679-870, with the arguments of
 * pose_graph_builder.h:834-841 (returnMultiple = true, one path tested), batched: one warp per (src, dst) query,
 * std::priority_queue's push_heap / pop_heap order replayed exactly (SURVEY App. A.3), so a query returns the path
 * the reference's search returns.  The host (pgb.h) keeps the pose graph; this is its device mirror:
 * per-vertex edge lists in insertion order (pose_graph.h:219-220), committed entries first, then the entries
 * PREDICTED by the positions of the open speculative wave, tagged with position + 1.  A query with cutoff k sees the
 * committed entries and the predicted ones of positions < k.  The composed pose (recoverPath, graph_traversal.h:
 * 290-348) is left to the caller, who owns the edge poses: the result carries the vertex path. */
typedef struct pgi_adj_entry {
    uint32_t vertex, index; /* edge list of `vertex`, slot `index`                                  */
    uint32_t next;          /* the other endpoint (graph_traversal.h:838-840)                       */
    uint32_t tag;           /* 0: committed, p + 1: predicted by wave position p                    */
    double score;           /* PoseGraphEdge score = inlierNumber / matches.size()  (PGB:645-654)   */
} pgi_adj_entry;

typedef struct pgi_query {
    uint32_t src, dst; /* search from src to dst                                                    */
    uint32_t cutoff;   /* predicted entries with tag <= cutoff are part of the graph                */
    uint32_t budget;   /* > 0: give up (status 4) once more than this many nodes were pushed         */
} pgi_query;

typedef struct pgi_search_result {
    uint32_t touched;  /* nodes popped: touchedNodes_ (graph_traversal.h:750)                       */
    uint32_t pushes;   /* nodes pushed                                                              */
    uint16_t path[8];  /* vertices src .. dst of the tested path (path_len entries)                 */
    uint8_t found;     /* destination popped (graph_traversal.h:766)                                */
    uint8_t path_len;
    uint8_t status;    /* 0 ok; 1 heap slab full, 2 arena full, 3 vertex without edge list, 4 push budget of the query
                          exceeded: the caller repeats the search with its own (host) implementation   */
    uint8_t pad;
    uint32_t kcycles;  /* SM clock cycles the search took on its warp, / 1024 (diagnostics)        */
} pgi_search_result;

typedef struct pgi_search_stats {
    double ms_search;      /* K6 kernel time (CUDA events)                                          */
    uint64_t launches;     /* K6 + apply kernels launched                                           */
    uint64_t queries, pops, pushes, overflows;
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t kcycles_sum;     /* sum over searches of their duration on the device (SM kilocycles)          */
    uint64_t kcycles_longest; /* sum over launches of the longest search: what a launch lasts at least    */
} pgi_search_stats;

/* (Re)create the device graph for n_views vertices (<= 65535).  sim_to_next is the V x V similarity table already
 * clamped to [0,1] and TRANSPOSED: sim_to_next[to * V + next] = clamp(similarity(next, to))  (graph_traversal.h:594). */
pgi_status pgi_graph_init(pgi_ctx *ctx, uint32_t n_views, const double *sim_to_next);
/* Write edge-list entries and set the per-vertex counts (both arrays have n_views entries; total >= committed). */
pgi_status pgi_graph_apply(pgi_ctx *ctx, uint32_t n_entries, const pgi_adj_entry *entries,
                           const uint32_t *committed_count, const uint32_t *total_count);
/* Run n searches.  expanded_bits receives n x ceil(V/32) words: bit v set iff vertex v's edge list was iterated
 * (expanded below the maximum depth, graph_traversal.h:814-822).  Synchronous. max_depth <= 7. */
pgi_status pgi_graph_search(pgi_ctx *ctx, uint32_t n, const pgi_query *queries, uint32_t max_depth, double weight,
                            pgi_search_result *results, uint32_t *expanded_bits);
pgi_status pgi_graph_stats(pgi_ctx *ctx, pgi_search_stats *out, int32_t reset);

/* ---- epipolar-hashing guided matcher (K10) ---------------------------------------------------------------
 * HashingBasedMatcherWithPose<false, 45>::match (matcher.h:199-405), the matcher PoseGraphBuilder::guidedMatching runs
 * on an accepted pair (pose_graph_builder.h:717-783): keypoints of the destination image are hashed by the angle of
 * their epipolar line, every source keypoint searches its bin for the descriptor nearest neighbour among the points
 * within 0.75 px symmetric epipolar distance, count-corrected Lowe ratio.  kp_*: n x 2 float pixels (cv::KeyPoint.pt),
 * desc_*: n x dim float (dim 64 or 128, else PGI_ERR_INVALID); pose_q_t: T_dst_src; K_*: 3x3 row-major intrinsics;
 * size_*: width, height.  Any number of keypoints: the pair runs as a batch of one of pgi_guided_match_pairs without
 * the selection.
 * matches_out (capacity n_src x 2: source index, destination index, in source order) and ratios_out (capacity n_src)
 * receive match()'s output, *n_out their number.  The top-`maximum_points` selection of guidedMatching is host work on
 * that list (pose_graph_builder.h:760-782).  prepared_or_null: 14 doubles (F, epipole, min angle, range, bins). */
pgi_status pgi_guided_match(pgi_ctx *ctx, uint32_t n_src, const float *kp_src, const float *desc_src, uint32_t n_dst,
                            const float *kp_dst, const float *desc_dst, uint32_t dim, const double *pose_q_t,
                            const double *K_src, const double *K_dst, const int32_t *size_src, const int32_t *size_dst,
                            int32_t bin_number, uint32_t *matches_out, double *ratios_out, uint32_t *n_out,
                            double *prepared_or_null);

/* PoseGraphBuilder::guidedMatching (pose_graph_builder.h:717-783) of views src -> dst of the registered scene: K10 on the
 * device-resident keypoints and descriptors (pgi_register_scene_descriptors or pgi_set_scene_descriptors), K = [f 0 w/2;
 * 0 f h/2; 0 0 1] of each view, then the selection of :760-782.  matches_out (capacity max_points x 2) and values_out
 * (capacity max_points) receive the selected rows: the max_points smallest (value, index) entries in ascending order if
 * match() returned more than max_points, else all of them in source order, each with the first match's value.  No
 * allocation after the first calls and no descriptor copy.  PGI_ERR_STATE without a scene or without descriptors. */
pgi_status pgi_guided_match_views(pgi_ctx *ctx, uint32_t src, uint32_t dst, const double *pose_q_t, int32_t bin_number,
                                  uint32_t max_points, uint32_t *matches_out, double *values_out, uint32_t *n_out);

/* guidedMatching (pose_graph_builder.h:717-783) for n_pairs cases of the registered scene in one call (K10, spread over the
 * whole GPU).  pair_views[n][2] (src, dst); poses_q_t[n][7] T_dst_src; bin_number as pgi_guided_match_views.
 * max_points > 0: pair k's rows are exactly what pgi_guided_match_views(src, dst, pose, bin_number, max_points) returns.
 * max_points == 0: match()'s rows and adapted ratios, as pgi_guided_match returns them.
 * offsets_out[n+1]; matches_out[capacity_rows][2] (src idx, dst idx); values_out[capacity_rows]: pair k's rows are
 * offsets_out[k] .. offsets_out[k+1] - 1.  capacity_rows >= sum_k (max_points ? min(n_src(k), max_points) : n_src(k)), else
 * PGI_ERR_INVALID before any work; so is, with max_points > 0, a view of more than 16384 keypoints.  Device scratch is bounded per
 * chunk of pairs (512 MB); only the final rows are copied to the host.  PGI_ERR_STATE without a scene, without descriptors
 * or while a wave is in flight. */
pgi_status pgi_guided_match_pairs(pgi_ctx *ctx, uint64_t n_pairs, const uint32_t *pair_views, const double *poses_q_t,
                                  int32_t bin_number, uint32_t max_points, uint64_t *offsets_out,
                                  uint32_t *matches_out, double *values_out, uint64_t capacity_rows);

/* ---- brute-force descriptor matching (K9 on one pair) -------------------------------------------------------
 * matchFeatures (feature_utils.h:103-210) without its HDF5 cache: BRUTEFORCE_SL2 2-NN in both directions, ratio test
 * best/second < 0.90 on the squared distances, mutual nearest neighbour, survivors sorted by the ratio.
 * desc_*: n x dim float descriptors (dim 128 or 64, at most 16384 per side, every value finite: PGI_ERR_INVALID
 * otherwise).  A row whose distances all overflow has no neighbour and no match.  matches_out (capacity n_src x 2:
 * queryIdx, trainIdx) and ratios_out (capacity n_src) receive the rows the reference appends to `matches_` (:196-204),
 * *n_out their number.  The registered scene is left as it is. */
pgi_status pgi_match_features(pgi_ctx *ctx, uint32_t n_src, const float *desc_src, uint32_t n_dst, const float *desc_dst,
                              uint32_t dim, uint32_t *matches_out, double *ratios_out, uint32_t *n_out);

pgi_status pgi_get_stats(pgi_ctx *ctx, pgi_stats *out);
pgi_status pgi_reset_stats(pgi_ctx *ctx);

/* Unit-level device entry points used by the parity tests (one launch each, host buffers). */
pgi_status pgi_dbg_sampson(pgi_ctx *ctx, const double *corr_xy4, uint64_t n, const double *E, double *out);
pgi_status pgi_dbg_five_point(pgi_ctx *ctx, const double *x1, const double *x2, uint32_t n_problems, int32_t dk_max_iters,
                              double dk_tol_sq, double *E_out /* n_problems x 90 */, int32_t *count_out);
pgi_status pgi_dbg_pose_from_essential(pgi_ctx *ctx, const double *E, const double *corr_xy4, uint64_t n, double *R,
                                       double *t, uint64_t *votes);
pgi_status pgi_dbg_fp64_peak(pgi_ctx *ctx, int32_t fused, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* PGI_H_ */
