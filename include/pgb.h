/*
 * pgb.h — C-ABI of the host side that drives the hypothesis-verification engine (pgi.h): the
 * similarity-ordered pair queue, the growing pose graph, the visibility table, the A* path search and
 * the sequential graph commit of the reference, re-organised as SPECULATIVE WAVES with exact validation
 * so the committed pose graph is identical to the reference's sequential (core_number = 1) result
 * (SURVEY §7 hard part 3, §8b).
 *
 * Reference (citations into /root/reference/src/pyposegraphbuilder/include/):
 *   PoseGraphBuilder::processImages       pose_graph_builder.h:352-715   (loop order, commit :645-654, :692)
 *   PoseGraphBuilder::findPath            pose_graph_builder.h:785-862
 *   AStarTraversal::getPath / recoverPath graph_traversal.h:679-870, :290-348
 *   SimilarityTable (queue)               imagesimilarity_graph.h:51-66, :108-171
 *   PoseGraph / VisibilityTable           pose_graph.h:136-224, visibility_table.h:45-171
 *
 * Protocol per wave (all ranks of a multi-GPU job run it identically — SPMD host, SURVEY §8e):
 *   n  = pgb_next_wave(b, max, items)        speculative A* on the current graph snapshot
 *   ... engine verifies items[i] with need_gpu != 0 (sharded by pair owner, verdicts all-gathered) ...
 *   pgb_commit_wave(b, verdicts, n_verdicts) sequential commit in queue order; the first item whose
 *                                            speculation no longer holds and whose verdict is unknown
 *                                            stops the commit; it and its successors are re-queued.
 */
#ifndef PGB_H_
#define PGB_H_

#include <stdint.h>

#include "pgi.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pgb_builder pgb_builder;

typedef struct pgb_config {
    double similarity_threshold;         /* cpp_example.cpp:40  (0.5)  */
    uint64_t minimum_inlier_number;      /* cpp_example.cpp:44  (20)   */
    uint64_t minimum_point_number;       /* cpp_example.cpp:46  (50)   */
    uint64_t maximum_search_depth;       /* cpp_example.cpp:54  (5)    */
    double traversal_heuristics_weight;  /* cpp_example.cpp:50  (0.8)  */
    int32_t use_path_finding;            /* cpp_example.cpp:36  (true) */
    int32_t host_threads;                /* threads for the speculative A* (core_number analogue) */
    int32_t lazy_fallback;               /* 1: waves carry PATH|FALLBACK; 0: fallback verdicts are prefetched */
    int32_t reserved;                    /* re-search window behind the first stale position (0 = unlimited) */
} pgb_config;

typedef struct pgb_item {
    uint32_t pair_id;   /* index into the registered pair list                              */
    uint32_t src, dst;  /* views                                                            */
    uint8_t has_hyp;    /* A* composed a hypothesis (graph_traversal.h:766-797)             */
    uint8_t need_gpu;   /* 1: engine must verify this item (verdict not cached)             */
    uint8_t visible;    /* visibilityTable.hasLink at speculation time                      */
    uint8_t pad;
    double hyp[7];      /* qx qy qz qw tx ty tz                                             */
} pgb_item;

typedef struct pgb_edge {
    uint32_t src, dst;
    double q[4], t[3];
    double score;         /* inlierNumber / matches.size()  pose_graph_builder.h:645-646    */
    uint32_t inlier_number, n_corr;
    uint8_t branch, pad[7];
} pgb_edge;

typedef struct pgb_log {  /* one record per pair popped from the queue, in processing order */
    uint32_t src, dst;
    int64_t pair_index;
    uint8_t visible, had_path, test_passed, branch, committed, pad[3];
    uint32_t test_count, inlier_number, n_corr, touched_nodes;
    double E[9], q[4], t[3], score;
    double hyp[7];        /* the hypothesis A* composed for the pair (qx qy qz qw tx ty tz), zero if had_path == 0:
                             with pair_index it is the (pair, hypothesis) tuple the engine verified */
} pgb_log;

/* Exchange record of one wave position (multi-rank): filled by the position's owner, zero elsewhere, merged by a
 * byte-wise SUM all-reduce. */
typedef struct pgb_record {
    uint8_t valid, has_hyp, has_path_verdict, final_is_path;
    uint32_t touched;
    pgi_verdict v;   /* the owner's verdict for (pair, hypothesis) if has_path_verdict */
    double hyp[7];   /* the hypothesis the owner's search composed (has_hyp): every rank logs the same tuples */
} pgb_record;

enum { PGB_WAVE_DONE = 0, PGB_WAVE_NEED_GPU = 1, PGB_WAVE_NEED_EXCHANGE = 2 };

typedef struct pgb_counters {
    uint64_t pairs_popped, committed, path_accepted, fallback_accepted, rejected, skipped;
    uint64_t waves, items_speculated, items_requeued, astar_runs, astar_reruns, verdict_cache_hits;
    uint64_t astar_pops, astar_pushes; /* heap traffic of all searches (touched nodes / pushed nodes) */
    double sec_astar, sec_commit, sec_visibility;
    uint64_t gpu_searches;      /* searches answered by the device backend (K6)                          */
    uint64_t gpu_search_redo;   /* device searches repeated on the host (slab overflow)                  */
    uint64_t search_mismatches; /* PGB_SEARCH_CHECK=1: device results that differ from the host search   */
    double sec_search_gpu;      /* wall time inside the device backend                                   */
    double sec_search_host_part;/* wall time of the host pool's share of device rounds (runs beside the device) */
    uint64_t floor_retries;     /* host searches repeated because their cost-floor guess was too high (pgb_host.cpp: aStar) */
    uint64_t stale_spared;      /* search results kept although an expanded vertex gained a changed edge (fine staleness rule) */
} pgb_counters;

/* sim: V x V row-major similarity matrix (the text file of imagesimilarity_graph.h:108-171 already parsed).
 * pair_views/m_offset describe the pairs that have correspondences (pair id = row). */
int32_t pgb_create(const pgb_config *cfg, uint64_t n_views, const double *sim, uint64_t n_pairs,
                   const uint32_t *pair_views, const uint64_t *m_offset, pgb_builder **out);
void pgb_destroy(pgb_builder *b);

/* Number of queued pairs not yet committed/rejected (0 = done). */
uint64_t pgb_remaining(pgb_builder *b);

/* Install prefetched fallback verdicts (one per registered pair, index = pair id). */
int32_t pgb_set_fallback_verdicts(pgb_builder *b, const pgi_verdict *verdicts, uint64_t n_pairs);

/* Same for a subset: verdicts[i] belongs to pair_ids[i] (the prefetch may arrive in chunks, in queue order). */
int32_t pgb_set_fallback_verdicts_some(pgb_builder *b, const uint32_t *pair_ids, const pgi_verdict *verdicts, uint64_t n);

/* The static similarity-ordered queue: number of queued pairs / their registered pair ids in pop order
 * (UINT32_MAX for a queued pair without correspondences). */
uint64_t pgb_queue_size(pgb_builder *b);
void pgb_queue_pairs(pgb_builder *b, uint32_t *pair_ids_out);

/* Pop up to max_items pairs in queue order, run the speculative A* and emit them. Returns the item count. */
uint32_t pgb_next_wave(pgb_builder *b, uint32_t max_items, pgb_item *items);

/* verdicts: one per item with need_gpu != 0, in item order.  Returns the number of items committed
 * (accepted, rejected or skipped); the rest were re-queued. */
uint32_t pgb_commit_wave(pgb_builder *b, const pgi_verdict *verdicts, uint32_t n_verdicts);

/* Multi-rank (SPMD, one process per GPU): rank r searches and verifies only the positions whose pair id is
 * congruent to r modulo world (interleaved ownership keeps every wave balanced); after each round the ranks exchange pgb_record arrays (pgb_export_records -> byte-wise
 * SUM all-reduce -> pgb_import_records) so that every rank applies the same outcomes and commits the same graph.
 * pgb_wave_status tells the driver what the open wave waits for. */
int32_t pgb_set_partition(pgb_builder *b, int32_t rank, int32_t world);
int32_t pgb_wave_status(pgb_builder *b);

/* Native driver of one wave (single rank): pgb_next_wave, then engine rounds (submit / wait / pgb_commit_wave) until
 * the wave is committed — the loop of PoseGraphBuilder::processImages' worker (pose_graph_builder.h:352-715) with the
 * engine behind two function pointers whose signatures are those of pgi_submit_wave / pgi_wait_wave (pgi.h), so the
 * product passes exactly those two and its pgi_ctx.  Host state is guarded by an internal mutex that is released while
 * the engine works; pgb_set_fallback_verdicts_some takes the same mutex and may be called from another thread.
 * Returns PGB_WAVE_DONE, PGB_WAVE_NEED_EXCHANGE (several ranks: the caller exchanges records and calls again), or the
 * engine's negative status.  `stats` (optional) accumulates rounds and seconds. */
typedef int32_t (*pgb_submit_fn)(void *engine, uint32_t n, const uint32_t *pair_id, const uint32_t *hyp_offset,
                                 const double *hyp_q_t, uint32_t flags);
typedef int32_t (*pgb_wait_fn)(void *engine, pgi_verdict *out, uint8_t *masks_or_null);
typedef struct pgb_drive_stats {
    double engine_s, host_s;
    uint32_t rounds, items;
} pgb_drive_stats;
int32_t pgb_run_wave(pgb_builder *b, uint32_t wave_size, pgb_submit_fn submit, pgb_wait_fn wait, void *engine,
                     uint32_t flags, pgb_drive_stats *stats);

/* ---- Epipolar-hashing mode (use_epipolar_hashing, cpp_example.cpp:38): exact sequential loop --------------------------
 * processImages with core_number = 1 and the quick-matching branch (pose_graph_builder.h:492-547, :657-707): for every
 * queue position (src, dst) that is not a duplicate edge, q = Tracklets::getCorrespondences(src, dst, maximum_tracklet_number);
 * if |q| >= minimum_point_number the position is QUICK-matched on q (registered with pgi_register_extra_pairs, verified
 * with PGI_WAVE_EXTRA), otherwise FULL-matched on the scene's matches (`matches`, rows as in pgb_create's m_offset);
 * fewer than minimum_point_number rows skip it.  A* and the commit are those of the wave host; the edge score is
 * inliers / rows of the chosen list.  After an accepted position the tracklets grow: a quick-matched one by the rows of
 * guidedMatching with the committed pose (all inliers), a full-matched one by its matches under the estimatePose inlier
 * mask.  Each position is one engine wave of one pair with PATH | FALLBACK | MASKS (plus EXTRA): the next position's
 * matches depend on this one's tracks, so nothing is speculated.  The engine sits behind function pointers whose
 * signatures are those of pgi_submit_wave, pgi_wait_wave, pgi_register_extra_pairs and pgi_guided_match_views.  Runs
 * the whole queue of a builder on which no wave was run; returns 0 or the engine's negative status (-1: bad argument). */
typedef struct pgb_hashing_config {
    uint64_t maximum_tracklet_number;  /* kMaximumTrackletNumber_, cpp_example.cpp (5000)                   */
    uint64_t maximum_point_number;     /* kMaximumPointNumberForEpipolarHashing_ (100)                      */
    int32_t bin_number;                /* HashingBasedMatcherWithPose<false, 45>: 45                        */
    int32_t pad;
} pgb_hashing_config;
typedef int32_t (*pgb_register_extra_fn)(void *engine, uint64_t n_pairs, const uint32_t *pair_views, const uint64_t *m_offset,
                                         const uint32_t *matches);
typedef int32_t (*pgb_guided_fn)(void *engine, uint32_t src, uint32_t dst, const double *pose_q_t, int32_t bin_number,
                                 uint32_t max_points, uint32_t *matches_out, double *values_out, uint32_t *n_out);
typedef struct pgb_hashing_stats {  /* accumulated by pgb_run_hashing */
    uint64_t positions, quick_matched, full_matched, guided_calls, guided_rows, tracklet_adds;
    double sec_astar, sec_engine, sec_guided, sec_tracklets;
} pgb_hashing_stats;
enum { PGB_MATCH_SKIPPED = 0, PGB_MATCH_QUICK = 1, PGB_MATCH_FULL = 2 };
int32_t pgb_run_hashing(pgb_builder *b, const uint32_t *matches, const pgb_hashing_config *cfg, pgb_submit_fn submit,
                        pgb_wait_fn wait, pgb_register_extra_fn register_extra, pgb_guided_fn guided, void *engine,
                        pgb_hashing_stats *stats);
/* Per log record of pgb_run_hashing: the match source (PGB_MATCH_*) and the rows guidedMatching added to the tracklets.
 * Either output may be null.  Returns the number of records (0 for a builder driven by waves). */
uint64_t pgb_copy_match_sources(pgb_builder *b, uint8_t *source_out, uint32_t *guided_rows_out);

/* Device search backend: with it, the speculative A* searches of a wave round (graph_traversal.h:679-870) run as ONE
 * batched device call instead of on the host thread pool — the two function pointers have the signatures of
 * pgi_graph_apply / pgi_graph_search (pgi.h) and the product passes exactly those and its pgi_ctx, after
 * pgi_graph_init with the table of pgb_copy_sim_table.  The host mirrors its graph to the device (committed edges at
 * every commit, the open wave's predicted edges before a round), composes the poses of the returned vertex paths
 * itself (recoverPath, graph_traversal.h:290-348) and repeats on the host any search the device reports as unfinished.
 * Rounds with fewer than min_batch searches stay on the host pool.  Results are identical either way
 * (tests/test_gpu_astar.py; PGB_SEARCH_CHECK=1 re-checks every device search at run time). */
typedef int32_t (*pgb_graph_apply_fn)(void *engine, uint32_t n_entries, const pgi_adj_entry *entries,
                                      const uint32_t *committed_count, const uint32_t *total_count);
typedef int32_t (*pgb_graph_search_fn)(void *engine, uint32_t n, const pgi_query *queries, uint32_t max_depth,
                                       double weight, pgi_search_result *results, uint32_t *expanded_bits);
int32_t pgb_set_search_backend(pgb_builder *b, pgb_graph_apply_fn apply, pgb_graph_search_fn search, void *engine,
                               uint32_t min_batch);
/* The V x V table the A* heuristic reads: clamp(similarity(next, to), 0, 1) at [to * V + next] (graph_traversal.h:594). */
void pgb_copy_sim_table(pgb_builder *b, double *out);
uint32_t pgb_wave_size(pgb_builder *b);
void pgb_export_records(pgb_builder *b, pgb_record *out);
uint32_t pgb_import_records(pgb_builder *b, const pgb_record *in);

uint64_t pgb_edge_count(pgb_builder *b);
void pgb_copy_edges(pgb_builder *b, pgb_edge *out);
uint64_t pgb_log_count(pgb_builder *b);
void pgb_copy_log(pgb_builder *b, pgb_log *out);
void pgb_get_counters(pgb_builder *b, pgb_counters *out);

/* Stand-alone A* on the builder's current graph (testing). Returns 1 if a hypothesis was composed. */
int32_t pgb_astar(pgb_builder *b, uint32_t src, uint32_t dst, double *hyp_q_t, uint32_t *touched_nodes);

/* ---- Tracklets (point_track.h:541-712): multi-view point tracks built from verified matches ------------------------
 * Replaces reconstruction::Tracklets for the quick-matching branch of processImages (pose_graph_builder.h:492-520 reads
 * them, :663-676 / :697-703 feed them).  Not thread-safe by itself: the reference serialises add() behind a writer lock
 * and the wave host commits in order from one thread.  Keypoint indices are the caller's (cv::DMatch query/train idx). */
typedef struct pgb_tracklets pgb_tracklets;
pgb_tracklets *pgb_tracklets_create(uint64_t view_number);
void pgb_tracklets_destroy(pgb_tracklets *t);
/* Tracklets::add(imageIdxSource, imageIdxDestination, matches, inlierMask)  point_track.h:638-712.  0, or -1 on null input. */
int32_t pgb_tracklets_add(pgb_tracklets *t, uint64_t view_src, uint64_t view_dst, uint64_t n, const uint64_t *point_src,
                          const uint64_t *point_dst, const uint8_t *inlier_mask);
/* Tracklets::getCorrespondences(matches, viewIdSource, viewIdDestination, maximumCorrespondenceNumber)  :575-636.
 * Returns the number of matches written (up to maximum + 1, as the reference), -1 if `capacity` is too small. */
int64_t pgb_tracklets_get_correspondences(pgb_tracklets *t, uint64_t view_src, uint64_t view_dst, uint64_t maximum,
                                          uint64_t *out_src, uint64_t *out_dst, uint64_t capacity);
uint64_t pgb_tracklets_track_count(pgb_tracklets *t);

#ifdef __cplusplus
}
#endif
#endif /* PGB_H_ */
