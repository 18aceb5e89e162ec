"""PoseGraphBuilder — host-side mirror of the reference's one public class
(pose_graph_builder.h:27-71: 17-argument constructor + run()), driving the sm_100a engine (pgi.h) through
the speculative-wave host of pgb.h.

File-system inputs of the reference (image path, workspace HDF5 caches, similarity-matrix text,
list_with_focals.txt) are replaced by an in-memory scene dict (scene.py, SURVEY App. D); every other
constructor argument keeps its name, meaning and default (examples/cpp_example.cpp:32-66).

Multi-GPU (SURVEY §8e): one process per GPU.  Pair p is owned by rank p % world (interleaved); each rank verifies
the wave items it owns and the 160-byte verdict records are all-gathered (torch.distributed: NCCL over
NVLink on device buffers, gloo on CPU tensors in the tests) so that every rank runs the same deterministic
commit.  With world_size == 1 no collective is issued.
"""
import ctypes as C
import threading
import time

import numpy as np

from . import engine as _engine
from .engine import VERDICT_DTYPE, WAVE_FALLBACK, WAVE_PATH

ITEM_DTYPE = np.dtype([("pair_id", np.uint32), ("src", np.uint32), ("dst", np.uint32), ("has_hyp", np.uint8),
                       ("need_gpu", np.uint8), ("visible", np.uint8), ("pad", np.uint8), ("hyp", np.float64, (7,))],
                      align=True)
EDGE_DTYPE = np.dtype([("src", np.uint32), ("dst", np.uint32), ("q", np.float64, (4,)), ("t", np.float64, (3,)),
                       ("score", np.float64), ("inlier_number", np.uint32), ("n_corr", np.uint32), ("branch", np.uint8),
                       ("pad", np.uint8, (7,))], align=True)
LOG_DTYPE = np.dtype([("src", np.uint32), ("dst", np.uint32), ("pairIndex", np.int64), ("visible", np.uint8),
                      ("hadPath", np.uint8), ("testPassed", np.uint8), ("branch", np.uint8), ("committed", np.uint8),
                      ("pad", np.uint8, (3,)), ("testCount", np.uint32), ("inlierNumber", np.uint32), ("nCorr", np.uint32),
                      ("touchedNodes", np.uint32), ("E", np.float64, (9,)), ("q", np.float64, (4,)),
                      ("t", np.float64, (3,)), ("score", np.float64), ("hyp", np.float64, (7,))], align=True)


class PgbConfig(C.Structure):
    _fields_ = [("similarity_threshold", C.c_double), ("minimum_inlier_number", C.c_uint64),
                ("minimum_point_number", C.c_uint64), ("maximum_search_depth", C.c_uint64),
                ("traversal_heuristics_weight", C.c_double), ("use_path_finding", C.c_int32), ("host_threads", C.c_int32),
                ("lazy_fallback", C.c_int32), ("reserved", C.c_int32)]


class PgbCounters(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("pairs_popped", "committed", "path_accepted", "fallback_accepted", "rejected",
                                          "skipped", "waves", "items_speculated", "items_requeued", "astar_runs",
                                          "astar_reruns", "verdict_cache_hits", "astar_pops", "astar_pushes")] + \
               [(k, C.c_double) for k in ("sec_astar", "sec_commit", "sec_visibility")] + \
               [(k, C.c_uint64) for k in ("gpu_searches", "gpu_search_redo", "search_mismatches")] + \
               [("sec_search_gpu", C.c_double), ("sec_search_host_part", C.c_double), ("floor_retries", C.c_uint64), ("stale_spared", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


RECORD_DTYPE = np.dtype([("valid", np.uint8), ("has_hyp", np.uint8), ("has_path_verdict", np.uint8), ("final_is_path", np.uint8),
                         ("touched", np.uint32), ("v", VERDICT_DTYPE), ("hyp", np.float64, (7,))], align=True)
WAVE_DONE, WAVE_NEED_GPU, WAVE_NEED_EXCHANGE = 0, 1, 2

PGB_EXPORTS = ["pgb_create", "pgb_destroy", "pgb_remaining", "pgb_set_fallback_verdicts", "pgb_set_fallback_verdicts_some",
               "pgb_queue_size", "pgb_queue_pairs", "pgb_set_partition", "pgb_wave_status", "pgb_wave_size", "pgb_run_wave",
               "pgb_export_records", "pgb_import_records", "pgb_next_wave", "pgb_set_search_backend", "pgb_copy_sim_table",
               "pgb_commit_wave", "pgb_edge_count", "pgb_copy_edges", "pgb_log_count", "pgb_copy_log", "pgb_get_counters",
               "pgb_astar", "pgb_tracklets_create", "pgb_tracklets_destroy", "pgb_tracklets_add",
               "pgb_tracklets_get_correspondences", "pgb_tracklets_track_count", "pgb_run_hashing", "pgb_copy_match_sources"]


def _host_lib():
    lib = _engine.load_library()
    if not getattr(lib, "_pgb_ready", False):
        for name in PGB_EXPORTS:
            getattr(lib, name)
        lib.pgb_create.restype = C.c_int32
        lib.pgb_remaining.restype = C.c_uint64
        lib.pgb_queue_size.restype = C.c_uint64
        lib.pgb_edge_count.restype = C.c_uint64
        lib.pgb_log_count.restype = C.c_uint64
        lib.pgb_next_wave.restype = C.c_uint32
        lib.pgb_commit_wave.restype = C.c_uint32
        lib.pgb_import_records.restype = C.c_uint32
        lib.pgb_wave_size.restype = C.c_uint32
        lib.pgb_run_wave.restype = C.c_int32
        lib.pgb_wave_status.restype = C.c_int32
        lib.pgb_set_partition.restype = C.c_int32
        lib.pgb_set_search_backend.restype = C.c_int32
        lib.pgb_tracklets_create.restype = C.c_void_p
        lib.pgb_tracklets_add.restype = C.c_int32
        lib.pgb_tracklets_get_correspondences.restype = C.c_int64
        lib.pgb_tracklets_track_count.restype = C.c_uint64
        lib.pgb_run_hashing.restype = C.c_int32
        lib.pgb_copy_match_sources.restype = C.c_uint64
        for name in PGB_EXPORTS[1:]:
            getattr(lib, name).argtypes = None
        lib._pgb_ready = True
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class DriveStats(C.Structure):
    _fields_ = [("engine_s", C.c_double), ("host_s", C.c_double), ("rounds", C.c_uint32), ("items", C.c_uint32)]


class HashingConfig(C.Structure):
    _fields_ = [("maximum_tracklet_number", C.c_uint64), ("maximum_point_number", C.c_uint64), ("bin_number", C.c_int32),
                ("pad", C.c_int32)]


class HashingStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("positions", "quick_matched", "full_matched", "guided_calls", "guided_rows",
                                          "tracklet_adds")] + \
               [(k, C.c_double) for k in ("sec_astar", "sec_engine", "sec_guided", "sec_tracklets")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "pad"}


MATCH_SKIPPED, MATCH_QUICK, MATCH_FULL = 0, 1, 2
SOURCE_DTYPE = np.dtype([("source", np.uint8), ("guided_rows", np.uint32)])


class Tracklets:
    """reconstruction::Tracklets (point_track.h:541-712) behind pgb_tracklets_*: `add(src, dst, matches, inlierMask)` and
    `getCorrespondences(src, dst, maximum)` with the reference's argument meaning (matches = (srcIdx, dstIdx[, value])
    rows; the returned rows carry the value 0.0 the reference leaves in the third tuple member)."""

    def __init__(self, viewNumber_):
        self.lib = _host_lib()
        self.h = C.c_void_p(self.lib.pgb_tracklets_create(C.c_uint64(int(viewNumber_))))
        if not self.h:
            raise MemoryError("pgb_tracklets_create failed")

    def close(self):
        if self.h:
            self.lib.pgb_tracklets_destroy(self.h)
            self.h = None

    __del__ = close

    def add(self, imageIdxSource_, imageIdxDestination_, matches_, inlierMask_):
        m = np.asarray(matches_, dtype=np.float64).reshape(-1, np.shape(matches_)[1] if len(matches_) else 2)
        src = np.ascontiguousarray(m[:, 0], dtype=np.uint64)
        dst = np.ascontiguousarray(m[:, 1], dtype=np.uint64)
        mask = np.ascontiguousarray(inlierMask_, dtype=np.uint8)
        if len(mask) != len(src):
            raise ValueError("inlierMask_ must have one entry per match")
        rc = self.lib.pgb_tracklets_add(self.h, C.c_uint64(int(imageIdxSource_)), C.c_uint64(int(imageIdxDestination_)),
                                        C.c_uint64(len(src)), _ptr(src), _ptr(dst), _ptr(mask))
        if rc != 0:
            raise RuntimeError("pgb_tracklets_add failed")

    def getCorrespondences(self, viewIdSource_, viewIdDestination_, maximumCorrespondenceNumber_):
        cap = int(maximumCorrespondenceNumber_) + 1
        a, b = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint64)
        n = self.lib.pgb_tracklets_get_correspondences(self.h, C.c_uint64(int(viewIdSource_)), C.c_uint64(int(viewIdDestination_)),
                                                       C.c_uint64(int(maximumCorrespondenceNumber_)), _ptr(a), _ptr(b), C.c_uint64(cap))
        if n < 0:
            raise RuntimeError("pgb_tracklets_get_correspondences failed")
        return [(int(a[i]), int(b[i]), 0.0) for i in range(n)]

    def track_count(self):
        return int(self.lib.pgb_tracklets_track_count(self.h))


class HostBuilder:
    """Thin wrapper of the pgb_* C-ABI (queue + graph + A* + commit).  Pure host code: usable without a GPU."""

    def __init__(self, scene, similarity_threshold=0.5, minimum_inlier_number=20, minimum_point_number=50,
                 maximum_search_depth=5, traversal_heuristics_weight=0.8, use_path_finding=True, host_threads=0,
                 lazy_fallback=False, research_window=0):
        self.lib = _host_lib()
        cfg = PgbConfig(similarity_threshold, minimum_inlier_number, minimum_point_number, maximum_search_depth,
                        traversal_heuristics_weight, 1 if use_path_finding else 0, host_threads, 1 if lazy_fallback else 0, research_window)
        sim = np.ascontiguousarray(scene["sim"], dtype=np.float64)
        pv = np.ascontiguousarray(scene["pair_views"], dtype=np.uint32)
        mo = np.ascontiguousarray(scene["m_offset"], dtype=np.uint64)
        h = C.c_void_p()
        st = self.lib.pgb_create(C.byref(cfg), C.c_uint64(len(sim)), _ptr(sim), C.c_uint64(len(pv)), _ptr(pv), _ptr(mo), C.byref(h))
        if st != 0:
            raise RuntimeError(f"pgb_create failed: {st}")
        self.h = h
        self.n_pairs = len(pv)
        self._sim_shape = range(len(sim))
        self._items = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.pgb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def remaining(self):
        return int(self.lib.pgb_remaining(self.h))

    def set_fallback_verdicts(self, verdicts):
        verdicts = np.ascontiguousarray(verdicts, dtype=VERDICT_DTYPE)
        if self.lib.pgb_set_fallback_verdicts(self.h, _ptr(verdicts), C.c_uint64(len(verdicts))) != 0:
            raise RuntimeError("pgb_set_fallback_verdicts failed")

    def set_fallback_verdicts_some(self, pair_ids, verdicts):
        pair_ids = np.ascontiguousarray(pair_ids, dtype=np.uint32)
        verdicts = np.ascontiguousarray(verdicts, dtype=VERDICT_DTYPE)
        if self.lib.pgb_set_fallback_verdicts_some(self.h, _ptr(pair_ids), _ptr(verdicts), C.c_uint64(len(pair_ids))) != 0:
            raise RuntimeError("pgb_set_fallback_verdicts_some failed")

    def queue_pairs(self):
        n = int(self.lib.pgb_queue_size(self.h))
        out = np.zeros(n, dtype=np.uint32)
        if n:
            self.lib.pgb_queue_pairs(self.h, _ptr(out))
        return out

    def next_wave(self, max_items):
        items = np.zeros(max_items, dtype=ITEM_DTYPE)
        n = self.lib.pgb_next_wave(self.h, C.c_uint32(max_items), _ptr(items))
        return items[:n]

    def run_wave(self, wave_size, submit_fn, wait_fn, engine_handle, flags, stats=None):
        """pgb_run_wave: the native driver of one wave.  submit_fn / wait_fn are C function pointers with the signatures
        of pgi_submit_wave / pgi_wait_wave (the product passes exactly those two and the engine's pgi_ctx)."""
        st = stats if stats is not None else DriveStats()
        rc = int(self.lib.pgb_run_wave(self.h, C.c_uint32(wave_size), submit_fn, wait_fn, engine_handle, C.c_uint32(flags),
                                       C.byref(st)))
        return rc

    def run_hashing(self, matches, submit_fn, wait_fn, register_extra_fn, guided_fn, engine_handle, maximum_tracklet_number=5000,
                    maximum_point_number=100, bin_number=45, stats=None):
        """pgb_run_hashing: the whole queue in the exact sequential epipolar-hashing mode.  matches: the scene's match list
        (rows as m_offset says).  The four function pointers have the signatures of pgi_submit_wave, pgi_wait_wave,
        pgi_register_extra_pairs and pgi_guided_match_views.  Returns (status, HashingStats)."""
        m = np.ascontiguousarray(matches, dtype=np.uint32).reshape(-1, 2)
        cfg = HashingConfig(int(maximum_tracklet_number), int(maximum_point_number), int(bin_number), 0)
        st = stats if stats is not None else HashingStats()
        rc = int(self.lib.pgb_run_hashing(self.h, _ptr(m), C.byref(cfg), submit_fn, wait_fn, register_extra_fn, guided_fn,
                                          engine_handle, C.byref(st)))
        return rc, st

    def match_sources(self):
        """Per log record of run_hashing: (source: MATCH_SKIPPED / MATCH_QUICK / MATCH_FULL, guided_rows)."""
        n = int(self.lib.pgb_copy_match_sources(self.h, None, None))
        src, rows = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint32)
        if n:
            self.lib.pgb_copy_match_sources(self.h, _ptr(src), _ptr(rows))
        out = np.zeros(n, dtype=SOURCE_DTYPE)
        out["source"], out["guided_rows"] = src, rows
        return out

    def commit_wave(self, verdicts):
        verdicts = np.ascontiguousarray(verdicts, dtype=VERDICT_DTYPE)
        return int(self.lib.pgb_commit_wave(self.h, _ptr(verdicts), C.c_uint32(len(verdicts))))

    def set_partition(self, rank, world):
        if self.lib.pgb_set_partition(self.h, C.c_int32(rank), C.c_int32(world)) != 0:
            raise RuntimeError("pgb_set_partition failed")

    def wave_status(self):
        return int(self.lib.pgb_wave_status(self.h))

    def export_records(self):
        out = np.zeros(int(self.lib.pgb_wave_size(self.h)), dtype=RECORD_DTYPE)
        if len(out):
            self.lib.pgb_export_records(self.h, _ptr(out))
        return out

    def import_records(self, records):
        records = np.ascontiguousarray(records, dtype=RECORD_DTYPE)
        return int(self.lib.pgb_import_records(self.h, _ptr(records)))

    def edges(self):
        n = int(self.lib.pgb_edge_count(self.h))
        out = np.zeros(n, dtype=EDGE_DTYPE)
        if n:
            self.lib.pgb_copy_edges(self.h, _ptr(out))
        return out

    def log(self):
        n = int(self.lib.pgb_log_count(self.h))
        out = np.zeros(n, dtype=LOG_DTYPE)
        if n:
            self.lib.pgb_copy_log(self.h, _ptr(out))
        return out

    def counters(self):
        c = PgbCounters()
        self.lib.pgb_get_counters(self.h, C.byref(c))
        return c.as_dict()

    def sim_table(self):
        """The V x V table the A* heuristic reads (transposed, clamped) — what pgi_graph_init takes."""
        V = len(self._sim_shape)
        out = np.zeros((V, V), dtype=np.float64)
        self.lib.pgb_copy_sim_table(self.h, _ptr(out))
        return out

    def set_search_backend(self, engine, min_batch=8):
        """Run the speculative A* searches on the engine's device (K6): pgi_graph_init + pgb_set_search_backend with
        the engine's own pgi_graph_apply / pgi_graph_search entry points.  engine=None restores the host pool."""
        lib = _engine.load_library()
        if engine is None:
            if self.lib.pgb_set_search_backend(self.h, None, None, None, C.c_uint32(0)) != 0:
                raise RuntimeError("pgb_set_search_backend failed")
            return
        engine.graph_init(self.sim_table())
        apply_fn = C.cast(lib.pgi_graph_apply, C.c_void_p)
        search_fn = C.cast(lib.pgi_graph_search, C.c_void_p)
        if self.lib.pgb_set_search_backend(self.h, apply_fn, search_fn, engine.h, C.c_uint32(min_batch)) != 0:
            raise RuntimeError("pgb_set_search_backend failed")

    def astar(self, src, dst):
        hyp = np.zeros(7)
        touched = C.c_uint32(0)
        r = self.lib.pgb_astar(self.h, C.c_uint32(src), C.c_uint32(dst), _ptr(hyp), C.byref(touched))
        return bool(r > 0), hyp, int(touched.value)


# ---- pair ownership / verdict exchange (SURVEY §8e) ------------------------------------------------------
def owner_of(pair_ids, world_size):
    """Interleaved ownership: pair p belongs to rank p % world (consecutive queue positions share views, so
    contiguous ranges would leave most ranks idle within a wave)."""
    return np.asarray(pair_ids, dtype=np.int64) % world_size


def local_id(pair_ids, world_size):
    return (np.asarray(pair_ids, dtype=np.int64) // world_size).astype(np.uint32)


def shard_scene(scene, rank, world_size):
    """The sub-scene holding the pairs rank `rank` owns (pairs rank, rank + world, ...; keypoints of all views kept).
    Local pair id = global id // world."""
    sub = dict(scene)
    mo = np.asarray(scene["m_offset"], dtype=np.int64)
    ids = np.arange(rank, len(scene["pair_views"]), world_size)
    sub["pair_views"] = np.ascontiguousarray(scene["pair_views"][ids])
    n = mo[ids + 1] - mo[ids]
    sub["m_offset"] = np.concatenate([[0], np.cumsum(n)]).astype(np.uint64)
    if len(ids) and np.all(n == n[0]) and np.all(np.diff(mo) == n[0]):  # equal-sized pairs: strided view, one copy
        sub["matches"] = np.ascontiguousarray(np.asarray(scene["matches"]).reshape(len(mo) - 1, int(n[0]), 2)[rank::world_size]).reshape(-1, 2)
    else:
        rows = np.concatenate([np.arange(mo[i], mo[i + 1]) for i in ids]) if len(ids) else np.zeros(0, dtype=np.int64)
        sub["matches"] = np.ascontiguousarray(np.asarray(scene["matches"])[rows])
    return sub


def needs_matching(scene):
    """A scene with keypoint descriptors and no matches yet: PoseGraphBuilder matches it on the device in prepare()."""
    return "desc" in scene and "matches" not in scene


def allgather_verdicts(local, counts, group=None, device=None):
    """All-gather variable-length verdict arrays (counts[r] records from rank r, known to every rank).
    Returns the list of per-rank arrays.  One collective; payload is padded to max(counts)."""
    import torch
    import torch.distributed as dist

    world = len(counts)
    mx = int(max(counts)) if world else 0
    if world == 1 or mx == 0:
        return [np.asarray(local, dtype=VERDICT_DTYPE)] + [np.zeros(0, dtype=VERDICT_DTYPE)] * (world - 1)
    send = np.zeros(mx, dtype=VERDICT_DTYPE)
    send[:len(local)] = local
    t = torch.from_numpy(send.view(np.uint8).reshape(-1))
    if device is not None:
        t = t.to(device, non_blocking=True)
    out = torch.empty(world * t.numel(), dtype=torch.uint8, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group)
    arr = out.cpu().numpy().view(VERDICT_DTYPE).reshape(world, mx)
    return [arr[r, :int(counts[r])] for r in range(world)]


def allreduce_records(records, group=None, device=None):
    """Merge the ranks' record buffers (each rank fills only the positions it owns): byte-wise SUM all-reduce."""
    import torch
    import torch.distributed as dist

    t = torch.from_numpy(records.view(np.uint8).reshape(-1).copy())
    if device is not None:
        t = t.to(device, non_blocking=True)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy().view(RECORD_DTYPE)


class RecordExchanger:
    """allreduce_records on a GPU with persistent pinned staging buffers and a persistent device buffer: the exchange
    is a ~100 KB latency-bound message once per wave round, so the allocations and pageable copies are what it costs."""

    def __init__(self, max_records, device, group=None):
        import torch
        self.torch, self.group = torch, group
        n = int(max_records) * RECORD_DTYPE.itemsize
        self.pin_in = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        self.pin_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        self.dev = torch.empty(n, dtype=torch.uint8, device=device)
        self.np_in, self.np_out = self.pin_in.numpy(), self.pin_out.numpy()

    def __call__(self, records):
        import torch.distributed as dist
        n = records.nbytes
        if n > self.dev.numel():
            raise ValueError("record buffer larger than the exchanger's capacity")
        self.np_in[:n] = records.view(np.uint8).reshape(-1)
        d = self.dev[:n]
        d.copy_(self.pin_in[:n], non_blocking=True)
        dist.all_reduce(d, op=dist.ReduceOp.SUM, group=self.group)
        self.pin_out[:n].copy_(d, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()
        return self.np_out[:n].copy().view(RECORD_DTYPE)


def default_wave_size(n_views, world_size=1, gpu_search=False):
    """Queue positions per speculative wave.  Host-pool searches: 256 on one GPU (fewest searches; the step is bound by
    the GPU's fallback work there, not by the rounds), 1024 with several ranks: every round of a wave costs an engine
    round trip and a record exchange that do not shrink with the rank count, and since the fine staleness rule
    (pgb_host.cpp) a 4x longer wave needs 63 % fewer rounds for 43 % more searches.  Device searches (K6) need large
    rounds to fill the GPU: 2048."""
    if not gpu_search:
        return 256 if world_size == 1 else 1024
    return 1024 if n_views < 600 else 2048


class PoseGraph:
    """Result container: committed edges in commit order (pose_graph.h:62-106)."""

    def __init__(self, n_views, edges):
        self.n_views = n_views
        self.edges = edges

    def numVertices(self):
        return self.n_views

    def numEdges(self):
        return len(self.edges)

    def hasEdge(self, s, d):
        return bool(np.any((self.edges["src"] == s) & (self.edges["dst"] == d)))


class PoseGraphBuilder:
    """Drop-in for reconstruction::PoseGraphBuilder (pose_graph_builder.h:27-71).  Argument names, order and
    defaults follow examples/cpp_example.cpp:86-103; the four path arguments are accepted and ignored (the
    data comes from `scene`), `kCoreNumber_` sizes the host thread pool of the speculative A*, and
    `kUseGPU_` must be true (there is no CPU path).  kUseEpipolarHashing_=True runs the reference's quick matching from
    point tracks and guided matching after accepted quick-matched pairs, exactly as the reference with core_number = 1
    (pgb_run_hashing); it needs a scene with descriptors (`desc`) and one GPU, and does not use the device A* (K6)."""

    def __init__(self, kCoreNumber_=20, kMaximumTrackletNumber_=5000, kMaximumSearchDepth_=5, kMaximumPathNumber_=100,
                 kMinimumInlierNumber_=20, kMinimumPointNumber_=50, kMaximumPointNumberForEpipolarHashing_=100,
                 kTraversalHeuristicsWeight_=0.8, kSimilarityThreshold_=0.5, kInlierOutlierThreshold_=0.4,
                 kImagePath_="", kWorkspacePath_="", kSimilarityGraphPath_="", kFocalLengthPath_="",
                 kUsePathFinding_=True, kUseGPU_=True, kUseEpipolarHashing_=False, *, scene=None, device=0,
                 wave_size=None, prefetch_fallback=True, fallback_wave=1024, overlap_fallback=True, research_window=0,
                 prefetch_streams=2, native_loop=True, gpu_search=False, gpu_search_min_batch=64,
                 group=None, rank=0, world_size=1):
        if not kUseGPU_:
            raise ValueError("the B200 path has no CPU implementation (kUseGPU_ must be true)")
        if scene is None:
            raise ValueError("scene=... is required (the reference's HDF5/1DSfM inputs are replaced by scene.py)")
        self.hashing = bool(kUseEpipolarHashing_)
        if self.hashing:
            # each position's matches come from the tracks the positions before it left: the mode is sequential
            if "desc" not in scene:
                raise ValueError("kUseEpipolarHashing_ needs a scene with descriptors (desc): guided matching reads them")
            if world_size > 1:
                raise ValueError("kUseEpipolarHashing_ runs on one GPU (world_size must be 1)")
            if gpu_search:
                raise ValueError("kUseEpipolarHashing_ searches on the host: gpu_search must be False")
            prefetch_fallback = overlap_fallback = False
        if world_size > 1 and not prefetch_fallback:
            # the exchange records carry path verdicts only: a non-owner rank could never learn a remote pair's
            # fallback verdict and the ranks' wave loops would diverge
            raise ValueError("world_size > 1 requires prefetch_fallback=True")
        self.scene = scene
        self.cfg = dict(similarity_threshold=kSimilarityThreshold_, minimum_inlier_number=kMinimumInlierNumber_,
                        minimum_point_number=kMinimumPointNumber_, maximum_search_depth=kMaximumSearchDepth_,
                        traversal_heuristics_weight=kTraversalHeuristicsWeight_, use_path_finding=kUsePathFinding_,
                        host_threads=kCoreNumber_, research_window=research_window)
        self.thr_px = kInlierOutlierThreshold_
        self.max_tracklets = kMaximumTrackletNumber_
        self.max_points_hashing = kMaximumPointNumberForEpipolarHashing_
        self.min_inliers = kMinimumInlierNumber_
        self.device = device
        # gpu_search=True: the speculative A* searches of a wave round run as one batched device call (K6) beside the host
        # thread pool.  Exact, but measured no faster than the pool alone on the benchmark scenes (DESIGN.md section 4): a
        # round lasts as long as its longest search and a search is a chain of dependent heap operations, so it is off by
        # default.
        self.gpu_search = bool(gpu_search)
        # measured on cfg2 (scripts/gpu_sweep.sh): 256 positions per wave is the optimum on one GPU (fewer A* re-searches
        # per position, rounds are cheap); with several ranks every round also costs a record exchange
        self.wave_size = wave_size if wave_size else default_wave_size(len(scene["focal"]), world_size, self.gpu_search)
        self.prefetch_fallback = prefetch_fallback
        self.fallback_wave = fallback_wave
        self.group, self.rank, self.world = group, rank, world_size
        # overlap the hypothesis-independent fallback (second context, own low-priority stream, driven by a worker
        # thread) with the sequential waves; with several ranks the worker exchanges each chunk's verdicts over its own
        # gloo group so that it never shares a communicator (or NCCL's ordering requirements) with the wave loop
        self.overlap = bool(overlap_fallback and prefetch_fallback)
        self.pf_group = None
        self.engine = None
        self.engine_fb = None
        self.engine_fb2 = None
        self._exchanger = None
        # one rank: the wave loop itself runs in C++ (pgb_run_wave calling pgi_submit_wave / pgi_wait_wave directly);
        # several ranks: the Python loop below, because the record exchange goes through torch.distributed
        self.native_loop = bool(native_loop)
        self.gpu_search_min_batch = int(gpu_search_min_batch)
        self.prefetch_streams = int(prefetch_streams)
        self.timing = {}
        self.graph = None
        self._desc_resident = False

    # -- engine + registration (H2D inside, counted by the engine's stats) -----------------------------------
    def prepare(self):
        if self.engine is None:
            self.engine = _engine.Engine(device=self.device, min_inliers=self.min_inliers)
        registered = False
        self._desc_resident = False
        if self.world == 1:
            sub = self.scene
            if needs_matching(sub):  # keypoints + descriptors only: matchFeatures on the device, registered in the same call
                self.engine.register_scene_descriptors(sub, self.thr_px)
                registered = self._desc_resident = True
        else:
            # the rank's shard is cut once (a 32 GB scene's shard is gigabytes: not something to copy on every registration)
            if getattr(self, "_sub", None) is None:
                if needs_matching(self.scene):
                    self._sub = self._match_owned_pairs()
                    registered = True
                else:
                    self._sub = shard_scene(self.scene, self.rank, self.world)
            sub = self._sub
        if not registered:
            self.engine.register_scene(sub, self.thr_px)
            if self.hashing:  # a scene that came with matches: guided matching still needs its descriptors on the device
                self.engine.set_scene_descriptors(sub["desc"])
                self._desc_resident = True
        self.prepared = True
        if self.overlap:
            if self.engine_fb is None:
                self.engine_fb = _engine.Engine(device=self.device, min_inliers=self.min_inliers, background=True)
            self.engine_fb.share_pairs(self.engine)
            if self.prefetch_streams > 1:
                # a second background context: its K4/K5 launches fill the tail waves of the first one's
                if self.engine_fb2 is None:
                    self.engine_fb2 = _engine.Engine(device=self.device, min_inliers=self.min_inliers, background=True)
                self.engine_fb2.share_pairs(self.engine)
            if self.world > 1:
                self._gloo_group()

    def _gloo_group(self):
        if self.pf_group is None:
            # The prefetch worker thread gathers its chunks' verdicts over its OWN communicator, and that communicator
            # is gloo (CPU tensors, as in round 1) on purpose.  A second NCCL communicator driven from the worker thread
            # was tried in round 2 and deadlocked on the 1 000-view scene at N=2 (all-gather #77 of the prefetch group
            # against all-reduce #283 of the wave loop, both ranks in the watchdog after 600 s): two NCCL communicators
            # used concurrently must enqueue their collectives in the same order on every rank, which two free-running
            # threads do not, and on a GPU saturated by the fallback kernels the two collective kernels cannot
            # co-schedule their way out of it.  (On the 300-view scene the same code happened to work.)  The payload is
            # 330 KB per chunk; gloo moves it in about a millisecond.
            import torch.distributed as dist
            self.pf_group = dist.new_group(backend="gloo")
        return self.pf_group

    def _match_owned_pairs(self):
        """world > 1 on a descriptor scene: match only the pairs this rank owns (the shard_scene pairs), registered as the
        rank's shard; the per-pair counts are all-gathered over the gloo group so that every rank's host gets the global
        m_offset (scene["m_offset"]).  The matches themselves stay with their owner."""
        import torch
        import torch.distributed as dist

        P = len(self.scene["pair_views"])
        sub = dict(self.scene)
        sub["pair_views"] = np.ascontiguousarray(self.scene["pair_views"][self.rank::self.world])
        self.engine.register_scene_descriptors(sub, self.thr_px)
        counts = np.diff(sub["m_offset"].astype(np.int64))
        per_rank = [len(range(r, P, self.world)) for r in range(self.world)]
        send = torch.zeros(max(per_rank), dtype=torch.int64)
        send[:len(counts)] = torch.from_numpy(counts)
        parts = [torch.empty_like(send) for _ in range(self.world)]
        dist.all_gather(parts, send, group=self._gloo_group())
        n = np.zeros(P, dtype=np.int64)
        for r in range(self.world):
            n[r::self.world] = parts[r].numpy()[:per_rank[r]]
        self.scene["m_offset"] = np.concatenate([[0], np.cumsum(n)]).astype(np.uint64)
        return sub

    def engine_stats(self):
        st = self.engine.stats()
        for e in (self.engine_fb, self.engine_fb2):
            if e is not None:
                for k, v in e.stats().items():
                    st[k] += v
        return st

    def reset_engine_stats(self):
        self.engine.reset_stats()
        for e in (self.engine_fb, self.engine_fb2):
            if e is not None:
                e.reset_stats()

    def close(self):
        for e in (self.engine_fb2, self.engine_fb, self.engine):
            if e is not None:
                e.close()
        self.engine = self.engine_fb = self.engine_fb2 = None

    def _exchange(self, local, counts):
        if self.world == 1:
            return [local]
        import torch
        dev = torch.device("cuda", self.device) if torch.cuda.is_available() else None
        return allgather_verdicts(local, counts, self.group, dev)

    def _prefetch(self, host):
        """Fallback verdicts are a pure function of the pair: compute them for every owned pair in big waves,
        all-gather once, hand them to the host."""
        P = len(self.scene["pair_views"])
        mine = np.arange(self.rank, P, self.world, dtype=np.int64)
        out = np.zeros(len(mine), dtype=VERDICT_DTYPE)
        for s in range(0, len(mine), self.fallback_wave):
            ids = local_id(mine[s:s + self.fallback_wave], self.world)
            out[s:s + len(ids)] = self.engine.run_wave(ids, None, None, flags=WAVE_FALLBACK)
        out["pair_id"] = mine.astype(np.uint32)
        counts = [len(range(r, P, self.world)) for r in range(self.world)]
        parts = self._exchange(out, counts)
        allv = np.zeros(P, dtype=VERDICT_DTYPE)
        for r in range(self.world):
            allv[r::self.world] = parts[r]
        host.set_fallback_verdicts(allv)
        return allv

    def run(self, reconstruction_=None, poseGraph_=None):
        """PoseGraphBuilder::run (pose_graph_builder.h:173-239) -> PoseGraph."""
        gen = self.run_in_batches(None)
        while True:
            try:
                next(gen)
            except StopIteration as done:
                return done.value

    def run_in_batches(self, batch=None):
        """The same run as a generator: with `batch` set it yields (the number of queue positions committed so far) at the
        first wave boundary after every further `batch` committed positions, so that a caller can bracket slices of ONE
        pass — bench.py's steps; the prefetch pipeline keeps running across the yields.  The PoseGraph is the generator's
        return value (StopIteration.value).  batch=None never yields: that is run()."""
        if self.hashing:
            if batch:
                raise ValueError("kUseEpipolarHashing_ runs the queue in one pass: run_in_batches needs batch=None")
            return self._run_hashing()
        t0 = time.perf_counter()
        if self.engine is None or not getattr(self, "prepared", False):
            self.prepare()
        t_reg = time.perf_counter()
        host = HostBuilder(self.scene, lazy_fallback=not self.prefetch_fallback, **self.cfg)
        self.host = host
        total0 = host.remaining()
        next_mark = int(batch) if batch else None
        if self.gpu_search:
            host.set_search_backend(self.engine, self.gpu_search_min_batch)
        lock = threading.Lock()
        progress = threading.Condition(lock)
        state = {"done_pos": 0, "error": None}
        worker = None
        Q = 0
        if self.prefetch_fallback and self.overlap:
            queue = host.queue_pairs()
            Q = len(queue)

            def prefetch_worker():
                try:
                    chunk = self.fallback_wave * self.world
                    engines = [e for e in (self.engine_fb, self.engine_fb2) if e is not None]
                    pending = []  # submitted chunks, oldest first: one in flight per background engine

                    def finish(job):
                        eng, s, ids, own, mine = job
                        v = eng.wait_wave() if len(mine) else np.zeros(0, dtype=VERDICT_DTYPE)
                        v["pair_id"] = mine.astype(np.uint32)
                        if self.world > 1:  # every rank needs every pair's fallback verdict (predictions + commit)
                            counts = [int(np.count_nonzero(own == r)) for r in range(self.world)]
                            parts = allgather_verdicts(v, counts, self.pf_group)
                            merged = np.zeros(len(ids), dtype=VERDICT_DTYPE)
                            for r in range(self.world):
                                merged[np.nonzero(own == r)[0]] = parts[r]
                            v = merged
                        with progress:
                            host.set_fallback_verdicts_some(ids, v)
                            state["done_pos"] = min(Q, s + chunk)
                            progress.notify_all()

                    for k, s in enumerate(range(0, Q, chunk)):
                        ids = queue[s:s + chunk]
                        ids = ids[ids != np.uint32(0xFFFFFFFF)]
                        own = owner_of(ids, self.world)
                        mine = ids[own == self.rank]
                        eng = engines[k % len(engines)]
                        if len(pending) == len(engines):
                            finish(pending.pop(0))
                        if len(mine):
                            eng.submit_wave(local_id(mine, self.world), None, None, flags=WAVE_FALLBACK)
                        pending.append((eng, s, ids, own, mine))
                    while pending:
                        finish(pending.pop(0))
                except Exception as exc:  # surface engine failures in the main thread
                    with progress:
                        state["error"] = exc
                        state["done_pos"] = Q
                        progress.notify_all()

            worker = threading.Thread(target=prefetch_worker, daemon=True)
            worker.start()
        elif self.prefetch_fallback:
            self._prefetch(host)
        t_pre = time.perf_counter()
        flags = WAVE_PATH if self.prefetch_fallback else (WAVE_PATH | WAVE_FALLBACK)
        if self.world > 1:
            host.set_partition(self.rank, self.world)
        prof = dict(engine_s=0.0, exchange_s=0.0, host_s=0.0, wait_prefetch_s=0.0, engine_rounds=0, exchanges=0)
        dev = None
        if self.world > 1:
            import torch
            dev = torch.device("cuda", self.device) if torch.cuda.is_available() else None
        if self.world == 1 and self.native_loop:
            lib = _engine.load_library()
            submit_fn = C.cast(lib.pgi_submit_wave, C.c_void_p)
            wait_fn = C.cast(lib.pgi_wait_wave, C.c_void_p)
            st = DriveStats()
            while True:
                remaining = host.remaining()
                if remaining == 0:
                    break
                if worker is not None:
                    need = min(Q, (Q - remaining) + self.wave_size)
                    t_w = time.perf_counter()
                    with progress:
                        while state["done_pos"] < need:
                            progress.wait()
                    prof["wait_prefetch_s"] += time.perf_counter() - t_w
                    if state["error"] is not None:
                        raise state["error"]
                rc = host.run_wave(self.wave_size, submit_fn, wait_fn, self.engine.h, flags, st)
                if rc < 0:
                    raise _engine.PgiError(f"status {rc}: {lib.pgi_last_error(self.engine.h).decode()}")
                if rc != WAVE_DONE:
                    raise RuntimeError(f"pgb_run_wave returned {rc}")
                if next_mark is not None:
                    left = host.remaining()
                    if left > 0 and total0 - left >= next_mark:
                        while total0 - left >= next_mark:
                            next_mark += int(batch)
                        yield total0 - left
            prof["engine_s"], prof["host_s"], prof["engine_rounds"] = st.engine_s, st.host_s, int(st.rounds)
        while self.world > 1 or not self.native_loop:
            with progress:
                remaining = host.remaining()
                if remaining == 0:
                    break
                if worker is not None:
                    need = min(Q, (Q - remaining) + self.wave_size)
                    t_w = time.perf_counter()
                    while state["done_pos"] < need:
                        progress.wait()
                    prof["wait_prefetch_s"] += time.perf_counter() - t_w
                    if state["error"] is not None:
                        raise state["error"]
                t_h = time.perf_counter()
                items = host.next_wave(self.wave_size)
                status = host.wave_status()
                prof["host_s"] += time.perf_counter() - t_h
            # drive the open wave to its fixed point: engine rounds for the positions this rank owns, record exchange
            # between ranks after every round (multi-rank only)
            while status != WAVE_DONE:
                t_a = time.perf_counter()
                if status == WAVE_NEED_GPU:
                    sel = np.nonzero(items["need_gpu"])[0]
                    hoff = np.zeros(len(sel) + 1, dtype=np.uint32)
                    hoff[1:] = np.cumsum(items["has_hyp"][sel])
                    hyp = items["hyp"][sel][items["has_hyp"][sel] > 0]
                    verdicts = self.engine.run_wave(local_id(items["pair_id"][sel], self.world), hoff, hyp, flags=flags)
                    verdicts["pair_id"] = items["pair_id"][sel]
                    t_b = time.perf_counter()
                    prof["engine_s"] += t_b - t_a
                    prof["engine_rounds"] += 1
                    with progress:
                        host.commit_wave(verdicts)
                    prof["host_s"] += time.perf_counter() - t_b
                else:  # WAVE_NEED_EXCHANGE
                    if dev is not None:
                        if self._exchanger is None:
                            self._exchanger = RecordExchanger(max(self.wave_size, 4096), dev, self.group)
                        merged = self._exchanger(host.export_records())
                    else:
                        merged = allreduce_records(host.export_records(), self.group, dev)
                    t_b = time.perf_counter()
                    prof["exchange_s"] += t_b - t_a
                    prof["exchanges"] += 1
                    with progress:
                        host.import_records(merged)
                    prof["host_s"] += time.perf_counter() - t_b
                with progress:
                    status = host.wave_status()
                    if status != WAVE_DONE:
                        items = host.next_wave(self.wave_size)
            if next_mark is not None:
                with progress:
                    left = host.remaining()
                if left > 0 and total0 - left >= next_mark:
                    while total0 - left >= next_mark:
                        next_mark += int(batch)
                    yield total0 - left
        if worker is not None:
            worker.join()
        t_end = time.perf_counter()
        self.timing = dict(register_s=t_reg - t0, prefetch_s=t_pre - t_reg, waves_s=t_end - t_pre, total_s=t_end - t0, **prof)
        edges = host.edges()
        self.log = host.log()
        self.counters = host.counters()
        self.search_stats = self.engine.search_stats() if self.gpu_search else {}
        self.graph = PoseGraph(len(self.scene["focal"]), edges)
        return self.graph

    def guided_match_edges(self, graph=None, max_points=None, bin_number=45):
        """guidedMatching (pose_graph_builder.h:717-783) for every edge of `graph` (default: the last run()'s), each with
        its own (q, t) as T_dst_src, in the graph's edge order, in one device call (K10) on the scene's resident keypoints
        and descriptors -> (offsets [E + 1] u64, matches [M, 2] u32 (src idx, dst idx), values [M] f64); edge k's rows are
        offsets[k]:offsets[k + 1].  max_points=None is kMaximumPointNumberForEpipolarHashing_, 0 gives all of match()'s
        rows with their adapted ratios."""
        if "desc" not in self.scene:
            raise ValueError("guided matching needs a scene with descriptors (desc)")
        if self.world > 1:
            raise ValueError("guided_match_edges runs on one GPU (world_size must be 1)")
        if graph is None:
            graph = getattr(self, "graph", None)
        if graph is None:
            raise ValueError("no pose graph: call run() first or pass graph=")
        if self.engine is None or not getattr(self, "prepared", False):
            self.prepare()
        if not self._desc_resident:  # a scene that came with matches: its descriptors go to the device once
            self.engine.set_scene_descriptors(self.scene["desc"])
            self._desc_resident = True
        e = graph.edges
        pv = np.stack([e["src"], e["dst"]], 1).astype(np.uint32)
        poses = np.concatenate([e["q"], e["t"]], 1) if len(e) else np.zeros((0, 7))
        mp = self.max_points_hashing if max_points is None else int(max_points)
        return self.engine.guided_match_pairs(pv, poses, bin_number, mp)

    def _run_hashing(self):
        """The exact sequential epipolar-hashing loop (pgb_run_hashing) with the engine's own entry points."""
        t0 = time.perf_counter()
        if self.engine is None or not getattr(self, "prepared", False):
            self.prepare()
        t_reg = time.perf_counter()
        host = HostBuilder(self.scene, lazy_fallback=True, **self.cfg)
        self.host = host
        lib = _engine.load_library()
        fns = [C.cast(getattr(lib, n), C.c_void_p) for n in ("pgi_submit_wave", "pgi_wait_wave", "pgi_register_extra_pairs",
                                                            "pgi_guided_match_views")]
        rc, st = host.run_hashing(self.scene["matches"], *fns, self.engine.h, self.max_tracklets, self.max_points_hashing)
        if rc < 0:
            raise _engine.PgiError(f"status {rc}: {lib.pgi_last_error(self.engine.h).decode()}")
        t_end = time.perf_counter()
        self.hashing_stats = st.as_dict()
        self.timing = dict(register_s=t_reg - t0, waves_s=t_end - t_reg, total_s=t_end - t0)
        edges = host.edges()
        self.log = host.log()
        self.match_sources = host.match_sources()
        self.counters = host.counters()
        self.search_stats = {}
        self.graph = PoseGraph(len(self.scene["focal"]), edges)
        return self.graph
