"""ctypes binding of the C-ABI in include/pgi.h (the sm_100a hypothesis-verification engine).

This is plumbing: numpy arrays in, numpy arrays out; every call goes through libpgi.so.  There is no
CPU compute path — `Engine()` raises if the library is missing or no sm_100 device is usable.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

PGI_OK = 0
WAVE_PATH, WAVE_FALLBACK, WAVE_MASKS, WAVE_NO_TEST, WAVE_EXTRA = 1, 2, 4, 8, 16

VERDICT_DTYPE = np.dtype(
    [
        ("pair_id", np.uint32), ("branch", np.uint8), ("accepted", np.uint8), ("test_passed", np.uint8),
        ("n_hypotheses", np.uint8), ("test_count", np.uint32), ("inlier_count", np.uint32), ("n_corr", np.uint32),
        ("path_inliers", np.uint32), ("E", np.float64, (9,)), ("q", np.float64, (4,)), ("t", np.float64, (3,)),
        ("iters", np.uint32), ("status", np.uint32),
    ],
    align=True,
)
assert VERDICT_DTYPE.itemsize == 160


class PgiConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("min_inliers", C.c_uint32), ("test_min_inliers", C.c_uint32),
                ("fallback_max_iters", C.c_uint32), ("threshold_multiplier", C.c_double), ("max_wave", C.c_uint32),
                ("flags", C.c_uint32)]


class PgiStats(C.Structure):
    _fields_ = [("ms_correspondences", C.c_double), ("ms_score", C.c_double), ("ms_fivept", C.c_double),
                ("ms_fallback_solve", C.c_double), ("ms_fallback_score", C.c_double), ("ms_decompose", C.c_double),
                ("ms_total", C.c_double), ("launches", C.c_uint64), ("pairs", C.c_uint64), ("corr_evals", C.c_uint64),
                ("fallback_pairs", C.c_uint64), ("fallback_models", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("ms_match", C.c_double), ("dist_evals", C.c_uint64), ("match_pairs", C.c_uint64),
                ("match_rows", C.c_uint64), ("ms_guided", C.c_double), ("guided_calls", C.c_uint64),
                ("ms_guided_pairs", C.c_double), ("guided_pairs", C.c_uint64), ("guided_dist_evals", C.c_uint64),
                ("guided_chunks", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


EXPORTS = [
    "pgi_version", "pgi_device_count", "pgi_create", "pgi_destroy", "pgi_last_error", "pgi_register_pairs",
    "pgi_register_scene", "pgi_share_pairs", "pgi_read_pair", "pgi_submit_wave", "pgi_wait_wave", "pgi_wait_wave_device",
    "pgi_estimate_pose", "pgi_test_pose", "pgi_graph_init", "pgi_graph_apply", "pgi_graph_search", "pgi_graph_stats",
    "pgi_guided_match", "pgi_match_features", "pgi_get_stats", "pgi_reset_stats", "pgi_dbg_sampson",
    "pgi_dbg_five_point", "pgi_dbg_pose_from_essential", "pgi_dbg_fp64_peak", "pgi_register_scene_descriptors",
    "pgi_read_scene_matches", "pgi_set_scene_descriptors", "pgi_register_extra_pairs", "pgi_read_extra_pair",
    "pgi_guided_match_views", "pgi_guided_match_pairs",
]

_lib = None


def library_path():
    return _build.LIB


def load_library():
    """dlopen libpgi.so (building it first if the sources are newer).  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB) or _build.needs_build():
        _build.build()
    lib = C.CDLL(_build.LIB)
    lib.pgi_version.restype = C.c_char_p
    lib.pgi_last_error.restype = C.c_char_p
    lib.pgi_last_error.argtypes = [C.c_void_p]
    lib.pgi_device_count.restype = C.c_int32
    lib.pgi_create.argtypes = [C.POINTER(PgiConfig), C.POINTER(C.c_void_p)]
    for name in EXPORTS:
        getattr(lib, name)  # AttributeError if a declared symbol is missing
    for name in EXPORTS[5:]:
        getattr(lib, name).restype = C.c_int32
    lib.pgi_share_pairs.argtypes = [C.c_void_p, C.c_void_p]
    lib.pgi_destroy.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


ADJ_ENTRY_DTYPE = np.dtype([("vertex", np.uint32), ("index", np.uint32), ("next", np.uint32), ("tag", np.uint32),
                            ("score", np.float64)], align=True)
QUERY_DTYPE = np.dtype([("src", np.uint32), ("dst", np.uint32), ("cutoff", np.uint32), ("budget", np.uint32)], align=True)
SEARCH_RESULT_DTYPE = np.dtype([("touched", np.uint32), ("pushes", np.uint32), ("path", np.uint16, (8,)), ("found", np.uint8),
                                ("path_len", np.uint8), ("status", np.uint8), ("pad", np.uint8), ("kcycles", np.uint32)],
                               align=True)
assert ADJ_ENTRY_DTYPE.itemsize == 24 and QUERY_DTYPE.itemsize == 16 and SEARCH_RESULT_DTYPE.itemsize == 32


class PgiSearchStats(C.Structure):
    _fields_ = [("ms_search", C.c_double)] + [(k, C.c_uint64) for k in ("launches", "queries", "pops", "pushes", "overflows",
                                                                         "h2d_bytes", "d2h_bytes", "kcycles_sum", "kcycles_longest")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class PgiError(RuntimeError):
    pass


class Engine:
    """One context per (process, GPU)."""

    def __init__(self, device=0, min_inliers=20, test_min_inliers=5, fallback_max_iters=1000, max_wave=4096, background=False):
        self.lib = load_library()
        if self.lib.pgi_device_count() <= 0:
            raise PgiError("no usable sm_100 CUDA device: the hypothesis-verification engine has no CPU path")
        cfg = PgiConfig(device, min_inliers, test_min_inliers, fallback_max_iters, 1.5, max_wave, 1 if background else 0)
        h = C.c_void_p()
        st = self.lib.pgi_create(C.byref(cfg), C.byref(h))
        if st != PGI_OK:
            raise PgiError(f"pgi_create failed with status {st}")
        self.h = h
        self.n_pairs = 0
        self.offset = None
        self.extra_offset = None
        self._kp_offset = None
        self._wave_n = 0
        self._wave_rows = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.pgi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st):
        if st != PGI_OK:
            raise PgiError(f"status {st}: {self.lib.pgi_last_error(self.h).decode()}")

    # ---- registration -------------------------------------------------------------------------------
    def register_pairs(self, corr, offset, thr_norm):
        corr = _f64(corr).reshape(-1, 4)
        offset = np.ascontiguousarray(offset, dtype=np.uint64)
        thr_norm = _f64(thr_norm)
        assert len(thr_norm) == len(offset) - 1 and int(offset[-1]) == len(corr)
        self._ck(self.lib.pgi_register_pairs(self.h, C.c_uint64(len(thr_norm)), _ptr(offset), _ptr(corr), _ptr(thr_norm)))
        self.n_pairs, self.offset = len(thr_norm), offset.copy()

    def register_scene(self, scene, thr_px=0.4):
        focal = _f64(scene["focal"]); size = _f64(scene["size"])
        kpo = np.ascontiguousarray(scene["kp_offset"], dtype=np.uint64)
        kp = np.ascontiguousarray(scene["kp"], dtype=np.float32)
        pv = np.ascontiguousarray(scene["pair_views"], dtype=np.uint32)
        mo = np.ascontiguousarray(scene["m_offset"], dtype=np.uint64)
        mt = np.ascontiguousarray(scene["matches"], dtype=np.uint32)
        self._ck(self.lib.pgi_register_scene(self.h, C.c_uint64(len(focal)), _ptr(focal), _ptr(size), _ptr(kpo), _ptr(kp),
                                             C.c_uint64(len(pv)), _ptr(pv), _ptr(mo), _ptr(mt), C.c_double(thr_px)))
        self.n_pairs, self.offset = len(pv), mo.copy()
        self._kp_offset = kpo.copy()

    def register_scene_descriptors(self, scene, thr_px=0.4):
        """matchFeatures for every pair of `scene` on the device (K9), then the registration of register_scene from the
        device-resident matches.  scene needs desc[sum K, dim] (float32, dim 64 or 128) beside the keys register_scene
        reads, except m_offset / matches, which this fills in — with scene["ratios"], the scene's correspondences.h5."""
        focal = _f64(scene["focal"]); size = _f64(scene["size"])
        kpo = np.ascontiguousarray(scene["kp_offset"], dtype=np.uint64)
        kp = np.ascontiguousarray(scene["kp"], dtype=np.float32)
        desc = np.ascontiguousarray(scene["desc"], dtype=np.float32)
        pv = np.ascontiguousarray(scene["pair_views"], dtype=np.uint32)
        if desc.ndim != 2 or len(desc) != len(kp) or len(kpo) != len(focal) + 1 or int(kpo[-1]) != len(kp):
            raise ValueError("desc must be a [sum K, dim] array row-aligned with kp / kp_offset")
        mo = np.zeros(len(pv) + 1, dtype=np.uint64)
        self._ck(self.lib.pgi_register_scene_descriptors(self.h, C.c_uint64(len(focal)), _ptr(focal), _ptr(size), _ptr(kpo),
                                                         _ptr(kp), _ptr(desc), C.c_uint32(desc.shape[1]), C.c_uint64(len(pv)),
                                                         _ptr(pv), C.c_double(thr_px), _ptr(mo)))
        self.n_pairs, self.offset = len(pv), mo.copy()
        self._kp_offset = kpo.copy()
        matches, ratios = self.read_scene_matches(int(mo[-1]))
        scene["m_offset"], scene["matches"], scene["ratios"] = mo, matches, ratios
        return mo

    def read_scene_matches(self, n_rows):
        """(matches [n_rows, 2] u32, ratios [n_rows]) of the last register_scene_descriptors."""
        m = np.zeros((n_rows, 2), dtype=np.uint32)
        r = np.zeros(n_rows)
        self._ck(self.lib.pgi_read_scene_matches(self.h, _ptr(m), _ptr(r), C.c_uint64(n_rows)))
        return m, r

    def set_scene_descriptors(self, desc):
        """Descriptors [sum K, dim] (float32, dim 64 or 128) of the scene registered by register_scene, row-aligned with its
        keypoints; they stay on the device for guided_match_views."""
        desc = np.ascontiguousarray(desc, dtype=np.float32)
        if desc.ndim != 2:
            raise ValueError("desc must be a [sum K, dim] array")
        self._ck(self.lib.pgi_set_scene_descriptors(self.h, _ptr(desc), C.c_uint32(desc.shape[1])))

    def register_extra_pairs(self, pair_views, m_offset, matches):
        """Correspondences of caller-supplied matches (pair_views [n, 2], m_offset [n + 1], matches [M, 2]) built on the
        device from the registered scene's keypoints; waves address them with WAVE_EXTRA."""
        pv = np.ascontiguousarray(pair_views, dtype=np.uint32).reshape(-1, 2)
        mo = np.ascontiguousarray(m_offset, dtype=np.uint64)
        mt = np.ascontiguousarray(matches, dtype=np.uint32).reshape(-1, 2)
        if len(mo) != len(pv) + 1 or int(mo[-1]) != len(mt):
            raise ValueError("m_offset must have n_pairs + 1 entries ending at len(matches)")
        self._ck(self.lib.pgi_register_extra_pairs(self.h, C.c_uint64(len(pv)), _ptr(pv), _ptr(mo), _ptr(mt)))
        self.extra_offset = mo.copy()

    def read_extra_pair(self, pair_id):
        n = int(self.extra_offset[pair_id + 1] - self.extra_offset[pair_id])
        corr = np.empty((n, 4))
        rows, thr = C.c_uint64(0), C.c_double(0)
        self._ck(self.lib.pgi_read_extra_pair(self.h, C.c_uint32(pair_id), _ptr(corr), C.c_uint64(n), C.byref(rows), C.byref(thr)))
        return corr, thr.value

    def share_pairs(self, owner):
        """Use the pairs registered in `owner` (same device) without copying them."""
        self._ck(self.lib.pgi_share_pairs(self.h, owner.h))
        self.n_pairs, self.offset = owner.n_pairs, owner.offset

    def read_pair(self, pair_id):
        n = int(self.offset[pair_id + 1] - self.offset[pair_id])
        corr = np.empty((n, 4))
        rows, thr = C.c_uint64(0), C.c_double(0)
        self._ck(self.lib.pgi_read_pair(self.h, C.c_uint32(pair_id), _ptr(corr), C.c_uint64(n), C.byref(rows), C.byref(thr)))
        return corr, thr.value

    # ---- waves ----------------------------------------------------------------------------------------
    def submit_wave(self, pair_ids, hyp_offset=None, hyp=None, flags=WAVE_PATH | WAVE_FALLBACK):
        pair_ids = np.ascontiguousarray(pair_ids, dtype=np.uint32)
        n = len(pair_ids)
        if hyp_offset is None:
            hyp_offset = np.zeros(n + 1, dtype=np.uint32)
        hyp_offset = np.ascontiguousarray(hyp_offset, dtype=np.uint32)
        hyp = _f64(hyp).reshape(-1, 7) if hyp is not None and len(hyp) else np.zeros((0, 7))
        self._ck(self.lib.pgi_submit_wave(self.h, C.c_uint32(n), _ptr(pair_ids), _ptr(hyp_offset), _ptr(hyp), C.c_uint32(flags)))
        self._wave_n = n
        off = self.extra_offset if flags & WAVE_EXTRA else self.offset
        self._wave_rows = int(sum(int(off[p + 1] - off[p]) for p in pair_ids)) if flags & WAVE_MASKS else 0

    def wait_wave(self, want_masks=False):
        out = np.zeros(self._wave_n, dtype=VERDICT_DTYPE)
        masks = np.zeros(self._wave_rows, dtype=np.uint8) if want_masks else None
        self._ck(self.lib.pgi_wait_wave(self.h, _ptr(out), _ptr(masks)))
        return (out, masks) if want_masks else out

    def wait_wave_device(self, device_ptr):
        self._ck(self.lib.pgi_wait_wave_device(self.h, C.c_void_p(device_ptr)))

    def run_wave(self, pair_ids, hyp_offset=None, hyp=None, flags=WAVE_PATH | WAVE_FALLBACK, want_masks=False):
        if want_masks:
            flags |= WAVE_MASKS
        self.submit_wave(pair_ids, hyp_offset, hyp, flags)
        return self.wait_wave(want_masks)

    # ---- reference-shaped single-pair calls --------------------------------------------------------------
    def estimate_pose(self, corr, thr_norm, guesses=()):
        """PoseGraphBuilder::estimatePose (pose_graph_builder.h:940-1078)."""
        corr = _f64(corr).reshape(-1, 4)
        g = _f64(np.asarray(guesses, dtype=np.float64).reshape(-1, 7)) if len(guesses) else np.zeros((0, 7))
        pose = np.zeros(7)
        mask = np.zeros(len(corr), dtype=np.uint8)
        inl = C.c_uint64(0)
        v = np.zeros(1, dtype=VERDICT_DTYPE)
        r = self.lib.pgi_estimate_pose(self.h, _ptr(corr), C.c_uint64(len(corr)), C.c_double(thr_norm), _ptr(g),
                                       C.c_uint32(len(g)), _ptr(pose), _ptr(mask), C.byref(inl), _ptr(v))
        if r < 0:
            self._ck(r)
        return dict(success=bool(r), pose=pose, mask=mask, inlier_number=int(inl.value), verdict=v[0])

    def test_pose(self, corr, thr, pose, min_inliers=5):
        """InTraversalPoseTester::test (graph_traversal.h:194-233)."""
        corr = _f64(corr).reshape(-1, 4)
        pose = _f64(pose)
        inl = C.c_uint64(0)
        r = self.lib.pgi_test_pose(self.h, _ptr(corr), C.c_uint64(len(corr)), C.c_double(thr), C.c_uint64(min_inliers),
                                   _ptr(pose), C.byref(inl))
        if r < 0:
            self._ck(r)
        return bool(r), int(inl.value)

    # ---- A* on the device (K6) ---------------------------------------------------------------------------
    def graph_init(self, sim_to_next):
        """sim_to_next: V x V, clamped and transposed (HostBuilder.sim_table())."""
        t = _f64(sim_to_next)
        self._graph_V = len(t)
        self._ck(self.lib.pgi_graph_init(self.h, C.c_uint32(len(t)), _ptr(t)))

    def graph_apply(self, entries, committed_count, total_count):
        entries = np.ascontiguousarray(entries, dtype=ADJ_ENTRY_DTYPE)
        cc = np.ascontiguousarray(committed_count, dtype=np.uint32)
        tc = np.ascontiguousarray(total_count, dtype=np.uint32)
        self._ck(self.lib.pgi_graph_apply(self.h, C.c_uint32(len(entries)), _ptr(entries), _ptr(cc), _ptr(tc)))

    def graph_search(self, queries, max_depth=5, weight=0.8):
        queries = np.ascontiguousarray(queries, dtype=QUERY_DTYPE)
        n = len(queries)
        words = (self._graph_V + 31) // 32
        res = np.zeros(n, dtype=SEARCH_RESULT_DTYPE)
        bits = np.zeros((n, words), dtype=np.uint32)
        self._ck(self.lib.pgi_graph_search(self.h, C.c_uint32(n), _ptr(queries), C.c_uint32(max_depth), C.c_double(weight),
                                           _ptr(res), _ptr(bits)))
        return res, bits

    def search_stats(self, reset=False):
        s = PgiSearchStats()
        self._ck(self.lib.pgi_graph_stats(self.h, C.byref(s), C.c_int32(1 if reset else 0)))
        return s.as_dict()

    # ---- epipolar-hashing guided matcher (K10) --------------------------------------------------------------
    def guided_match(self, kp_src, desc_src, kp_dst, desc_dst, pose_qt, K_src, K_dst, size_src, size_dst, bin_number=45,
                     max_points=100):
        """HashingBasedMatcherWithPose<false, 45>::match on the device + guidedMatching's selection
        (pose_graph_builder.h:717-783).  Returns dict(matches[n,2], ratios[n], selected[(src, dst, value)], prepared[14])."""
        ks = np.ascontiguousarray(kp_src, dtype=np.float32).reshape(-1, 2)
        kd = np.ascontiguousarray(kp_dst, dtype=np.float32).reshape(-1, 2)
        ds = np.ascontiguousarray(desc_src, dtype=np.float32)
        dd = np.ascontiguousarray(desc_dst, dtype=np.float32)
        if ds.ndim != 2 or dd.ndim != 2 or len(ds) != len(ks) or len(dd) != len(kd) or ds.shape[1] != dd.shape[1]:
            raise ValueError("descriptors must be [n_src, dim] / [n_dst, dim] arrays matching the keypoints")
        m = np.zeros((max(len(ks), 1), 2), dtype=np.uint32)
        r = np.zeros(max(len(ks), 1))
        n = C.c_uint32(0)
        prep = np.zeros(14)
        ss = np.asarray(size_src, dtype=np.int32)
        sd = np.asarray(size_dst, dtype=np.int32)
        self._ck(self.lib.pgi_guided_match(self.h, C.c_uint32(len(ks)), _ptr(ks), _ptr(ds), C.c_uint32(len(kd)), _ptr(kd), _ptr(dd),
                                           C.c_uint32(ds.shape[1]), _ptr(_f64(pose_qt)), _ptr(_f64(K_src)), _ptr(_f64(K_dst)),
                                           _ptr(ss), _ptr(sd), C.c_int32(bin_number), _ptr(m), _ptr(r), C.byref(n), _ptr(prep)))
        k = int(n.value)
        matches, ratios = m[:k].copy(), r[:k].copy()
        # guidedMatching's selection (pose_graph_builder.h:760-782): the max_points smallest values (min-heap order on
        # (value, index)); at most max_points matches: every match carries descriptorDistances[0]
        if k > max_points:
            order = np.lexsort((np.arange(k), ratios))[:max_points]
            selected = [(int(matches[i, 0]), int(matches[i, 1]), float(ratios[i])) for i in order]
        else:
            selected = [(int(a), int(b), float(ratios[0])) for a, b in matches]
        return dict(matches=matches, ratios=ratios, selected=selected, prepared=prep)

    def guided_match_views(self, src, dst, pose_qt, bin_number=45, max_points=100):
        """guidedMatching (pose_graph_builder.h:717-783) of views src -> dst of the registered scene on its device-resident
        keypoints and descriptors -> the selected rows [(src idx, dst idx, value)], as guided_match(...)["selected"]."""
        cap = max(int(max_points), 1)
        m = np.zeros((cap, 2), dtype=np.uint32)
        r = np.zeros(cap)
        n = C.c_uint32(0)
        pose = _f64(pose_qt).reshape(7)
        self._ck(self.lib.pgi_guided_match_views(self.h, C.c_uint32(src), C.c_uint32(dst), _ptr(pose), C.c_int32(bin_number),
                                                 C.c_uint32(max_points), _ptr(m), _ptr(r), C.byref(n)))
        k = int(n.value)
        return [(int(m[i, 0]), int(m[i, 1]), float(r[i])) for i in range(k)]

    def guided_match_pairs(self, pair_views, poses, bin_number=45, max_points=100):
        """guidedMatching (pose_graph_builder.h:717-783) for every (src, dst) row of pair_views [n, 2] with the pose of the
        same row of poses [n, 7] (T_dst_src) in one device call (K10) on the registered scene -> (offsets [n + 1] u64,
        matches [M, 2] u32 (src idx, dst idx), values [M] f64): pair k's rows are offsets[k]:offsets[k + 1], those of
        guided_match_views(src, dst, pose, bin_number, max_points); max_points=0 gives match()'s rows and adapted ratios."""
        pv = np.ascontiguousarray(pair_views, dtype=np.uint32).reshape(-1, 2)
        poses = _f64(poses).reshape(-1, 7)
        if len(poses) != len(pv):
            raise ValueError("poses must have one row (qx qy qz qw tx ty tz) per pair")
        # the capacity from the registered keypoint counts (the library itself rejects a missing scene or a bad view id)
        n_kp = np.diff(self._kp_offset.astype(np.int64)) if self._kp_offset is not None else np.zeros(0, dtype=np.int64)
        src = pv[:, 0].astype(np.int64)
        n_src = n_kp[src[src < len(n_kp)]]
        cap = int(np.minimum(n_src, max_points).sum() if max_points else n_src.sum())
        off = np.zeros(len(pv) + 1, dtype=np.uint64)
        m = np.zeros((max(cap, 1), 2), dtype=np.uint32)
        v = np.zeros(max(cap, 1))
        self._ck(self.lib.pgi_guided_match_pairs(self.h, C.c_uint64(len(pv)), _ptr(pv), _ptr(poses), C.c_int32(bin_number),
                                                 C.c_uint32(max_points), _ptr(off), _ptr(m), _ptr(v), C.c_uint64(cap)))
        k = int(off[-1])
        return off, m[:k].copy(), v[:k].copy()

    def match_features(self, desc_src, desc_dst):
        """matchFeatures (feature_utils.h:103-210) on the device: -> (matches [n, 2] (queryIdx, trainIdx), ratios [n]),
        sorted by ratio as the reference stores them."""
        ds = np.ascontiguousarray(desc_src, dtype=np.float32)
        dd = np.ascontiguousarray(desc_dst, dtype=np.float32)
        if ds.ndim != 2 or dd.ndim != 2 or ds.shape[1] != dd.shape[1] or ds.shape[1] not in (64, 128):
            raise ValueError("descriptors must be [n, 64] or [n, 128] float arrays of equal width")
        m = np.zeros((max(len(ds), 1), 2), dtype=np.uint32)
        r = np.zeros(max(len(ds), 1))
        n = C.c_uint32(0)
        self._ck(self.lib.pgi_match_features(self.h, C.c_uint32(len(ds)), _ptr(ds), C.c_uint32(len(dd)), _ptr(dd),
                                             C.c_uint32(ds.shape[1]), _ptr(m), _ptr(r), C.byref(n)))
        k = int(n.value)
        return m[:k].copy(), r[:k].copy()

    # ---- stats / debug -------------------------------------------------------------------------------------
    def stats(self):
        s = PgiStats()
        self._ck(self.lib.pgi_get_stats(self.h, C.byref(s)))
        return s.as_dict()

    def reset_stats(self):
        self._ck(self.lib.pgi_reset_stats(self.h))

    def dbg_sampson(self, corr, E):
        corr, E = _f64(corr).reshape(-1, 4), _f64(E).reshape(9)
        out = np.empty(len(corr))
        self._ck(self.lib.pgi_dbg_sampson(self.h, _ptr(corr), C.c_uint64(len(corr)), _ptr(E), _ptr(out)))
        return out

    def dbg_five_point(self, x1, x2, dk_max_iters=1000, dk_tol_sq=0.0):
        x1, x2 = _f64(x1).reshape(-1, 10), _f64(x2).reshape(-1, 10)
        n = len(x1)
        E = np.zeros((n, 10, 3, 3))
        cnt = np.zeros(n, dtype=np.int32)
        self._ck(self.lib.pgi_dbg_five_point(self.h, _ptr(x1), _ptr(x2), C.c_uint32(n), C.c_int32(dk_max_iters),
                                             C.c_double(dk_tol_sq), _ptr(E), _ptr(cnt)))
        return E, cnt

    def dbg_pose_from_essential(self, E, corr):
        E, corr = _f64(E).reshape(9), _f64(corr).reshape(-1, 4)
        R, t = np.empty(9), np.empty(3)
        votes = np.zeros(4, dtype=np.uint64)
        self._ck(self.lib.pgi_dbg_pose_from_essential(self.h, _ptr(E), _ptr(corr), C.c_uint64(len(corr)), _ptr(R), _ptr(t), _ptr(votes)))
        return R.reshape(3, 3), t, votes

    def fp64_peak(self, fused=False):
        out = C.c_double(0)
        self._ck(self.lib.pgi_dbg_fp64_peak(self.h, C.c_int32(1 if fused else 0), C.byref(out)))
        return out.value
