"""Epipolar-hashing mode on the device: extra pairs (pgi_register_extra_pairs + PGI_WAVE_EXTRA) against the oracle's
createCorrespondenceMatrix / estimatePose and against a static registration of the same rows; guided matching on the
resident scene (pgi_guided_match_views) against the oracle and pgi_guided_match on the same pair; descriptors added to a scene
registered with matches; PoseGraphBuilder(kUseEpipolarHashing_=True) against pgo_run_scene_hashing; bad input."""
import os
import subprocess

import numpy as np
import pytest

from helpers import perturbed_pose, pose_qt
from oracle import pgo_hashing
from test_hashing_host import LOG_FIELDS, assert_both_branches_ran, hashing_scene
from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import (WAVE_EXTRA, WAVE_FALLBACK, WAVE_MASKS, WAVE_PATH, Engine, PgiError,
                                                   library_path)

pytestmark = pytest.mark.gpu
FLAGS = WAVE_PATH | WAVE_FALLBACK | WAVE_MASKS


def _views(sc):
    ko = sc["kp_offset"].astype(np.int64)
    return ([sc["kp"][ko[v]:ko[v + 1]] for v in range(len(ko) - 1)], [sc["desc"][ko[v]:ko[v + 1]] for v in range(len(ko) - 1)])


def _K(sc, v):
    f, (w, h) = float(sc["focal"][v]), sc["size"][v]
    return np.array([[f, 0.0, w / 2.0], [0.0, f, h / 2.0], [0.0, 0.0, 1.0]])


@pytest.fixture(scope="module")
def desc_scene():
    """12 views registered from descriptors (K9 fills m_offset / matches); view 3 has no keypoint, view 7 has one."""
    counts = np.random.default_rng(11).integers(700, 1600, 12)
    counts[3], counts[7] = 0, 1
    sc = S.make_descriptor_scene(n_views=12, kp_counts=counts, dim=128, seed=11, arc=np.pi, visible_half_angle=0.6 * np.pi)
    eng = Engine(device=0)
    eng.register_scene_descriptors(sc, 0.4)
    yield sc, eng
    eng.close()


# ---- extra pairs ---------------------------------------------------------------------------------------------------------
def test_extra_pairs_equal_the_oracle_and_a_static_registration(desc_scene, oracle):
    sc, eng = desc_scene
    kp, _ = _views(sc)
    rng = np.random.default_rng(1)
    # (src, dst, matches): a scene pair's own matches; duplicated indices; index-0 rows (the tracklets' "not set");
    # an empty pair; maximum + 1 = 5 001 rows
    p = int(np.argmax(np.diff(sc["m_offset"].astype(np.int64))))
    s0, d0 = (int(x) for x in sc["pair_views"][p])
    own = sc["matches"][int(sc["m_offset"][p]):int(sc["m_offset"][p + 1])]
    dup = np.vstack([own[:60], own[:60], own[10:40]])
    zero = own[:80].copy()
    zero[::3, 0] = 0
    zero[1::4, 1] = 0
    big = np.stack([rng.integers(0, len(kp[1]), 5001), rng.integers(0, len(kp[2]), 5001)], 1)
    cases = [(s0, d0, own), (s0, d0, dup), (s0, d0, zero), (4, 5, np.zeros((0, 2))), (1, 2, big), (d0, s0, own[:, ::-1])]
    pv = np.array([(s, d) for s, d, _ in cases], dtype=np.uint32)
    mo = np.concatenate([[0], np.cumsum([len(m) for _, _, m in cases])]).astype(np.uint64)
    mt = np.vstack([np.asarray(m, dtype=np.uint32).reshape(-1, 2) for _, _, m in cases])
    eng.register_extra_pairs(pv, mo, mt)
    corr_all, thr_all = [], []
    for k, (s, d, m) in enumerate(cases):
        corr, thr = eng.read_extra_pair(k)
        f = float(sc["focal"][s])
        cx, cy = sc["size"][s] / 2.0
        ref, rthr = oracle.create_correspondences(kp[s], kp[d], np.asarray(m, dtype=np.uint32).reshape(-1, 2), f, f, cx, cy, 0.4)
        assert corr.view(np.uint64).tobytes() == ref.view(np.uint64).tobytes(), k
        assert np.float64(thr).view(np.uint64) == np.float64(rthr).view(np.uint64)
        corr_all.append(corr)
        thr_all.append(thr)
    # waves on the extra registration: without a hypothesis, and with a good / a wrong one
    ids = np.arange(len(cases), dtype=np.uint32)
    R, t = S.relative_gt(sc, s0, d0)
    good = perturbed_pose(R, t / np.linalg.norm(t), rng, 1e-4, 1e-4)
    bad = np.array([0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0])
    static = Engine(device=0)
    static.register_pairs(np.vstack(corr_all), mo, np.array(thr_all))
    for hyps in ([None] * len(cases), [good, good, bad, None, None, None]):
        hoff = np.concatenate([[0], np.cumsum([h is not None for h in hyps])]).astype(np.uint32)
        hyp = np.array([h for h in hyps if h is not None]).reshape(-1, 7)
        v, masks = eng.run_wave(ids, hoff, hyp, flags=FLAGS | WAVE_EXTRA, want_masks=True)
        vs, ms = static.run_wave(ids, hoff, hyp, flags=FLAGS, want_masks=True)
        assert v.tobytes() == vs.tobytes() and masks.tobytes() == ms.tobytes()
        for k in range(len(cases)):
            corr, thr = corr_all[k], thr_all[k]
            guesses = []
            if hyps[k] is not None and oracle.test_pose(corr, hyps[k], 1.5 * thr, 5)[0]:
                guesses = [hyps[k]]
            o = oracle.estimate_pose(corr, thr, guesses) if len(corr) else dict(success=False, inlier_number=0,
                                                                                  mask=np.zeros(0, np.uint8))
            assert bool(v[k]["accepted"]) == o["success"] and int(v[k]["inlier_count"]) == o["inlier_number"], k
            assert np.array_equal(masks[int(mo[k]):int(mo[k + 1])], o["mask"]), k
            if o["success"]:
                assert np.array_equal(v[k]["E"].reshape(3, 3), o["E"]) and int(v[k]["branch"]) == o["branch"]
                assert np.array_equal(np.concatenate([v[k]["q"], v[k]["t"]]), o["pose"])
    # the scene's own registration is untouched by the extra pairs
    corr, _ = eng.read_pair(p)
    assert np.array_equal(corr, corr_all[0])
    static.close()


# ---- guided matching on the resident scene ------------------------------------------------------------------------------
def _guided_cases(sc, rng, n):
    V = len(sc["focal"])
    out = []
    pairs = [(int(a), int(b)) for a, b in sc["pair_views"]]
    rng.shuffle(pairs)
    for s, d in pairs[:n] + [(d, s) for s, d in pairs[:10]]:
        R, t = S.relative_gt(sc, s, d)
        qt = pose_qt(R, t / max(np.linalg.norm(t), 1e-12))
        out.append((s, d, qt if len(out) % 3 else perturbed_pose(R, t, rng, 1e-3, 1e-2)))
    out += [(3, 0, out[0][2]), (0, 3, out[0][2]), (7, 2, out[1][2]), (2, 7, out[1][2]), (V - 1, 0, out[2][2])]
    return out


@pytest.mark.parametrize("dim", [128, 64])
def test_guided_match_views_equals_the_oracle_and_guided_match(desc_scene, engine, oracle, dim):
    if dim == 128:
        sc, eng = desc_scene
    else:
        counts = np.random.default_rng(12).integers(300, 1200, 10)
        counts[2] = 1
        sc = S.make_descriptor_scene(n_views=10, kp_counts=counts, dim=64, seed=12, arc=np.pi, visible_half_angle=0.6 * np.pi)
        eng = Engine(device=0)
        eng.register_scene_descriptors(sc, 0.4)
    kp, desc = _views(sc)
    rng = np.random.default_rng(dim)
    cases = _guided_cases(sc, rng, 50)
    sizes = set()
    for s, d, qt in cases:
        for max_points in (100, 10, 3):
            got = eng.guided_match_views(s, d, qt, 45, max_points)
            args = (kp[s], desc[s], kp[d], desc[d], qt, _K(sc, s), _K(sc, d), sc["size"][s], sc["size"][d])
            single = engine.guided_match(*args, bin_number=45, max_points=max_points)
            ref = oracle.guided_match(*args, bin_number=45, max_points=max_points)
            sel = [(int(a), int(b), float(r)) for (a, b), r in zip(ref["selected_matches"], ref["selected_ratios"])]
            assert got == sel == single["selected"], (s, d, max_points)
            sizes.add((len(ref["matches"]) > max_points, len(got) > 0))
    assert len(cases) >= 50 and {(True, True), (False, True)} <= sizes
    if dim == 64:
        eng.close()


def test_set_scene_descriptors_gives_the_guided_results_of_the_descriptor_registration(desc_scene):
    sc, eng = desc_scene
    withm = {k: sc[k] for k in ("focal", "size", "sim", "kp_offset", "kp", "pair_views", "m_offset", "matches", "desc")}
    e2 = Engine(device=0)
    e2.register_scene(withm, 0.4)
    with pytest.raises(PgiError, match="status -4"):  # no descriptors yet
        e2.guided_match_views(0, 1, np.array([0, 0, 0, 1.0, 1, 0, 0]))
    e2.set_scene_descriptors(withm["desc"])
    for s, d, qt in _guided_cases(sc, np.random.default_rng(5), 12):
        assert e2.guided_match_views(s, d, qt) == eng.guided_match_views(s, d, qt)
    e2.close()


# ---- end to end ---------------------------------------------------------------------------------------------------------
def _compare_with_oracle(oracle, sc, pgb, path_finding):
    olog, oedges, osrc = pgo_hashing.run_scene_hashing(sc, sim_threshold=0.0, use_path_finding=path_finding)
    plog, src = pgb.log, pgb.match_sources
    assert len(plog) == len(olog)
    for f in LOG_FIELDS:
        assert np.array_equal(plog[f], olog[f]), f
    g = pgb.host.edges()
    assert len(g) == len(oedges)
    for f in ("src", "dst", "q", "t", "score"):
        assert np.array_equal(g[f], oedges[f]), f
    assert np.array_equal(g["n_corr"], plog["nCorr"][plog["committed"] > 0])
    assert np.array_equal(src["source"], osrc["source"]) and np.array_equal(src["guided_rows"], osrc["guided_rows"])
    assert_both_branches_ran(src, plog)


@pytest.mark.parametrize("which,path_finding", [("12v", True), ("24v", False), ("12v-container", True), ("40v-device", True)])
def test_builder_hashing_mode_commits_what_the_oracle_commits(oracle, tmp_path, which, path_finding):
    if which == "40v-device":  # keypoints + descriptors only: matched by K9 in prepare()
        sc = S.make_descriptor_scene(n_views=40, kp_range=(500, 900), dim=64, seed=7, arc=np.pi, visible_half_angle=0.6 * np.pi)
    else:
        sc = hashing_scene(12, 3) if which.startswith("12v") else hashing_scene(24, 4)
    if which.endswith("container"):  # version-2 container carrying desc and matches
        path = str(tmp_path / "scene.pgi")
        S.save_scene(path, sc)
        sc = S.load_scene(path)
        assert "desc" in sc and "matches" in sc
    pgb = B.PoseGraphBuilder(kUseEpipolarHashing_=True, kUsePathFinding_=path_finding, kSimilarityThreshold_=0.0, scene=sc)
    g = pgb.run()
    assert pgb.engine_fb is None and pgb.engine_fb2 is None  # no background contexts in this mode
    st = pgb.hashing_stats
    assert st["positions"] == len(pgb.log) and st["quick_matched"] > 0 and st["guided_calls"] > 0
    assert g.numEdges() == int(pgb.log["committed"].sum())
    _compare_with_oracle(oracle, sc, pgb, path_finding)
    es = pgb.engine.stats()
    assert es["guided_calls"] == st["guided_calls"] and es["ms_guided"] > 0
    pgb.close()


# ---- bad input ----------------------------------------------------------------------------------------------------------
def test_bad_input(desc_scene):
    sc, _ = desc_scene
    nodesc = {k: v for k, v in sc.items() if k != "desc"}
    for kw in (dict(scene=nodesc), dict(scene=sc, world_size=2), dict(scene=sc, gpu_search=True)):
        with pytest.raises(ValueError):
            B.PoseGraphBuilder(kUseEpipolarHashing_=True, **kw)
    pgb = B.PoseGraphBuilder(kUseEpipolarHashing_=True, scene=hashing_scene(8, 6))
    with pytest.raises(ValueError):
        next(pgb.run_in_batches(5))
    pgb.close()
    e = Engine(device=0)
    qt = np.array([0, 0, 0, 1.0, 1, 0, 0])
    for call in (lambda: e.register_extra_pairs([[0, 1]], [0, 1], [[0, 0]]), lambda: e.guided_match_views(0, 1, qt),
                 lambda: e.set_scene_descriptors(sc["desc"])):
        with pytest.raises(PgiError, match="status -4"):  # before any scene registration
            call()
    e.register_scene_descriptors(dict(sc), 0.4)
    n0 = int(sc["kp_offset"][1] - sc["kp_offset"][0])
    for call in (lambda: e.register_extra_pairs([[0, 99]], [0, 1], [[0, 0]]),      # view out of range
                 lambda: e.register_extra_pairs([[0, 1]], [0, 1], [[n0, 0]]),      # keypoint index out of range
                 lambda: e.register_extra_pairs([[0, 1]], [1, 2], [[0, 0], [0, 0]]),  # m_offset[0] != 0
                 lambda: e.guided_match_views(0, 99, qt),
                 lambda: e.guided_match_views(0, 1, qt, bin_number=1000),
                 lambda: e.set_scene_descriptors(sc["desc"][:, :32]),
                 lambda: e.set_scene_descriptors(np.where(np.arange(sc["desc"].size).reshape(sc["desc"].shape) == 5, np.nan, sc["desc"]))):
        with pytest.raises(PgiError, match="status -1"):
            call()
    # a view of more keypoints than guided matching supports is rejected when its descriptors arrive
    big = dict(focal=np.array([1000.0, 1000.0]), size=np.array([[1600.0, 1200.0]] * 2), kp=np.zeros((16395, 2), np.float32),
               kp_offset=np.array([0, 16385, 16395], dtype=np.uint64), pair_views=np.array([[0, 1]], dtype=np.uint32),
               m_offset=np.zeros(2, dtype=np.uint64), matches=np.zeros((0, 2), dtype=np.uint32))
    e.register_scene(big, 0.4)
    with pytest.raises(PgiError, match="at most 16384"):
        e.set_scene_descriptors(np.zeros((16395, 128), np.float32))
    e.close()


def test_library_exports_the_new_symbols():
    out = subprocess.run(["nm", "-D", "--defined-only", library_path()], capture_output=True, text=True, check=True).stdout
    names = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for n in ("pgi_register_extra_pairs", "pgi_read_extra_pair", "pgi_guided_match_views", "pgi_set_scene_descriptors",
              "pgb_run_hashing", "pgb_copy_match_sources"):
        assert n in names, n
    assert os.path.basename(library_path()) == "libpgi.so"
