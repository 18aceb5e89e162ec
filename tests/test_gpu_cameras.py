"""Scenes in which every view has its own camera (focal length and image size), as 1DSfM's list_with_focals.txt gives them:
K0's correspondence rows against the oracle's createCorrespondenceMatrix and against a numpy statement of the reference's
quirk (both images normalised with the SOURCE view's K, threshold by the source focal length; pose_graph_builder.h:908-912,
:934-937), for scene, descriptor-matched and extra-pair registrations; guided matching with K_src != K_dst and different
image sizes, single-pair and on the resident scene, against the oracle; PoseGraphBuilder (waves and epipolar hashing) against the
oracle's sequential runs.  With one camera for all views, a swapped K or image size could not fail any of these."""
import numpy as np
import pytest

from helpers import intrinsics, per_view_camera_scene, pose_qt
from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import Engine
from test_gpu_hashing import _compare_with_oracle
from test_gpu_scene import run_and_compare

pytestmark = pytest.mark.gpu
THR_PX = 0.4


@pytest.fixture(scope="module")
def cam_scene():
    sc = per_view_camera_scene(n_views=12, seed=1, with_matches=True)
    assert len(set(sc["focal"])) >= 4 and sc["focal"].max() >= 3 * sc["focal"].min()
    assert len({tuple(s) for s in sc["size"]}) >= 4
    return sc


def _views(sc):
    ko = sc["kp_offset"].astype(np.int64)
    V = len(ko) - 1
    return [sc["kp"][ko[v]:ko[v + 1]] for v in range(V)], [sc["desc"][ko[v]:ko[v + 1]] for v in range(V)]


def _quirk_rows(kp_src, kp_dst, m, f_src, size_src):
    """createCorrespondenceMatrix as the reference computes it: all four columns (kp - size_src / 2) / f_src."""
    c = np.asarray(size_src, dtype=np.float64) / 2.0
    a = kp_src[m[:, 0]].astype(np.float64)
    b = kp_dst[m[:, 1]].astype(np.float64)
    return np.hstack([(a - c) / f_src, (b - c) / f_src]).reshape(-1, 4), THR_PX / f_src


def _check_rows(oracle, sc, kp, s, d, m, corr, thr):
    m = np.asarray(m, dtype=np.uint32).reshape(-1, 2)
    f = float(sc["focal"][s])
    cx, cy = sc["size"][s] / 2.0
    ref, rthr = oracle.create_correspondences(kp[s], kp[d], m, f, f, cx, cy, THR_PX)
    assert corr.tobytes() == ref.tobytes(), (s, d)
    assert np.float64(thr).tobytes() == np.float64(rthr).tobytes(), (s, d)
    q, qthr = _quirk_rows(kp[s], kp[d], m, f, sc["size"][s])
    assert corr.tobytes() == q.tobytes(), (s, d)
    assert np.float64(thr).tobytes() == np.float64(qthr).tobytes(), (s, d)


def _cross_camera(sc, s, d):
    return sc["focal"][s] != sc["focal"][d] and tuple(sc["size"][s]) != tuple(sc["size"][d])


def test_scene_and_descriptor_registrations_normalise_with_the_source_camera(cam_scene, oracle):
    sc = cam_scene
    kp, _ = _views(sc)
    eng = Engine(device=0)
    eng.register_scene(sc, THR_PX)
    cross = 0
    for p, (s, d) in enumerate(sc["pair_views"]):
        s, d = int(s), int(d)
        corr, thr = eng.read_pair(p)
        m = sc["matches"][int(sc["m_offset"][p]):int(sc["m_offset"][p + 1])]
        assert len(m) > 50
        _check_rows(oracle, sc, kp, s, d, m, corr, thr)
        cross += _cross_camera(sc, s, d)
    assert cross >= 40
    # the same views matched on the device from their descriptors (K9), then registered from the resident matches
    dsc = {k: v for k, v in sc.items() if k not in ("m_offset", "matches")}
    eng.register_scene_descriptors(dsc, THR_PX)
    rows = 0
    for p, (s, d) in enumerate(dsc["pair_views"]):
        corr, thr = eng.read_pair(p)
        m = dsc["matches"][int(dsc["m_offset"][p]):int(dsc["m_offset"][p + 1])]
        _check_rows(oracle, dsc, kp, int(s), int(d), m, corr, thr)
        rows += len(m)
    assert rows > 10000
    eng.close()


def test_extra_pairs_on_asymmetric_pairs_normalise_with_the_source_camera(cam_scene, oracle):
    sc = cam_scene
    kp, _ = _views(sc)
    eng = Engine(device=0)
    eng.register_scene(sc, THR_PX)
    cases = []
    for p, (s, d) in enumerate(sc["pair_views"]):
        s, d = int(s), int(d)
        if _cross_camera(sc, s, d) and len(cases) < 16:
            m = sc["matches"][int(sc["m_offset"][p]):int(sc["m_offset"][p + 1])]
            cases += [(s, d, m), (d, s, m[:, ::-1])]  # both directions: the source camera changes with the direction
    pv = np.array([(s, d) for s, d, _ in cases], dtype=np.uint32)
    mo = np.concatenate([[0], np.cumsum([len(m) for _, _, m in cases])]).astype(np.uint64)
    eng.register_extra_pairs(pv, mo, np.vstack([np.ascontiguousarray(m) for _, _, m in cases]))
    for k, (s, d, m) in enumerate(cases):
        corr, thr = eng.read_extra_pair(k)
        assert len(corr) > 50
        _check_rows(oracle, sc, kp, s, d, m, corr, thr)
    assert len(cases) == 16
    eng.close()


def _guided_cases(sc):
    """Neighbouring views with different cameras, in both directions, at the ground-truth relative pose."""
    V = len(sc["focal"])
    out = []
    for s in range(V - 1):
        for d in (s + 1, s + 2):
            if d < V and _cross_camera(sc, s, d):
                for a, b in ((s, d), (d, s)):
                    R, t = S.relative_gt(sc, a, b)
                    out.append((a, b, pose_qt(R, t / np.linalg.norm(t))))
    return out


def test_guided_matching_with_different_cameras_equals_the_oracle(cam_scene, engine, oracle):
    sc = cam_scene
    kp, desc = _views(sc)
    eng = Engine(device=0)
    eng.register_scene(sc, THR_PX)
    eng.set_scene_descriptors(sc["desc"])
    cases = _guided_cases(sc)
    assert len(cases) >= 8
    cut = 0
    for s, d, qt in cases:
        Ks, Kd = intrinsics(sc["focal"][s], sc["size"][s]), intrinsics(sc["focal"][d], sc["size"][d])
        args = (kp[s], desc[s], kp[d], desc[d], qt, Ks, Kd, sc["size"][s], sc["size"][d])
        for max_points in (100, 1000):
            ref = oracle.guided_match(*args, bin_number=45, max_points=max_points)
            out = engine.guided_match(*args, bin_number=45, max_points=max_points)
            assert len(ref["matches"]) > 50, (s, d)
            assert out["prepared"].tobytes() == ref["prepared"].tobytes(), (s, d)
            assert np.array_equal(out["matches"], ref["matches"]), (s, d)
            assert out["ratios"].tobytes() == ref["ratios"].tobytes(), (s, d)
            sel = [(int(a), int(b), float(r)) for (a, b), r in zip(ref["selected_matches"], ref["selected_ratios"])]
            assert out["selected"] == sel, (s, d, max_points)
            assert eng.guided_match_views(s, d, qt, 45, max_points) == sel, (s, d, max_points)
            cut += len(ref["matches"]) > max_points
    assert cut > 0
    eng.close()


def test_builder_waves_commit_what_the_oracle_commits(cam_scene, oracle):
    pgb, ostats = run_and_compare(oracle, cam_scene, prefetch_fallback=True, wave_size=16)
    assert ostats["edges"] >= 20 and ostats["rejected"] > 0


def test_builder_hashing_mode_commits_what_the_oracle_commits(cam_scene, oracle):
    sc = dict(cam_scene)
    pgb = B.PoseGraphBuilder(kUseEpipolarHashing_=True, kSimilarityThreshold_=0.0, scene=sc)
    g = pgb.run()
    st = pgb.hashing_stats
    assert g.numEdges() >= 20 and st["quick_matched"] > 0 and st["guided_calls"] > 0
    _compare_with_oracle(oracle, sc, pgb, True)
    pgb.close()
