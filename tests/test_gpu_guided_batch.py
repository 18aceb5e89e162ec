"""Batched guided matching (K10, pgi_guided_match_pairs / Engine.guided_match_pairs / PoseGraphBuilder.guided_match_edges),
bit for bit: every pair of a batch against the oracle's guided matcher and the single-pair calls (guided_match_views and
guided_match), on
descriptor scenes (128-D and 64-D), per-view cameras, degenerate epipolar geometry and bin numbers; a pair's rows do not
depend on its batch, across scratch chunks too; the builder's edges after a wave-mode and a hashing-mode run; errors."""
import ctypes as C

import numpy as np
import pytest

from helpers import intrinsics, per_view_camera_scene, perturbed_pose, pose_qt, rodrigues, two_view_keypoints_posed
from test_gpu_cameras import _guided_cases as _camera_cases
from test_gpu_hashing import _guided_cases
from test_hashing_host import hashing_scene
from test_matcher_reference import K_DST, K_SRC, R_GEN, SIZE_DST, SIZE_SRC, T_GEN, lateral_case
from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import WAVE_PATH, Engine, PgiError, _ptr

pytestmark = pytest.mark.gpu


def _views(sc):
    ko = sc["kp_offset"].astype(np.int64)
    return ([sc["kp"][ko[v]:ko[v + 1]] for v in range(len(ko) - 1)], [sc["desc"][ko[v]:ko[v + 1]] for v in range(len(ko) - 1)])


def _args(sc, kp, desc, s, d, qt):
    Ks, Kd = intrinsics(sc["focal"][s], sc["size"][s]), intrinsics(sc["focal"][d], sc["size"][d])
    return (kp[s], desc[s], kp[d], desc[d], qt, Ks, Kd, sc["size"][s], sc["size"][d])


def _batch(eng, cases, max_points, bin_number=45):
    pv = np.array([(s, d) for s, d, _ in cases], dtype=np.uint32).reshape(-1, 2)
    poses = np.array([qt for _, _, qt in cases]).reshape(-1, 7)
    off, m, v = eng.guided_match_pairs(pv, poses, bin_number, max_points)
    assert len(off) == len(cases) + 1 and off[0] == 0 and int(off[-1]) == len(m) == len(v)
    return [(m[int(off[k]):int(off[k + 1])], v[int(off[k]):int(off[k + 1])]) for k in range(len(cases))]


def _rows(sel):
    """[(src, dst, value)] -> (matches [n, 2] u32, values [n] f64)"""
    return (np.array([(a, b) for a, b, _ in sel], dtype=np.uint32).reshape(-1, 2), np.array([r for _, _, r in sel], dtype=np.float64))


def _same(got, matches, values):
    m, v = got
    return np.array_equal(m, np.asarray(matches, dtype=np.uint32).reshape(-1, 2)) and v.tobytes() == np.asarray(values, np.float64).tobytes()


def _check_against_oracle(eng, sc, cases, oracle, engine=None, max_points_list=(100, 10, 3, 0), bin_number=45):
    """Every pair of one batch per max_points equals the oracle and the single-pair calls; returns the set of (more than
    max_points?) seen."""
    kp, desc = _views(sc)
    regimes = set()
    for mp in max_points_list:
        got = _batch(eng, cases, mp, bin_number)
        for k, (s, d, qt) in enumerate(cases):
            args = _args(sc, kp, desc, s, d, qt)
            ref = oracle.guided_match(*args, bin_number=bin_number, max_points=mp if mp else 10 ** 9)
            if mp:
                assert _same(got[k], ref["selected_matches"], ref["selected_ratios"]), (k, s, d, mp)
                assert _same(got[k], *_rows(eng.guided_match_views(s, d, qt, bin_number, mp))), (k, s, d, mp)
                regimes.add(len(ref["matches"]) > mp)
            else:
                assert _same(got[k], ref["matches"], ref["ratios"]), (k, s, d)
                if engine is not None:
                    single = engine.guided_match(*args, bin_number=bin_number, max_points=10 ** 9)
                    assert _same(got[k], single["matches"], single["ratios"]), (k, s, d)
    return regimes


def _descriptor_scene(dim):
    if dim == 128:  # test_gpu_hashing's desc_scene: view 3 has no keypoint, view 7 has one
        counts = np.random.default_rng(11).integers(700, 1600, 12)
        counts[3], counts[7] = 0, 1
        return S.make_descriptor_scene(n_views=12, kp_counts=counts, dim=128, seed=11, arc=np.pi, visible_half_angle=0.6 * np.pi)
    counts = np.random.default_rng(12).integers(300, 1200, 10)  # test_gpu_hashing's 64-D scene: view 2 has one keypoint
    counts[2] = 1
    return S.make_descriptor_scene(n_views=10, kp_counts=counts, dim=64, seed=12, arc=np.pi, visible_half_angle=0.6 * np.pi)


@pytest.fixture(scope="module")
def scenes():
    out = {}
    for dim in (128, 64):
        sc = _descriptor_scene(dim)
        eng = Engine(device=0)
        eng.register_scene_descriptors(sc, 0.4)
        out[dim] = (sc, eng)
    yield out
    for _, eng in out.values():
        eng.close()


# ---- 1. descriptor scenes ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [128, 64])
def test_batches_equal_the_oracle_and_single_pair_calls(scenes, engine, oracle, dim):
    sc, eng = scenes[dim]
    cases = _guided_cases(sc, np.random.default_rng(dim), 50)  # ground truth and perturbed poses, both directions, empty views
    cases += cases[:6]  # repeated pairs
    assert len(cases) >= 60
    regimes = _check_against_oracle(eng, sc, cases, oracle, engine)
    assert regimes == {True, False}


# ---- 2. per-view cameras -------------------------------------------------------------------------------------------------
def test_per_view_cameras_equal_the_oracle(oracle, engine):
    sc = per_view_camera_scene(n_views=12, seed=1, with_matches=True)
    eng = Engine(device=0)
    eng.register_scene(sc, 0.4)
    eng.set_scene_descriptors(sc["desc"])
    cases = _camera_cases(sc)
    assert len(cases) >= 8
    _check_against_oracle(eng, sc, cases, oracle, engine, max_points_list=(100, 0))
    eng.close()


# ---- 3. degenerate geometry on a registered scene ------------------------------------------------------------------------
def _two_view_engine(args):
    kp_s, d_s, kp_d, d_d, qt, K_s, K_d, size_s, size_d = args
    for K, size in ((K_s, size_s), (K_d, size_d)):
        assert np.array_equal(K, intrinsics(K[0, 0], size))  # what a registered view's camera is
    sc = dict(focal=np.array([K_s[0, 0], K_d[0, 0]]), size=np.array([size_s, size_d], dtype=np.float64),
              kp_offset=np.array([0, len(kp_s), len(kp_s) + len(kp_d)], dtype=np.uint64), kp=np.vstack([kp_s, kp_d]),
              desc=np.vstack([d_s, d_d]), pair_views=np.array([[0, 1]], dtype=np.uint32), m_offset=np.zeros(2, dtype=np.uint64),
              matches=np.zeros((0, 2), dtype=np.uint32))
    eng = Engine(device=0)
    eng.register_scene(sc, 0.4)
    eng.set_scene_descriptors(sc["desc"])
    return sc, eng


def _epipole_pose(ex, ey):
    C_ = np.linalg.inv(K_SRC) @ np.array([ex, ey, 1.0])
    return np.eye(3), -C_


def _posed(R, t, seed):
    d = two_view_keypoints_posed(1500, np.random.default_rng(seed), R, t, K_SRC, K_DST, SIZE_SRC, SIZE_DST, desc_noise=0.02)
    return (d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], d["pose"], K_SRC, K_DST, SIZE_SRC, SIZE_DST)


W, H = SIZE_SRC
DEGENERATE = {
    "lateral_x_y1e-7": lambda: lateral_case("x_y1e-7"),
    "lateral_x": lambda: lateral_case("x"),
    "epipole_inside": lambda: _posed(*_epipole_pose(0.5, H / 2.0), 3),
    "epipole_outside": lambda: _posed(*_epipole_pose(-0.5, H / 2.0), 3),
    "generic": lambda: _posed(R_GEN, T_GEN, 1),
}


@pytest.mark.parametrize("name,bins", [(n, 45) for n in DEGENERATE] + [("generic", 1), ("generic", 192), ("generic", 0)])
def test_degenerate_geometry_and_bin_numbers(oracle, engine, name, bins):
    args = DEGENERATE[name]()
    sc, eng = _two_view_engine(args)
    qt = args[4]
    R = rodrigues(np.array([1e-3, 0.0, 0.0]))
    cases = [(0, 1, qt), (0, 1, qt), (0, 1, perturbed_pose(R, qt[4:], np.random.default_rng(0), 1e-4, 1e-4))]
    _check_against_oracle(eng, sc, cases, oracle, engine, max_points_list=(100, 0), bin_number=bins)
    ref = oracle.guided_match(*args, bin_number=bins, max_points=100)
    assert len(ref["matches"]) > 50
    if name == "lateral_x_y1e-7":
        assert ref["prepared"][12] == 0.0  # the angular range is 0: every keypoint is in bin 0
    if name.startswith("epipole"):
        assert (ref["prepared"][12] == -180.0) == (name == "epipole_inside")
    eng.close()


# ---- 4. batch independence -----------------------------------------------------------------------------------------------
def test_rows_do_not_depend_on_the_batch(scenes):
    sc, eng = scenes[128]
    cases = _guided_cases(sc, np.random.default_rng(3), 20)
    for mp in (100, 0):
        full = _batch(eng, cases, mp)
        perm = np.random.default_rng(4).permutation(len(cases))
        permuted = _batch(eng, [cases[i] for i in perm], mp)
        repeated = _batch(eng, cases * 3, mp)
        for k in range(len(cases)):
            assert _same(permuted[int(np.nonzero(perm == k)[0][0])], *full[k])
            for r in range(3):
                assert _same(repeated[r * len(cases) + k], *full[k])
        for k in range(0, len(cases), 5):
            assert _same(_batch(eng, [cases[k]], mp)[0], *full[k])


def test_a_batch_over_several_scratch_chunks(engine, oracle):
    d = two_view_keypoints_posed(12800, np.random.default_rng(2), R_GEN, T_GEN, K_SRC, K_DST, SIZE_SRC, SIZE_DST, desc_noise=0.02)
    args = (d["kp_src"][:16384], d["desc_src"][:16384], d["kp_dst"][:16384], d["desc_dst"][:16384], d["pose"], K_SRC, K_DST,
            SIZE_SRC, SIZE_DST)
    assert len(args[0]) == 16384 and len(args[2]) == 16384
    sc, eng = _two_view_engine(args)
    qt = args[4]
    alone = _batch(eng, [(0, 1, qt)], 100)[0]
    ref = oracle.guided_match(*args, bin_number=45, max_points=100)
    assert len(ref["matches"]) > 1000 and _same(alone, ref["selected_matches"], ref["selected_ratios"])
    # 16 384 keypoints on both sides: about 0.6 MB of scratch per pair, so 1 000 pairs need two 512 MB chunks
    n = 1000
    c0 = eng.stats()["guided_chunks"]
    rows = _batch(eng, [(0, 1, qt)] * n, 100)
    assert eng.stats()["guided_chunks"] - c0 >= 2
    for r in rows:
        assert _same(r, *alone)
    every = oracle.guided_match(*args, max_points=10 ** 9)
    assert _same(_batch(eng, [(0, 1, qt)] * 3, 0)[2], every["matches"], every["ratios"])
    eng.close()


# ---- 5. builder ----------------------------------------------------------------------------------------------------------
def _check_edges(pgb, graph, oracle, max_points=None):
    sc = pgb.scene
    kp, desc = _views(sc)
    off, m, v = pgb.guided_match_edges(max_points=max_points)
    if max_points is None:
        max_points = pgb.max_points_hashing
    e = graph.edges
    assert len(off) == len(e) + 1 and len(e) > 0
    for k in range(len(e)):
        s, d = int(e["src"][k]), int(e["dst"][k])
        qt = np.concatenate([e["q"][k], e["t"][k]])
        ref = oracle.guided_match(*_args(sc, kp, desc, s, d, qt), max_points=max_points if max_points else 10 ** 9)
        got = (m[int(off[k]):int(off[k + 1])], v[int(off[k]):int(off[k + 1])])
        if max_points:
            assert _same(got, ref["selected_matches"], ref["selected_ratios"]), k
        else:
            assert _same(got, ref["matches"], ref["ratios"]), k
    return off


def test_builder_wave_mode(oracle):
    sc = S.make_descriptor_scene(n_views=16, kp_range=(500, 900), dim=64, seed=7, arc=np.pi, visible_half_angle=0.6 * np.pi)
    pgb = B.PoseGraphBuilder(kSimilarityThreshold_=0.0, scene=sc)
    g = pgb.run()
    assert g.numEdges() >= 10
    _check_edges(pgb, g, oracle)
    _check_edges(pgb, g, oracle, 0)
    st = pgb.engine.stats()
    assert st["guided_pairs"] == 2 * g.numEdges() and st["guided_dist_evals"] > 0 and st["ms_guided_pairs"] > 0
    pgb.close()


def test_builder_hashing_mode_rows_equal_the_loop(oracle):
    sc = hashing_scene(12, 3)  # desc and matches: the descriptors went to the device in prepare()
    pgb = B.PoseGraphBuilder(kUseEpipolarHashing_=True, kSimilarityThreshold_=0.0, scene=sc)
    g = pgb.run()
    off = _check_edges(pgb, g, oracle)
    _check_edges(pgb, g, oracle, 0)
    committed = pgb.log["committed"] > 0
    src = pgb.match_sources
    quick = src["source"][committed] == B.MATCH_QUICK
    assert quick.sum() > 0
    counts = np.diff(off.astype(np.int64))
    assert np.array_equal(counts[quick], src["guided_rows"][committed][quick].astype(np.int64))
    pgb.close()


# ---- 6. errors and state -------------------------------------------------------------------------------------------------
def test_errors_empty_batch_and_statistics(scenes):
    sc, eng = scenes[64]
    qt = np.array([[0, 0, 0, 1.0, 1, 0, 0]])
    e = Engine(device=0)
    with pytest.raises(PgiError, match="status -4"):  # no scene
        e.guided_match_pairs([[0, 1]], qt)
    nodesc = {k: sc[k] for k in ("focal", "size", "kp_offset", "kp", "pair_views", "m_offset", "matches")}
    e.register_scene(nodesc, 0.4)
    with pytest.raises(PgiError, match="status -4"):  # no descriptors
        e.guided_match_pairs([[0, 1]], qt)
    e.set_scene_descriptors(sc["desc"])
    ids = np.arange(2, dtype=np.uint32)
    e.submit_wave(ids, flags=WAVE_PATH)
    with pytest.raises(PgiError, match="status -4"):  # a wave in flight
        e.guided_match_pairs([[0, 1]], qt)
    e.wait_wave()
    V = len(sc["focal"])
    for call in (lambda: e.guided_match_pairs([[0, V]], qt), lambda: e.guided_match_pairs([[V, 0]], qt),
                 lambda: e.guided_match_pairs([[0, 1]], qt, bin_number=193)):
        with pytest.raises(PgiError, match="status -1"):
            call()
    lib, h = e.lib, e.h
    pv = np.array([[0, 1]], dtype=np.uint32)
    off = np.zeros(2, dtype=np.uint64)
    m = np.zeros((100, 2), dtype=np.uint32)
    v = np.zeros(100)
    n0 = int(sc["kp_offset"][1] - sc["kp_offset"][0])
    assert n0 > 20
    call = lambda cap, *ptrs: lib.pgi_guided_match_pairs(h, C.c_uint64(1), *ptrs[:2], C.c_int32(45), C.c_uint32(20), *ptrs[2:],
                                                          C.c_uint64(cap))
    good = (_ptr(pv), _ptr(qt), _ptr(off), _ptr(m), _ptr(v))
    assert call(19, *good) == -1  # capacity below min(n_src, max_points)
    for k in range(5):
        bad = list(good)
        bad[k] = None
        assert call(100, *bad) == -1, k
    assert call(20, *good) == 0 and int(off[1]) <= 20
    st0 = e.stats()
    o, mm, vv = e.guided_match_pairs(np.zeros((0, 2)), np.zeros((0, 7)))
    assert o.tolist() == [0] and len(mm) == 0 and len(vv) == 0
    cases = [(0, 1, qt[0]), (1, 0, qt[0]), (2, 3, qt[0])]
    _batch(e, cases, 100)
    st1 = e.stats()
    assert st1["guided_pairs"] - st0["guided_pairs"] == 3 and st1["guided_chunks"] - st0["guided_chunks"] == 1
    assert st1["ms_guided_pairs"] > st0["ms_guided_pairs"]
    e.close()
