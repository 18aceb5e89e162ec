"""The pose path (K1, K2, K4a/b/c + K5, K3) on inputs the two_view / make_scene generators never produce, on every launch
form a wave can select, against the oracle:
- one set of regime pairs (tests/helpers.py: wide field of view, off-centre, forward motion, pure rotation, tiny
  baseline, planar, duplicated and identical rows, outlier ratios 0..1, non-finite rows, focal-0 rows with an infinite
  threshold, at the kernels' size edges, thresholds across three decades), fallback termination-edge pairs, the crafted
  pair of K2's "first finite solution" rule and two_view filler pairs, run in waves of 1 pair, 100 pairs with masks, 600
  pairs, and all 4 200 pairs with and without masks.  That covers the direct and streaming K1, K2's warp-per-pair and
  64-pairs-per-CTA forms, K3 with 8, 6, 2 and 1 CTAs per pair, and K5's FP32-staged path next to its FP64-only path
  (pairs over 11 264 rows).  A verdict is a pure function of (pair, hypotheses), so every form must write the same bytes;
- K1's threshold tests with the threshold a few ulps from a row's residual, and at its epipoles;
- pgi_test_pose at negative, zero, NaN, infinite, subnormal and huge thresholds;
- scene registrations with extreme cameras and with a focal length of 0."""
import concurrent.futures as cf
import os

import numpy as np
import pytest
import torch

from helpers import (first_finite_pair, per_view_camera_scene, perturbed_pose, pose_qt, regime_set, rodrigues,
                     termination_pairs, two_view)
from pose_graph_initialization_b200.engine import WAVE_FALLBACK, WAVE_NO_TEST, WAVE_PATH

pytestmark = pytest.mark.gpu
FILLER_THR = 0.4 / 800.0
N_PAIRS = 4200  # > 4 096: K2's 64-pairs-per-CTA form; a multiple of 100 and 600, so those waves are all full


def _pool_map(fn, items):
    with cf.ThreadPoolExecutor(max(1, os.cpu_count() or 1)) as ex:  # the oracle's ctypes calls release the GIL
        return list(ex.map(fn, items))


def _expect(oracle, corr, thr, hyps):
    """The wave's verdict of one pair by the oracle: the in-traversal test per hypothesis (the last one sets test_count,
    the passing ones are estimatePose's guesses), estimatePose, and the fallback's own run for its iteration count."""
    guesses, count = [], 0
    for h in hyps:
        ok, count = oracle.test_pose(corr, h, 1.5 * thr, 5)
        if ok:
            guesses.append(h)
    o = oracle.estimate_pose(corr, thr, guesses)
    fb = oracle.fallback(corr, thr) if o["branch"] != 1 else None
    return dict(o=o, test_passed=bool(guesses), test_count=count, fb=fb)


def _check(v, mask, e, what):
    o = e["o"]
    assert bool(v["test_passed"]) == e["test_passed"] and int(v["test_count"]) == e["test_count"], what
    assert int(v["path_inliers"]) == o["path_inliers"], what
    assert bool(v["accepted"]) == o["success"] and int(v["branch"]) == o["branch"], what
    assert int(v["inlier_count"]) == o["inlier_number"], what
    if o["success"]:
        assert v["E"].reshape(3, 3).tobytes() == o["E"].tobytes(), what
        assert np.concatenate([v["q"], v["t"]]).tobytes() == o["pose"].tobytes(), what
    assert int(v["status"]) & 1 == (e["fb"] is not None), what
    assert int(v["iters"]) == (e["fb"]["iterations"] if e["fb"] else 0), what
    assert np.array_equal(mask, o["mask"]), what


@pytest.fixture(scope="module")
def pose_set(oracle):
    special = [(lab, c, thr, h) for lab, c, thr, h in regime_set()]
    special += [(f"term-{lab}", c, thr, []) for lab, _, c, thr in termination_pairs()]
    c, thr, hyp, _ = first_finite_pair()
    special.append(("first-finite", c, thr, [hyp]))
    rng = np.random.default_rng(606)
    filler = []
    for i in range(N_PAIRS - len(special)):
        c, R, t = two_view(int(rng.integers(40, 121)), 0.3, rng)
        h = [] if i % 3 == 0 else [perturbed_pose(R, t, rng) if i % 3 == 1 else pose_qt(np.eye(3), np.array([1.0, 0.0, 0.0]))]
        filler.append((f"filler-{i}", c, FILLER_THR, h))
    pairs = special + filler
    order = np.random.default_rng(7).permutation(len(pairs))  # spread the special pairs over every wave
    pairs = [pairs[k] for k in order]
    is_special = np.array([not lab.startswith("filler") for lab, *_ in pairs])
    sizes = np.array([len(c) for _, c, _, _ in pairs])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    # expectations: estimatePose per special pair; the batch oracle for the filler (one guess: the hypothesis if it passes)
    exp = {}
    sp = np.flatnonzero(is_special)
    for k, e in zip(sp, _pool_map(lambda k: _expect(oracle, pairs[k][1], pairs[k][2], pairs[k][3]), sp)):
        exp[int(k)] = e
    fl = np.flatnonzero(~is_special)
    guess, has = np.zeros((len(fl), 7)), np.zeros(len(fl), dtype=np.uint8)
    tests = {}
    for j, k in enumerate(fl):
        _, c, thr, h = pairs[k]
        if h:
            tests[int(k)] = oracle.test_pose(c, h[0], 1.5 * thr, 5)
            if tests[int(k)][0]:
                guess[j], has[j] = h[0], 1
    fc = np.vstack([pairs[k][1] for k in fl])
    fo = np.concatenate([[0], np.cumsum(sizes[fl])])
    batch = oracle.estimate_pose_batch(fc, fo, np.array([pairs[k][2] for k in fl]), guess, has)
    ran = [int(k) for j, k in enumerate(fl) if batch["info"][j, 1] != 1]
    fbs = dict(zip(ran, _pool_map(lambda k: oracle.fallback(pairs[k][1], pairs[k][2]), ran)))
    fb_models = np.zeros(len(pairs), dtype=np.int64)  # models + LO refits of each pair's fallback (0 if it did not run)
    for k, e in exp.items():
        if e["fb"]:
            fb_models[k] = e["fb"]["models"] + e["fb"]["lo_runs"]
    for k, r in fbs.items():
        fb_models[k] = r["models"] + r["lo_runs"]
    return dict(pairs=pairs, off=off, exp=exp, filler=dict(ids=fl, batch=batch, tests=tests, fbs=fbs), fb_models=fb_models,
                is_special=is_special)


def _wave(engine, pairs, ids, masks):
    ids = np.asarray(ids, dtype=np.uint32)
    hs = [pairs[k][3] for k in ids]
    hoff = np.concatenate([[0], np.cumsum([len(h) for h in hs])]).astype(np.uint32)
    hyp = np.array([x for h in hs for x in h]).reshape(-1, 7)
    engine.reset_stats()
    res = engine.run_wave(ids, hoff, hyp, flags=WAVE_PATH | WAVE_FALLBACK, want_masks=masks)
    return res, engine.stats()["fallback_models"]


def test_every_launch_form_writes_the_oracle_verdict(engine, oracle, pose_set):
    pairs, off, fbm = pose_set["pairs"], pose_set["off"], pose_set["fb_models"]
    n = len(pairs)
    assert n == N_PAIRS and n > 4096 and n >= 2 * torch.cuda.get_device_properties(0).multi_processor_count
    assert max(len(c) for _, c, _, _ in pairs) > 11264 and any(1000 < len(c) <= 11264 for _, c, _, _ in pairs)
    engine.register_pairs(np.vstack([c for _, c, _, _ in pairs]), off, np.array([thr for _, _, thr, _ in pairs]))
    all_ids = np.arange(n)
    ref, models = _wave(engine, pairs, all_ids, False)  # streaming K1, K2 64 pairs per CTA, K3 one CTA per pair
    # statistic: K5 counts every model it scores, minimal and LO refit alike -> the oracle's models + lo_runs
    assert models == int(fbm.sum())
    ref_m, masks = None, None
    (ref_m, masks), models = _wave(engine, pairs, all_ids, True)  # the same with the direct K1
    assert models == int(fbm.sum())
    assert ref_m.tobytes() == ref.tobytes()
    mask_of = {k: masks[int(off[k]):int(off[k + 1])] for k in range(n)}
    # every regime and termination pair against estimatePose, the fallback's iteration count included
    for k, e in pose_set["exp"].items():
        _check(ref[k], mask_of[k], e, pairs[k][0])
    # the filler against the batch oracle
    fl, batch = pose_set["filler"]["ids"], pose_set["filler"]["batch"]
    for j, k in enumerate(fl):
        v, info = ref[k], batch["info"][j]
        if k in pose_set["filler"]["tests"]:
            ok, cnt = pose_set["filler"]["tests"][k]
            assert bool(v["test_passed"]) == ok and int(v["test_count"]) == cnt, pairs[k][0]
        assert bool(v["accepted"]) == bool(info[0]) and int(v["branch"]) == info[1] and int(v["inlier_count"]) == info[2], pairs[k][0]
        assert int(v["path_inliers"]) == info[3], pairs[k][0]
        if info[0]:
            assert v["E"].tobytes() == batch["E"][j].tobytes(), pairs[k][0]
            assert np.concatenate([v["q"], v["t"]]).tobytes() == batch["pose"][j].tobytes(), pairs[k][0]
        fb = pose_set["filler"]["fbs"].get(int(k))
        assert int(v["iters"]) == (fb["iterations"] if fb else 0), pairs[k][0]
    # the same bytes from every other form
    forms = [("100 pairs with masks", [all_ids[i:i + 100] for i in range(0, n, 100)], True),
             ("600 pairs", [all_ids[i:i + 600] for i in range(0, n, 600)], False),
             ("1 pair", [[k] for k in all_ids if pose_set["is_special"][k] or k % 50 == 0], True)]
    for name, waves, want_masks in forms:
        for ids in waves:
            res, models = _wave(engine, pairs, ids, want_masks)
            assert models == int(fbm[ids].sum()), name
            out, m = res if want_masks else (res, None)
            row = 0
            for i, k in enumerate(ids):
                assert out[i].tobytes() == ref[k].tobytes(), (name, pairs[k][0])
                if want_masks:
                    nk = int(off[k + 1] - off[k])
                    assert np.array_equal(m[row:row + nk], mask_of[k]), (name, pairs[k][0])
                    row += nk
    # the comparisons above are about real work on every branch
    assert ref["accepted"].sum() > 1000 and (ref["branch"] == 1).sum() > 100 and (ref["status"] & 1).sum() > 1000
    assert {int(ref[k]["iters"]) for k in pose_set["exp"]} >= {1, 16, 17, 32, 33, 124, 125, 126, 251, 1000}


# ---- K1's threshold certificate ---------------------------------------------------------------------------------------
def _ulps(q, s):
    return np.asarray(q, dtype=np.float64).view(np.int64) - np.float64(s).view(np.int64)


def _boundary_cases(oracle):
    """[(corr, thr)] pairs of 5 copies of one row whose threshold puts fl(1.5 thr)^2 (the test's) or fl(1.5 thr) (getInliers'
    un-squared one) exactly on the row's squared Sampson residual, at +-1, +-2, +-4 ulps of it, and at (1 +- 2^-51),
    (1 +- 2^-50), (1 +- 2^-49) times it; plus rows at and near both epipoles of a forward motion and rows with r = 0."""
    rng = np.random.default_rng(91)
    c, R, t = two_view(96, 0.5, rng)
    pose = perturbed_pose(R, t, rng, 1e-3, 1e-3)
    E = oracle.essential_from_pose(pose)
    s = oracle.sampson_sq(c, E)
    cases = []
    for kind, scale in (("test", lambda x: (1.5 * x) * (1.5 * x)), ("inliers", lambda x: 1.5 * x)):
        ulp_hits = {u: [] for u in (0, 1, -1, 2, -2, 4, -4)}
        rel_hits = {d: [] for d in (2.0 ** -51, -2.0 ** -51, 2.0 ** -50, -2.0 ** -50, 2.0 ** -49, -2.0 ** -49)}
        for k in np.flatnonzero(np.isfinite(s) & (s > 1e-12)):
            g = np.sqrt(s[k]) / 1.5 if kind == "test" else s[k] / 1.5
            cand = (np.float64(g).view(np.int64) + np.arange(-64, 65)).view(np.float64)
            q = scale(cand)
            off = _ulps(q, s[k])
            for u, lst in ulp_hits.items():
                hit = np.flatnonzero(off == u)
                if len(hit) and len(lst) < 8:
                    lst.append((k, cand[hit[0]]))
            rel = (q - s[k]) / s[k]  # exact: q and s[k] are within a few ulps (Sterbenz), one rounding in the quotient
            for d, lst in rel_hits.items():
                j = int(np.argmin(np.abs(rel - d)))
                if abs(rel[j] - d) <= 2.0 ** -54 and len(lst) < 8:
                    lst.append((k, cand[j]))
        for hits in (ulp_hits, rel_hits):
            for key, lst in hits.items():
                assert len(lst) >= 4, (kind, key)
                for k, thr in lst:
                    q = scale(np.float64(thr))
                    if hits is ulp_hits:
                        assert _ulps(q, s[k]) == key
                    else:
                        assert abs((q - s[k]) / s[k] - key) <= 2.0 ** -54
                    cases.append((np.repeat(c[k:k + 1], 5, 0), float(thr), pose))
    # forward motion along z: E = [e_z]x, epipoles at the origin of both images; r = x1 y2 - y1 x2
    fwd = pose_qt(np.eye(3), np.array([0.0, 0.0, 1.0]))
    rows = []
    for d in (0.0, 1e-146, 1e-150, 1e-155, 1e-160, 1e-162, 1e-300):
        rows += [[d, 0.0, 0.0, d], [d, d, d, d], [d, 0.0, 0.0, 1.0], [0.0, 0.0, d, -d]]
    rows += [[0.3, -0.2, 0.3, -0.2], [1.5, 2.5, 1.5, 2.5]]  # x2 = x1: r = 0 exactly, den > 0
    for r in rows:
        for thr in (1e-5, 1e-3, 1.0):
            cases.append((np.repeat(np.array([r], dtype=np.float64), 5, 0), thr, fwd))
    return cases


def test_k1_threshold_boundary_on_both_k1_forms(engine, oracle):
    cases = _boundary_cases(oracle)
    n = len(cases)
    assert n >= 2 * torch.cuda.get_device_properties(0).multi_processor_count  # the wave without masks streams
    corr = np.vstack([c for c, _, _ in cases])
    off = np.arange(n + 1, dtype=np.uint64) * 5
    engine.register_pairs(corr, off, np.array([thr for _, thr, _ in cases]))
    hoff = np.arange(n + 1, dtype=np.uint32)
    hyp = np.array([p for _, _, p in cases])
    for gate in (0, WAVE_NO_TEST):
        streamed = engine.run_wave(np.arange(n), hoff, hyp, flags=WAVE_PATH | gate)
        direct, masks = engine.run_wave(np.arange(n), hoff, hyp, flags=WAVE_PATH | gate, want_masks=True)
        assert streamed.tobytes() == direct.tobytes()
        for k, (c, thr, p) in enumerate(cases):
            ok, cnt = oracle.test_pose(c, p, 1.5 * thr, 5)
            inl = oracle.get_inliers(c, oracle.essential_from_pose(p), 1.5 * thr)
            passed = ok or gate != 0
            want = np.zeros(5, dtype=np.uint8)
            if passed:
                want[inl.astype(np.int64)] = 1
            v = direct[k]
            assert bool(v["test_passed"]) == passed and int(v["test_count"]) == cnt, (k, thr, c[0])
            assert int(v["path_inliers"]) == (len(inl) if passed else 0), (k, thr, c[0])
            assert np.array_equal(masks[5 * k:5 * k + 5], want), (k, thr, c[0])


def test_test_pose_uses_the_threshold_it_is_given(engine, oracle):
    """pgi_test_pose counts sres < thr^2 for every thr, as InTraversalPoseTester does; a negative thr is not replaced by
    the pair's 1.5 x thr_norm."""
    rng = np.random.default_rng(95)
    c, R, t = two_view(400, 0.3, rng)
    c = np.vstack([c, [[0.0, 0.0, 0.0, 0.0], [1e-160, 0.0, 0.0, 1e-160]]])
    pose = perturbed_pose(R, t, rng)
    every = len(c) + 1  # a minimum no pair reaches: the count of every inlier
    assert oracle.test_pose(c, pose, -1e-3, every)[1] != oracle.test_pose(c, pose, 1.5e-3, every)[1]
    for thr in (-1e-3, -0.0, 0.0, np.nan, np.inf, 1e-310, 1e200, 1e-3):
        for m in (5, every):
            assert engine.test_pose(c, thr, pose, m) == oracle.test_pose(c, pose, thr, m), (thr, m)


# ---- scenes -----------------------------------------------------------------------------------------------------------
# focal lengths down to a quarter of the image width; views 0-1 (640 x 480) and 2-3 (2 560 x 1 920, 4x the width) pair up
EXTREME_CAMERAS = ((160.0, (640, 480)), (640.0, (2560, 1920)), (400.0, (1600, 1200)), (2400.0, (1200, 1600)))


def _scene_tuples(sc, rng):
    P = len(sc["pair_views"])
    hyp, has = np.zeros((P, 7)), np.zeros(P, dtype=np.uint8)
    for p, (s, d) in enumerate(sc["pair_views"]):
        if p % 3 == 2:
            continue
        R = sc["gt_R"][d] @ sc["gt_R"][s].T
        t = sc["gt_t"][d] - R @ sc["gt_t"][s]
        hyp[p] = perturbed_pose(R, t / np.linalg.norm(t), rng) if p % 3 == 0 else pose_qt(rodrigues(np.array([0.0, 0.5, 0.0])), np.array([1.0, 0, 0]))
        has[p] = 1
    return hyp, has


@pytest.mark.parametrize("focal_zero", [False, True])
def test_extreme_camera_scenes_match_the_scene_pipeline(engine, oracle, focal_zero):
    sc = per_view_camera_scene(n_views=8, seed=5, cameras=EXTREME_CAMERAS, group=2, n_points=1200, kp_max=700, with_matches=True)
    assert (sc["focal"] / sc["size"][:, 0]).min() == 0.25 and (sc["size"][:, 0].max() / sc["size"][:, 0].min()) == 4
    if focal_zero:
        sc["focal"] = sc["focal"].copy()
        sc["focal"][3] = 0.0  # a list line without a focal length
    hyp, has = _scene_tuples(sc, np.random.default_rng(8))
    P = len(sc["pair_views"])
    ids = np.arange(P, dtype=np.uint32)
    o = oracle.scene_pipeline_batch(sc, ids, hyp, has, thr_px=0.4)
    engine.register_scene(sc, 0.4)
    hoff = np.concatenate([[0], np.cumsum(has)]).astype(np.uint32)
    out = engine.run_wave(ids, hoff, hyp[has > 0])
    for p in range(P):
        v, info = out[p], o["info"][p]
        what = (p, tuple(sc["pair_views"][p]))
        assert bool(v["test_passed"]) == bool(o["test_passed"][p]) and int(v["test_count"]) == int(o["test_count"][p]), what
        assert bool(v["accepted"]) == bool(info[0]) and int(v["branch"]) == info[1] and int(v["inlier_count"]) == info[2], what
        assert int(v["path_inliers"]) == info[3], what
        if info[0]:
            assert v["E"].tobytes() == o["E"][p].tobytes(), what
            assert np.concatenate([v["q"], v["t"]]).tobytes() == o["pose"][p].tobytes(), what
    assert out["accepted"].sum() >= P // 4
    if focal_zero:
        zero = [p for p, (s, d) in enumerate(sc["pair_views"]) if s == 3]
        assert zero and all(engine.read_pair(p)[1] == np.inf for p in zero)
