"""Edge cases of the C-ABI path on the GPU: ragged and degenerate pair sizes, pairs too large for the shared-memory
staging of K5 (exact FP64 path), several guesses per pair (pose_graph_builder.h:974-1029 semantics), error codes."""
import ctypes as C

import numpy as np
import pytest

from helpers import perturbed_pose, pose_qt, two_view
from pose_graph_initialization_b200.engine import PgiError, VERDICT_DTYPE, WAVE_FALLBACK, WAVE_PATH

pytestmark = pytest.mark.gpu
THR = 0.4 / 800.0


def _check(v, mask, corr, o):
    assert bool(v["accepted"]) == o["success"] and int(v["branch"]) == o["branch"]
    assert int(v["inlier_count"]) == o["inlier_number"]
    if o["success"]:
        assert np.array_equal(v["E"].reshape(3, 3), o["E"])
        assert np.array_equal(np.concatenate([v["q"], v["t"]]), o["pose"])
    assert np.array_equal(mask, o["mask"])


def test_ragged_wave_with_tiny_and_empty_pairs(engine, oracle):
    rng = np.random.default_rng(31)
    sizes = [0, 1, 4, 5, 6, 19, 20, 21, 33, 257, 1000]
    pairs = [two_view(n, 0.2, rng)[0] if n else np.zeros((0, 4)) for n in sizes]
    off = np.concatenate([[0], np.cumsum(sizes)])
    engine.register_pairs(np.vstack(pairs), off, [THR] * len(sizes))
    out, masks = engine.run_wave(np.arange(len(sizes)), None, None, flags=WAVE_FALLBACK, want_masks=True)
    for k, n in enumerate(sizes):
        o = oracle.estimate_pose(pairs[k], THR, []) if n else dict(success=False, branch=0, inlier_number=0, mask=np.zeros(0, np.uint8))
        _check(out[k], masks[off[k]:off[k + 1]], pairs[k], o)
        assert int(out[k]["n_corr"]) == n


def test_pair_larger_than_the_k5_staging_area_takes_the_exact_path(engine, oracle):
    rng = np.random.default_rng(32)
    n = 11600  # > 11,264 staged points: K5 scores every point in FP64 and keeps its LO mask in global memory
    corr, R, t = two_view(n, 0.5, rng)
    g = engine.estimate_pose(corr, THR, [])
    o = oracle.estimate_pose(corr, THR, [])
    _check(g["verdict"], g["mask"], corr, o)
    # and a mixed wave: the big pair next to a small one (smemPts is clamped to the limit, the small one is staged)
    small, _, _ = two_view(300, 0.3, rng)
    engine.register_pairs(np.vstack([corr, small]), [0, n, n + 300], [THR, THR])
    out = engine.run_wave(np.arange(2), None, None, flags=WAVE_FALLBACK)
    assert int(out[0]["inlier_count"]) == o["inlier_number"] and np.array_equal(out[0]["E"].reshape(3, 3), o["E"])
    o2 = oracle.estimate_pose(small, THR, [])
    assert int(out[1]["inlier_count"]) == o2["inlier_number"] and np.array_equal(out[1]["E"].reshape(3, 3), o2["E"])


def test_several_guesses_last_one_decides_and_mask_accumulates(engine, oracle):
    rng = np.random.default_rng(33)
    corr, R, t = two_view(600, 0.3, rng)
    good = perturbed_pose(R, t, rng, 1e-4, 1e-4)
    other = perturbed_pose(R, t, rng, 2e-2, 2e-2)
    for guesses in ([good, other], [other, good], [good, good], [other, other, good]):
        g = engine.estimate_pose(corr, THR, guesses)
        o = oracle.estimate_pose(corr, THR, guesses)
        _check(g["verdict"], g["mask"], corr, o)
        assert int(g["verdict"]["path_inliers"]) == o["path_inliers"]


def test_status_codes(engine):
    lib, h = engine.lib, engine.h
    rng = np.random.default_rng(34)
    corr, _, _ = two_view(100, 0.2, rng)
    engine.register_pairs(corr, [0, 100], [THR])
    out = np.zeros(1, dtype=VERDICT_DTYPE)
    assert lib.pgi_wait_wave(h, out.ctypes.data_as(C.c_void_p), None) == -4  # PGI_ERR_STATE: nothing in flight
    with pytest.raises(PgiError):
        engine.run_wave(np.array([7], dtype=np.uint32), None, None, flags=WAVE_PATH)  # pair id out of range
    assert b"out of range" in lib.pgi_last_error(h)
    empty = engine.run_wave(np.zeros(0, dtype=np.uint32), None, None)
    assert len(empty) == 0
    st = engine.stats()
    assert st["launches"] > 0 and st["h2d_bytes"] > 0


def test_three_kernel_k4_matches_the_oracle(engine, oracle):
    """K4a/K4b/K4c (lane-refill Durand-Kerner) must solve every polynomial with the oracle's sweep sequence: the same
    solutions in the same order, hence the oracle's verdict and inlier mask for every fallback pair of a wave."""
    rng = np.random.default_rng(41)
    sizes = [5, 9, 64, 500, 1200, 2000, 2000, 777]
    pairs = [two_view(n, 0.35, rng)[0] for n in sizes]
    off = np.concatenate([[0], np.cumsum(sizes)])
    engine.register_pairs(np.vstack(pairs), off, [THR] * len(sizes))
    out, masks = engine.run_wave(np.arange(len(sizes)), None, None, flags=WAVE_FALLBACK, want_masks=True)
    for k in range(len(sizes)):
        _check(out[k], masks[off[k]:off[k + 1]], pairs[k], oracle.estimate_pose(pairs[k], THR, []))
    assert int(out["accepted"].sum()) >= 5  # the comparison is about real fallback runs
