"""Oracle restatement of matchFeatures (feature_utils.h:103-210) against the cv2 4.13.0 wheel's BFMatcher(NORM_L2SQR) —
the library call the reference makes, its surviving matches stored in tests/golden/cv_match_features.npz by
make_golden.py: the same surviving matches, ratios to 1e-6 (OpenCV accumulates the squared distances with SIMD lanes, the
restatement in dimension order)."""
import os

import numpy as np
import pytest

from helpers import two_view_keypoints

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cv_match_features.npz")


def _cv2_match(n, seed):
    """cv2's survivors on two_view_keypoints(n, default_rng(seed)): [(ratio, query, train)] sorted by ratio."""
    d = np.load(G)
    k = f"{n}_{seed}"
    return [(float(x), int(i), int(j)) for x, i, j in zip(d["ratio_" + k], d["query_" + k], d["train_" + k])]


@pytest.mark.parametrize("n,seed", [(200, 0), (900, 1)])
def test_match_features_agrees_with_cv2(oracle, n, seed):
    d = two_view_keypoints(n, np.random.default_rng(seed))
    m, r = oracle.match_features(d["desc_src"], d["desc_dst"])
    ref = _cv2_match(n, seed)
    assert len(m) > n // 2
    assert [(int(a), int(b)) for a, b in m] == [(i, j) for _, i, j in ref] or \
        sorted((int(a), int(b)) for a, b in m) == sorted((i, j) for _, i, j in ref)  # (order may differ between equal-to-1e-7 ratios)
    by_pair = {(i, j): x for x, i, j in ref}
    for (a, b), x in zip(m, r):
        assert abs(x - by_pair[(int(a), int(b))]) <= 1e-6 * max(1.0, x)
    assert np.all(np.diff(r) >= 0)
    assert (d["truth"][m[:, 0]] == m[:, 1]).mean() > 0.98


def test_match_features_degenerate_inputs(oracle):
    rng = np.random.default_rng(3)
    a = rng.standard_normal((5, 128)).astype(np.float32)
    m, r = oracle.match_features(a, a[:1])          # one train descriptor: no second neighbour, nothing survives (:174-176)
    assert len(m) == 0 and len(r) == 0
    m, r = oracle.match_features(a[:0], a)
    assert len(m) == 0
    b = np.vstack([a, a[2:3]])                      # a duplicated train row: best == second, ratio 1 -> rejected
    m, r = oracle.match_features(a, b)
    assert 2 not in m[:, 0]
