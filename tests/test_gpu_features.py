"""pgi_match_features against the oracle's restatement of matchFeatures (feature_utils.h:103-210): identical matches in
identical order, bit-identical ratios (same float32 accumulation order on both sides); a row whose distances all overflow
has no match; inputs beyond 16 384 descriptors per side or with a non-finite value are rejected, and so is a call while a
wave is in flight."""
import numpy as np
import pytest

from helpers import two_view_keypoints
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import WAVE_PATH, Engine, PgiError

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,seed,dim", [(40, 0, 128), (700, 1, 128), (2500, 2, 128), (1300, 3, 64)])
def test_match_features_equals_oracle(engine, oracle, n, seed, dim):
    d = two_view_keypoints(n, np.random.default_rng(seed))
    a, b = d["desc_src"][:, :dim].copy(), d["desc_dst"][:, :dim].copy()
    m, r = engine.match_features(a, b)
    mo, ro = oracle.match_features(a, b)
    assert np.array_equal(m, mo)
    assert np.array_equal(r.view(np.uint64), ro.view(np.uint64))
    if dim == 128 and n >= 700:
        assert len(m) > n // 2 and (d["truth"][m[:, 0]] == m[:, 1]).mean() > 0.98


def test_match_features_ties_and_degenerate_inputs(engine, oracle):
    rng = np.random.default_rng(5)
    a = rng.integers(-3, 4, (300, 128)).astype(np.float32)   # small integers: many exactly equal distances
    b = np.vstack([a[rng.permutation(300)[:200]] + rng.integers(0, 2, (200, 128)).astype(np.float32), a[:50]])
    m, r = engine.match_features(a, b)
    mo, ro = oracle.match_features(a, b)
    assert np.array_equal(m, mo) and np.array_equal(r.view(np.uint64), ro.view(np.uint64))
    for x, y in ((a[:5], a[:1]), (a[:0], a), (a, a[:0])):
        m, r = engine.match_features(x, y)
        assert len(m) == 0 and len(r) == 0
    with pytest.raises(ValueError):
        engine.match_features(a[:, :100], b[:, :100])


def test_a_row_whose_distances_overflow_has_no_match(engine, oracle):
    d = two_view_keypoints(700, np.random.default_rng(6))
    a, b = d["desc_src"].copy(), d["desc_dst"]
    bad = int(np.nonzero(d["truth"] >= 0)[0][0])  # a source row that has a true match
    a[bad] = 1e20  # finite, but every squared distance to it overflows to inf
    m, r = engine.match_features(a, b)
    with np.errstate(over="ignore"):
        mo, ro = oracle.match_features(a, b)
    assert bad not in m[:, 0] and len(m) > 300
    keep = mo[:, 0] != bad
    assert np.array_equal(m, mo[keep]) and np.array_equal(r.view(np.uint64), ro[keep].view(np.uint64))


def test_oversized_and_non_finite_inputs_are_rejected(engine):
    rng = np.random.default_rng(7)
    a = rng.standard_normal((16385, 64)).astype(np.float32)
    for x, y in ((a, a[:10]), (a[:10], a)):
        with pytest.raises(PgiError, match="at most 16384"):
            engine.match_features(x, y)
    for v in (np.nan, np.inf):
        b = a[:50].copy()
        b[7, 3] = v
        for x, y in ((b, a[:40]), (a[:40], b)):
            with pytest.raises(PgiError, match="non-finite"):
                engine.match_features(x, y)
    m, _ = engine.match_features(a[:300], a[:300])  # the context is still usable after the rejections
    assert len(m) == 300


def test_a_wave_in_flight_is_left_alone():
    e = Engine(device=0)
    e.register_scene(S.make_scene(n_views=6, n_corr=256, outlier_ratio=0.3, seed=1, n_points=600), 0.4)
    a = np.random.default_rng(8).standard_normal((200, 128)).astype(np.float32)
    e.submit_wave(np.arange(2, dtype=np.uint32), flags=WAVE_PATH)
    with pytest.raises(PgiError, match="in flight"):
        e.match_features(a, a)
    e.wait_wave()
    assert len(e.match_features(a, a)[0]) == 200
    e.close()
