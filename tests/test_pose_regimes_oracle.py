"""CPU checks of the pose-path regime generator (tests/helpers.py) that tests/test_gpu_pose_regimes.py runs on the device:
each kind is what it claims to be, no pair can push the LO refit's fixed-point sums out of int64, the frozen fallback
termination pairs still end where they were picked to end, and the crafted pair of K2's "first finite solution" rule
still starts with a sample that has no finite solution."""
import numpy as np
import pytest

from helpers import (REGIME_KINDS, REGIME_OUTLIER_RATIOS, REGIME_SIZES, first_finite_pair, hypotheses_for, lo_fixed_point_bound,
                     regime_pair, regime_set, termination_pairs)


def _pair(kind, n=300, ratio=0.3, seed=7):
    return regime_pair(kind, n, np.random.default_rng(seed), ratio)


def test_regime_kinds_are_what_they_claim():
    p = _pair("wide_fov")
    assert np.abs(p["corr"][:, :2]).max() > 2.0
    p = _pair("off_centre")
    assert np.abs(p["corr"][:, :2].mean(0)).max() < 0.3 and np.abs(p["corr"][:, 2:].mean(0)).max() > 0.8
    p = _pair("forward")
    e2 = p["t"][:2] / p["t"][2]  # epipole of image 2 (x2 ~ R x1 + t): the image of camera 1's centre
    e1 = -(p["R"].T @ p["t"])[:2] / (p["R"].T @ p["t"])[2]
    for e, xy in ((e1, p["corr"][:, :2]), (e2, p["corr"][:, 2:])):
        assert (xy.min(0) < e).all() and (e < xy.max(0)).all()
    p = _pair("pure_rotation")
    assert not p["t"].any()
    assert np.isclose(np.linalg.norm(_pair("tiny_baseline")["t"]), 1e-6)
    # planar: x1 and x2 are related by one homography (up to the noise)
    p = _pair("planar")
    a, b = np.hstack([p["corr"][:, :2], np.ones((300, 1))]), np.hstack([p["corr"][:, 2:], np.ones((300, 1))])
    A = np.vstack([np.hstack([a, np.zeros((300, 3)), -a * b[:, :1]]), np.hstack([np.zeros((300, 3)), a, -a * b[:, 1:2]])])
    s = np.linalg.svd(A, compute_uv=False)
    assert s[-1] < 0.05 * s[-2]
    p = _pair("duplicated", 500)
    u, cnt = np.unique(p["corr"], axis=0, return_counts=True)
    assert len(u) == 50 and (cnt == 10).all()
    assert len(np.unique(_pair("identical", 500)["corr"], axis=0)) == 1
    for r in REGIME_OUTLIER_RATIOS:
        assert _pair("outliers", 2048, r)["n_outliers"] == int(round(2048 * r))
    p = _pair("nonfinite")
    c = p["corr"]
    assert np.isnan(c).any() and np.isposinf(c).any() and np.isneginf(c).any() and np.isfinite(c).all(1).sum() > 250
    p = _pair("focal_zero")
    assert p["thr"] == np.inf and not np.isfinite(p["corr"]).any() and np.isnan(p["corr"]).any()


def test_hypothesis_lists():
    g, b = np.zeros(7), np.ones(7)
    lists = [hypotheses_for(i, g, b) for i in range(6)]
    assert [len(h) for h in lists] == [0, 1, 3, 0, 1, 3]
    assert lists[2][0] is g and lists[2][1] is b and lists[2][2] is g and lists[5][0] is b and lists[5][2] is b


def test_regime_set_covers_every_kind_size_and_ratio_and_stays_in_the_lo_fixed_point_domain():
    """The LO refit accumulates a_r a_q 2^40 over the inlier rows in int64 (pgo_fallback.hpp lsRefit, K5's lsRefitBlock):
    parity with the oracle needs every sum below 2^62 whatever the inliers, which lo_fixed_point_bound bounds."""
    rs = regime_set()
    labels = [lab for lab, *_ in rs]
    for kind in REGIME_KINDS:
        assert any(lab.startswith(kind + "-") for lab in labels), kind
    assert {len(c) for _, c, _, _ in rs} >= set(REGIME_SIZES)
    assert len({thr for _, _, thr, _ in rs}) >= 5
    pairs = [c for _, c, _, _ in rs] + [c for _, _, c, _ in termination_pairs()] + [first_finite_pair()[0]]
    worst = max(lo_fixed_point_bound(c) for c in pairs)
    assert 0 < worst < 2.0 ** 62


@pytest.mark.parametrize("label,iterations,corr,thr", termination_pairs(), ids=lambda v: v if isinstance(v, str) else "")
def test_termination_edges(oracle, label, iterations, corr, thr):
    r = oracle.fallback(corr, thr)
    assert r["iterations"] == iterations
    if label == "no_inlier":
        assert r["ok"] and r["inliers"] == 0 and r["models"] == 1000
    elif label == "rejected":
        assert r["ok"] and r["inliers"] < 20
    else:
        assert r["ok"] and r["inliers"] >= 20


def test_first_finite_pair(oracle):
    c, thr, hyp, sample = first_finite_pair()
    sols = oracle.five_point(c[sample, :2], c[sample, 2:], 1000, 1e-22)
    assert len(sols) > 0 and not np.isfinite(sols).all(axis=(1, 2)).any()
    assert oracle.test_pose(c, hyp, 1.5 * thr, 5) == (True, 5)
    E = oracle.essential_from_pose(hyp)
    assert len(oracle.get_inliers(c, E, 1.5 * thr)) == len(c)  # k = N: the first sample's ranks are those rows
    nm, _, _, _, iters = oracle.find_essential_ransac_inf(c)
    assert nm > 0 and iters > 1  # the legacy RANSAC moved on to a later sample
    o = oracle.estimate_pose(c, thr, [hyp])
    assert o["success"] and o["branch"] == 1
