"""pgi_guided_match against the oracle's restatement of HashingBasedMatcherWithPose<false, 45>::match
(matcher.h:199-405) and of guidedMatching's selection (pose_graph_builder.h:760-782): same prepared quantities (F,
epipole, angular range), same matches in the same order, bit-identical adapted ratios."""
import numpy as np
import pytest

from helpers import two_view_keypoints

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,seed,bins", [(300, 1, 45), (1500, 2, 45), (4000, 3, 45), (1500, 4, 180), (40, 5, 45)])
def test_guided_match_equals_oracle(engine, oracle, n, seed, bins):
    d = two_view_keypoints(n, np.random.default_rng(seed))
    args = (d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], d["pose"], d["K"], d["K"], d["size"], d["size"])
    ref = oracle.guided_match(*args, bin_number=bins, max_points=100)
    out = engine.guided_match(*args, bin_number=bins, max_points=100)
    assert np.array_equal(out["prepared"].view(np.uint64), ref["prepared"].view(np.uint64))
    assert np.array_equal(out["matches"], ref["matches"])
    assert np.array_equal(out["ratios"].view(np.uint64), ref["ratios"].view(np.uint64))
    sel = [(int(a), int(b), float(r)) for (a, b), r in zip(ref["selected_matches"], ref["selected_ratios"])]
    assert out["selected"] == sel
    if n >= 1500:
        m = out["matches"]
        assert len(m) > 10 and (d["truth"][m[:, 0]] == m[:, 1]).mean() > 0.95


def test_guided_match_epipole_inside_the_image_and_degenerate_inputs(engine, oracle):
    # forward motion puts the epipole inside the source image: angular range = 0 - 180 (matcher.h:236-241, :271)
    rng = np.random.default_rng(7)
    d = two_view_keypoints(800, rng)
    pose = np.array([0.0, 0.0, 0.0, 1.0, 0.02, 0.01, 1.0])
    args = (d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], pose, d["K"], d["K"], d["size"], d["size"])
    ref = oracle.guided_match(*args)
    out = engine.guided_match(*args)
    assert ref["prepared"][12] == -180.0
    assert np.array_equal(out["prepared"].view(np.uint64), ref["prepared"].view(np.uint64))
    assert np.array_equal(out["matches"], ref["matches"]) and np.array_equal(out["ratios"].view(np.uint64), ref["ratios"].view(np.uint64))
    empty = engine.guided_match(d["kp_src"][:0], d["desc_src"][:0], d["kp_dst"], d["desc_dst"], pose, d["K"], d["K"], d["size"], d["size"])
    assert len(empty["matches"]) == 0
    with pytest.raises(ValueError):
        engine.guided_match(d["kp_src"], d["desc_src"][:5], d["kp_dst"], d["desc_dst"], pose, d["K"], d["K"], d["size"], d["size"])
