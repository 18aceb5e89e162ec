"""pgi_guided_match at its edges, bit for bit against the oracle's guided matcher: prepared quantities (F, epipole,
angular range, bin count), matches in order, adapted-ratio bits and guidedMatching's selection.
- Degenerate geometry: lateral motion (the epipole at infinity; with t = (1, 1e-7, 0) the angular range is exactly 0
  and every bin argument is NaN or +-inf), a small rotation with lateral motion, backward motion, and the epipole within
  a pixel of each border of the source image, on either side of the in-image test.
- Hand-built destination sets: exact candidate counts around the count-corrected ratio's steps, duplicated destination
  keypoints with identical descriptors (tests/test_matcher_reference.py checks the same cases against a numpy
  restatement).
- Sizes: source counts around the 256-thread block, one and 16 384 destination keypoints, 20 000 source and destination
  keypoints (more than a view of the registered scene may have), source keypoints outside the image, 64-d descriptors;
  other descriptor widths are rejected.
- Bin numbers 1, 2, 45, 180, 192 and 0 (the angular range's integer part).
- Selection at n == max_points and n == max_points + 1, and with equal values straddling the cut."""
import numpy as np
import pytest

from pose_graph_initialization_b200.engine import PgiError
from helpers import rodrigues, two_view_keypoints_posed
from test_matcher_reference import (COUNTS, K_DST, K_SRC, LATERAL_POSES, R_GEN, SIZE_DST, SIZE_SRC, T_GEN, count_case,
                                    lateral_case, tie_case)

pytestmark = pytest.mark.gpu


def _compare(engine, oracle, args, bin_number=45, max_points=100):
    ref = oracle.guided_match(*args, bin_number=bin_number, max_points=max_points)
    out = engine.guided_match(*args, bin_number=bin_number, max_points=max_points)
    assert out["prepared"].tobytes() == ref["prepared"].tobytes(), (out["prepared"], ref["prepared"])
    assert np.array_equal(out["matches"], ref["matches"]), (len(out["matches"]), len(ref["matches"]))
    assert out["ratios"].tobytes() == ref["ratios"].tobytes()
    sel = [(int(a), int(b), float(r)) for (a, b), r in zip(ref["selected_matches"], ref["selected_ratios"])]
    assert out["selected"] == sel
    return ref


def _args(d):
    return (d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], d["pose"], d["K_src"], d["K_dst"], d["size_src"],
            d["size_dst"])


def _posed(R, t, n=1500, seed=0, **kw):
    return two_view_keypoints_posed(n, np.random.default_rng(seed), R, t, K_SRC, K_DST, SIZE_SRC, SIZE_DST, desc_noise=0.02, **kw)


def _epipole_case(ex, ey):
    """R = I and the destination camera centre one unit in front of the source camera, on the ray through pixel (ex, ey)
    of the source image: the epipole in the source image is (ex, ey)."""
    C = np.linalg.inv(K_SRC) @ np.array([ex, ey, 1.0])
    return np.eye(3), -C


W, H = SIZE_SRC
GEOMETRY = {
    **{"lateral_" + k: None for k in LATERAL_POSES},
    "small_rotation_lateral": (rodrigues(np.array([0.0, 1e-3, 0.0])), np.array([1.0, 0.0, 0.0])),
    "backward": (rodrigues(np.array([0.02, -0.01, 0.03])), np.array([0.1, 0.05, -1.0]) / np.linalg.norm([0.1, 0.05, -1.0])),
}
EPIPOLES = {**{f"epipole_x={ex:g}": (ex, H / 2.0) for ex in (-0.5, 0.5, W - 0.5, W + 0.5)},
            **{f"epipole_y={ey:g}": (W / 2.0, ey) for ey in (-0.5, 0.5, H - 0.5, H + 0.5)}}
GEOMETRY.update({k: _epipole_case(*e) for k, e in EPIPOLES.items()})


@pytest.mark.parametrize("name", list(GEOMETRY))
def test_degenerate_geometry(engine, oracle, name):
    if name.startswith("lateral_"):
        args = lateral_case(name[len("lateral_"):])
    else:
        args = _args(_posed(*GEOMETRY[name]))
    ref = _compare(engine, oracle, args)
    assert len(ref["matches"]) > 50
    P = ref["prepared"]
    if name == "lateral_x_y1e-7":
        assert P[12] == 0.0  # every bin argument is NaN or +-inf: x86 puts them all in bin 0
    if name in EPIPOLES:  # inside the source image the angular range is 0 - 180 (matcher.h:236-241)
        ex, ey = EPIPOLES[name]
        assert abs(P[9] - ex) < 1e-6 and abs(P[10] - ey) < 1e-6
        assert (P[12] == -180.0) == (0 <= ex < W and 0 <= ey < H)


@pytest.mark.parametrize("k", COUNTS)
def test_candidate_counts(engine, oracle, k):
    args, best = count_case(k)
    ref = _compare(engine, oracle, args)
    assert ref["matches"].tolist() == ([] if k == 1 else [[0, best]])


def test_duplicated_destination_keypoints_first_in_keypoint_order_wins(engine, oracle):
    ref = _compare(engine, oracle, tie_case())
    assert ref["matches"].tolist() == [[0, 10]]


@pytest.fixture(scope="module")
def generic(oracle):
    """A generic pose with K_src != K_dst; source keypoints reordered so that the matched ones come first."""
    d = _posed(R_GEN, T_GEN, n=600, seed=1)
    ref = oracle.guided_match(*_args(d))
    first = ref["matches"][:, 0].astype(np.int64)
    order = np.concatenate([first, np.setdiff1d(np.arange(len(d["kp_src"])), first)])
    d["kp_src"], d["desc_src"] = d["kp_src"][order], d["desc_src"][order]
    assert len(first) > 100
    return d


@pytest.mark.parametrize("n_src", [1, 255, 256, 257, 513])
def test_source_counts(engine, oracle, generic, n_src):
    args = list(_args(generic))
    args[0], args[1] = args[0][:n_src], args[1][:n_src]
    ref = _compare(engine, oracle, tuple(args))
    assert len(ref["matches"]) >= min(n_src, 100)


def test_one_destination_keypoint(engine, oracle, generic):
    args = list(_args(generic))
    args[2], args[3] = args[2][:1], args[3][:1]
    ref = _compare(engine, oracle, tuple(args))
    assert len(ref["matches"]) == 0 and ref["prepared"][13] == 45  # one candidate at most: the ratio is "too good"


def test_16384_destination_keypoints(engine, oracle):
    d = _posed(R_GEN, T_GEN, n=12800, seed=2)
    d["kp_dst"], d["desc_dst"] = d["kp_dst"][:16384], d["desc_dst"][:16384]
    assert len(d["kp_dst"]) == 16384
    ref = _compare(engine, oracle, _args(d))
    assert len(ref["matches"]) > 1000


def test_20000_keypoints(engine, oracle):
    d = _posed(R_GEN, T_GEN, n=15400, seed=6)
    d["kp_src"], d["desc_src"] = d["kp_src"][:20000], d["desc_src"][:20000]
    assert len(d["kp_src"]) == 20000 and len(d["kp_dst"]) > 20000
    ref = _compare(engine, oracle, _args(d))
    assert len(ref["matches"]) > 1000


def test_descriptor_widths_other_than_64_and_128_are_rejected(engine, generic):
    args = list(_args(generic))
    args[1], args[3] = args[1][:, :96], args[3][:, :96]
    with pytest.raises(PgiError, match="64 or 128"):
        engine.guided_match(*args)


def test_source_keypoints_outside_the_image(engine, oracle, generic):
    rng = np.random.default_rng(3)
    m = 300
    side = rng.integers(0, 4, m)
    out = rng.uniform([0, 0], SIZE_SRC, (m, 2))
    out[side == 0, 0] = -rng.uniform(0.001, 400, (side == 0).sum())
    out[side == 1, 0] = W + rng.uniform(0, 400, (side == 1).sum())
    out[side == 2, 1] = -rng.uniform(0.001, 400, (side == 2).sum())
    out[side == 3, 1] = H + rng.uniform(0, 400, (side == 3).sum())
    args = list(_args(generic))
    args[0] = np.vstack([args[0], out.astype(np.float32)])
    args[1] = np.vstack([args[1], args[1][:m]])  # the descriptors of matched keypoints
    ref = _compare(engine, oracle, tuple(args))
    assert len(ref["matches"]) > 100


def test_64_dimensional_descriptors(engine, oracle):
    ref = _compare(engine, oracle, _args(_posed(R_GEN, T_GEN, seed=4, dim=64)))
    assert len(ref["matches"]) > 50


@pytest.mark.parametrize("bins", [1, 2, 45, 180, 192, 0])
def test_bin_numbers(engine, oracle, generic, bins):
    ref = _compare(engine, oracle, _args(generic), bin_number=bins)
    assert len(ref["matches"]) > 50
    if bins == 0:
        assert ref["prepared"][12] >= 1.0 and ref["prepared"][13] == int(ref["prepared"][12])


def test_selection_at_the_cut(engine, oracle, generic):
    args = _args(generic)
    n = len(oracle.guided_match(*args, max_points=10 ** 6)["matches"])
    assert n > 100
    for max_points in (n, n - 1):
        ref = _compare(engine, oracle, args, max_points=max_points)
        assert len(ref["selected_matches"]) == max_points


def test_equal_values_straddling_the_cut(engine, oracle, generic):
    args = list(_args(generic))
    dup = np.arange(0, 160, 2)  # matched source keypoints, each twice: equal ratios at different source indices
    args[0], args[1] = np.vstack([args[0], args[0][dup]]), np.vstack([args[1], args[1][dup]])
    ref = oracle.guided_match(*args, max_points=10 ** 6)
    r = np.sort(ref["ratios"])
    cuts = [k for k in range(1, len(r)) if r[k - 1] == r[k]]
    assert len(cuts) >= 10
    for k in cuts[:: max(1, len(cuts) // 10)]:
        sel = _compare(engine, oracle, tuple(args), max_points=k)["selected_matches"]
        assert len(sel) == k
