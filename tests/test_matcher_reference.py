"""A plain numpy restatement of the guided matcher's match() (matcher.h:285-406) against the oracle
(oracle/pgo_matcher.hpp) on hand-built destination sets: exact candidate counts around the count-corrected ratio's
steps (countSnn < 3 / 5 / 10 / 20), duplicated destination keypoints with identical descriptors, and a lateral pose whose
angular range is exactly 0.  The restatement takes the prepared quantities (F, epipole, angular range) from the oracle
and does the rest independently: float32 descriptor differences accumulated in float64 in dimension order (np.cumsum),
math.atan2 (the host libm, as std::atan2), std::round, and the x86 conversion of a bin argument that is NaN or out of
int range (cvttsd2si: INT_MIN, so bin 0).  The same cases run on the device in tests/test_gpu_matcher_edges.py."""
import math

import numpy as np

from helpers import intrinsics, pose_qt, rodrigues, two_view_keypoints_posed

INT_MIN = -2 ** 31


def round_half_away(v):
    """std::round of a finite double (Python's round() rounds halves to even)."""
    a = abs(v)
    fl = math.floor(a)
    r = fl + 1.0 if a - fl >= 0.5 else fl
    return math.copysign(r, v)


def x86_int(v):
    """static_cast<int>(std::round(v)) as x86-64 evaluates it: cvttsd2si gives INT_MIN for NaN and out-of-range values."""
    if not math.isfinite(v):
        return INT_MIN
    r = round_half_away(v)
    return int(r) if -2147483648.0 <= r < 2147483648.0 else INT_MIN


def line_angle(ny, nx):
    angle = (180.0 / math.pi) * math.atan2(ny, nx) + 180.0
    return angle - 180.0 if angle > 180 else angle


def bin_of(prepared, angle, to_int=x86_int):
    mn, rg, nb = (np.float64(x) for x in prepared[11:14])
    with np.errstate(all="ignore"):
        v = np.float64(nb - 1) * (np.float64(angle) - mn) / rg
    return min(max(0, to_int(float(v))), int(nb) - 1)


def match_reference(kp_src, desc_src, kp_dst, desc_dst, prepared, to_int=x86_int):
    """match(): (matches [n, 2], adapted ratios [n], countSnn per source keypoint)."""
    F = [float(x) for x in prepared[:9]]
    ex, ey = float(prepared[9]), float(prepared[10])
    nb = int(prepared[13])
    e11, e12, e13, e21, e22, e23, e31, e32, e33 = F
    bins = [[] for _ in range(nb)]
    for i, (x, y) in enumerate(np.asarray(kp_dst, dtype=np.float64)):
        nx = e11 * x + e21 * y + e31
        ny = e12 * x + e22 * y + e32
        bins[bin_of(prepared, line_angle(ny, nx), to_int)].append(i)
    kd = np.asarray(kp_dst, dtype=np.float64)
    matches, ratios, counts = [], [], []
    for i, (x1, y1) in enumerate(np.asarray(kp_src, dtype=np.float64)):
        x1, y1 = float(x1), float(y1)
        b = bin_of(prepared, line_angle(x1 - ex, -(y1 - ey)), to_int)
        cand = np.array(bins[b], dtype=np.int64)
        x2, y2 = kd[cand, 0], kd[cand, 1]
        with np.errstate(all="ignore"):
            rxc = e11 * x2 + e21 * y2 + e31
            ryc = e12 * x2 + e22 * y2 + e32
            rwc = e13 * x2 + e23 * y2 + e33
            r = x1 * rxc + y1 * ryc + rwc
            rx = e11 * x1 + e12 * y1 + e13
            ry = e21 * x1 + e22 * y1 + e23
            a1 = rxc * rxc + ryc * ryc
            b1 = rx * rx + ry * ry
            d2 = r * r * (a1 + b1) / (a1 * b1)
        near = cand[~(d2 >= 0.75 * 0.75)]
        diff = (desc_src[i][None, :] - desc_dst[near]).astype(np.float64)  # float32 subtraction, then widened
        dist = np.cumsum(diff * diff, axis=1)[:, -1] if len(near) else np.zeros(0)
        best = second = np.finfo(np.float64).max
        best_index = -1
        for nbr, dd in zip(near, dist):
            if dd < best:
                second, best, best_index = best, dd, int(nbr)
        count = len(near)
        corr = 1.0
        if count < 20:
            corr = 0.65 * 0.65
        if count < 10:
            corr = 0.6 * 0.6
        if count < 5:
            corr = 0.5 * 0.5
        if count < 3:
            corr = 0.25 * 0.25
        counts.append(count)
        with np.errstate(all="ignore"):
            adapted = float(np.float64(best) / np.float64(second) / np.float64(corr))
        if adapted < 0.00001:
            continue
        if best_index > -1 and (adapted < 0.8 * 0.8 or count == 1):
            matches.append((i, best_index))
            ratios.append(adapted)
    return np.array(matches, dtype=np.uint32).reshape(-1, 2), np.array(ratios, dtype=np.float64), np.array(counts)


# ---- hand-built cases (shared with tests/test_gpu_matcher_edges.py) ------------------------------------------------------
SIZE_SRC, SIZE_DST = (1601, 1199), (1280, 960)
K_SRC, K_DST = intrinsics(1000.0, SIZE_SRC), intrinsics(760.0, SIZE_DST)
R_GEN = rodrigues(np.array([0.05, -0.12, 0.03]))
T_GEN = np.array([0.8, 0.3, 0.2]) / np.linalg.norm([0.8, 0.3, 0.2])
SRC_POINT = (700.0, 500.0)


def _pose():
    return pose_qt(R_GEN, T_GEN)


def _fundamental():
    t = T_GEN
    E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ R_GEN
    return np.linalg.inv(K_DST).T @ E @ np.linalg.inv(K_SRC)


def _points_on_line(k, offset_px=0.0, start=0.0, step=23.0):
    """k destination points on the epipolar line of SRC_POINT (offset_px off it), `step` px apart, inside the image."""
    a, b, c = _fundamental() @ np.array([SRC_POINT[0], SRC_POINT[1], 1.0])
    n = np.array([a, b]) / math.hypot(a, b)
    c /= math.hypot(a, b)
    centre = np.array(SIZE_DST) / 2.0
    foot = centre - (n @ centre + c) * n  # closest point of the line to the image centre
    d = np.array([-n[1], n[0]])
    s = start + step * (np.arange(k) - (k - 1) / 2.0)
    return foot + s[:, None] * d + offset_px * n


def _line_distance(p):
    a, b, c = _fundamental() @ np.array([SRC_POINT[0], SRC_POINT[1], 1.0])
    return np.abs(p @ np.array([a, b]) + c) / math.hypot(a, b)


def _off_line(rng, m):
    """m destination points uniform in the image, every one more than 3 px from the epipolar line of SRC_POINT."""
    p = rng.uniform([1.0, 1.0], np.array(SIZE_DST) - 1.0, (4 * m + 64, 2))
    return p[_line_distance(p) > 3.0][:m]


def _scatter(rng, first, rest):
    """first and rest interleaved at random positions, each keeping its order -> (rows, positions of first's rows)."""
    n = len(first) + len(rest)
    slots = np.sort(rng.choice(n, len(first), replace=False))
    out = np.empty((n,) + first.shape[1:], dtype=first.dtype)
    out[slots] = first
    out[np.setdiff1d(np.arange(n), slots)] = rest
    return out, slots


def count_case(k, dim=128, seed=0):
    """One source keypoint with exactly k destination keypoints within 0.75 px of its epipolar line, among 24 keypoints
    more than 3 px off it whose descriptors are closer than any candidate's.  In keypoint order the first candidate is the
    worst (squared descriptor distance 2), the second the best (chosen so that the count-corrected ratio is 0.5 when the
    count is right), the rest in between.  Returns (guided_match arguments, index of the best candidate)."""
    rng = np.random.default_rng(seed + k)
    corr = 0.25 ** 2 if k < 3 else 0.5 ** 2 if k < 5 else 0.6 ** 2 if k < 10 else 0.65 ** 2 if k < 20 else 1.0
    sq = [2.0, 2.0 * 0.5 * corr] + list(np.linspace(1.2, 1.9, max(k - 2, 0)))
    desc_src = np.zeros((1, dim), dtype=np.float32)
    desc_src[0, 0] = 1.0
    cand = np.zeros((k, dim), dtype=np.float32)
    cand[:, 0] = 1.0
    for j in range(k):
        cand[j, 1 + j % (dim - 1)] = np.sqrt(sq[j])
    other = np.zeros((24, dim), dtype=np.float32)
    other[:, 0], other[:, 1] = 1.0, 0.01
    rows, slots = _scatter(rng, np.hstack([_points_on_line(k), cand]), np.hstack([_off_line(rng, 24), other]))
    kp_dst, desc_dst = rows[:, :2].astype(np.float32), np.ascontiguousarray(rows[:, 2:], dtype=np.float32)
    args = (np.array([SRC_POINT], dtype=np.float32), desc_src, kp_dst, desc_dst, _pose(), K_SRC, K_DST, SIZE_SRC, SIZE_DST)
    return args, int(slots[1]) if k > 1 else -1


def tie_case():
    """Duplicated destination keypoints with identical descriptors (same position, then another position on the line),
    spread over several 32-keypoint ballot chunks: the first in keypoint order must be the match."""
    rng = np.random.default_rng(5)
    dim = 128
    on = _points_on_line(6)
    kp_dst = _off_line(rng, 340).astype(np.float32)
    desc_dst = rng.standard_normal((len(kp_dst), dim)).astype(np.float32)
    src = np.zeros(dim, dtype=np.float32)
    src[0] = 1.0
    worst, good, mid = src.copy(), src.copy(), src.copy()
    worst[1], good[2], mid[3] = np.sqrt(2.0), np.sqrt(0.2), 1.0
    # keypoint index: 3 worst, 10 good, 45 good (same position), 300 good (other position), 60 and 200 mid
    for i, p, d in ((3, on[0], worst), (10, on[1], good), (45, on[1], good), (300, on[2], good), (60, on[3], mid),
                    (200, on[4], mid)):
        kp_dst[i], desc_dst[i] = p, d
    return (np.array([SRC_POINT], dtype=np.float32), src[None, :], kp_dst, desc_dst, _pose(), K_SRC, K_DST, SIZE_SRC, SIZE_DST)


COUNTS = (1, 2, 3, 4, 5, 9, 10, 19, 20, 21)
LATERAL_POSES = {"x": (np.eye(3), [1.0, 0.0, 0.0]), "y": (np.eye(3), [0.0, 1.0, 0.0]),
                 "x_y1e-7": (np.eye(3), [1.0, 1e-7, 0.0]), "x_z1e-9": (np.eye(3), [1.0, 0.0, 1e-9])}


def lateral_case(name, n=1500, seed=5):
    R, t = LATERAL_POSES[name]
    K = intrinsics(800.0, (1600, 1200))
    d = two_view_keypoints_posed(n, np.random.default_rng(seed), R, t, K, K, (1600, 1200), (1600, 1200))
    return (d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], d["pose"], K, K, (1600, 1200), (1600, 1200))


def _equal(oracle, args, **kw):
    ref = oracle.guided_match(*args, **kw)
    m, r, counts = match_reference(args[0], args[1], args[2], args[3], ref["prepared"])
    assert np.array_equal(m, ref["matches"])
    assert r.tobytes() == ref["ratios"].tobytes()
    return ref, counts


def test_candidate_counts_and_the_corrected_ratio(oracle):
    for k in COUNTS:
        args, best = count_case(k)
        ref, counts = _equal(oracle, args)
        assert counts.tolist() == [k], k
        if k == 1:  # second == DBL_MAX: the ratio is "too good to be true" whatever countSnn == 1 says
            assert len(ref["matches"]) == 0
        else:
            assert ref["matches"].tolist() == [[0, best]], k
            assert abs(ref["ratios"][0] - 0.5) < 1e-6, k


def test_duplicated_destination_keypoints_first_in_keypoint_order_wins(oracle):
    ref, counts = _equal(oracle, tie_case())
    assert counts.tolist() == [6]
    assert ref["matches"].tolist() == [[0, 10]]


def test_lateral_poses_equal_the_restatement(oracle):
    for name in LATERAL_POSES:
        ref, _ = _equal(oracle, lateral_case(name))
        assert len(ref["matches"]) > 50, name


def test_a_zero_angular_range_puts_every_keypoint_in_bin_0(oracle):
    """R = I, t = (1, 1e-7, 0): the destination corners' lines all have one angle, so the angular range is exactly 0.  The
    destination bin arguments are 0 / 0 = NaN and the source ones +-inf: x86 converts both to INT_MIN, i.e. bin 0, so
    every source keypoint sees every destination keypoint.  A conversion that saturates +inf to INT_MAX instead puts the
    source keypoints in the last bin, where no destination keypoint is, and finds nothing."""
    args = lateral_case("x_y1e-7")
    ref = oracle.guided_match(*args)
    P = ref["prepared"]
    assert P[12] == 0.0 and P[13] == 45
    F, (ex, ey) = P[:9], P[9:11]
    for x, y in args[2].astype(np.float64):
        assert bin_of(P, line_angle(F[1] * x + F[4] * y + F[7], F[0] * x + F[3] * y + F[6])) == 0
    for x, y in args[0].astype(np.float64):
        assert bin_of(P, line_angle(x - ex, -(y - ey))) == 0
    assert len(ref["matches"]) > 50

    def saturating(v):
        if math.isnan(v):
            return 0
        return max(INT_MIN, min(2 ** 31 - 1, int(round_half_away(v)) if math.isfinite(v) else (2 ** 31 - 1 if v > 0 else INT_MIN)))

    m, _, _ = match_reference(*args[:4], P, to_int=saturating)
    assert len(m) < len(ref["matches"])
