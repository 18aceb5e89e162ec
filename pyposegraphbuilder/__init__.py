"""pyposegraphbuilder — the module name the reference's Python binding was meant to have
(/root/reference/src/pyposegraphbuilder/__init__.py imports a module its build never produces, SURVEY §0.3), served by
the B200 path.  Entry points in the argument style of the reference's (stale) pybind11 sketch
(src/pyposegraphbuilder/src/bindings.cpp:74-82, :255-266): float64 arrays in, (model | None, inlier bool mask) out,
ValueError on shape errors.

    import pyposegraphbuilder as ppg
    pose, inliers = ppg.estimate_pose(corr, thr_norm, poses=[q_t])      # PoseGraphBuilder::estimatePose  PGB:940-1078
    ok, count = ppg.test_pose(corr, thr, pose)                          # InTraversalPoseTester::test    GT:194-233
    matches, ratios = ppg.guided_match(kp1, desc1, kp2, desc2, pose, K1, K2, size1, size2)   # matcher.h:199-405
    matches, ratios = ppg.match_features(desc1, desc2)                   # matchFeatures                  feature_utils.h:103-210
    tracks = ppg.Tracklets(n_views); tracks.add(i, j, matches, mask)    # reconstruction::Tracklets      point_track.h:541-712
    graph = ppg.PoseGraphBuilder(**flags, scene=scene).run()            # PoseGraphBuilder::run           PGB:173-239
    offsets, matches, values = builder.guided_match_edges()             # guidedMatching on every edge    PGB:717-783
    # a scene with keypoint descriptors (scene.make_descriptor_scene) and no matches is matched on the device first

Everything runs on the sm_100a engine through the C-ABI (include/pgi.h, include/pgb.h); there is no CPU path."""
import numpy as np

from pose_graph_initialization_b200 import Engine  # noqa: F401
from pose_graph_initialization_b200.builder import PoseGraphBuilder, Tracklets  # noqa: F401
from pose_graph_initialization_b200 import scene  # noqa: F401

_engine = None


def _eng():
    global _engine
    if _engine is None:
        _engine = Engine(device=0)
    return _engine


def _corr(corr):
    corr = np.ascontiguousarray(corr, dtype=np.float64)
    if corr.ndim != 2 or corr.shape[1] != 4:
        raise ValueError("correspondences must be an [n, 4] array of normalised [x1 y1 x2 y2] rows")
    return corr


def estimate_pose(corr, thr_norm, poses=()):
    """-> (pose qx qy qz qw tx ty tz | None, inlier bool[n]).  `poses` are the path hypotheses (0 or more [7] rows)."""
    corr = _corr(corr)
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 7) if len(poses) else np.zeros((0, 7))
    r = _eng().estimate_pose(corr, float(thr_norm), poses)
    return (r["pose"] if r["success"] else None), r["mask"].astype(bool)


def test_pose(corr, thr, pose, min_inliers=5):
    """-> (passed, inlier count capped at min_inliers)."""
    pose = np.asarray(pose, dtype=np.float64)
    if pose.shape != (7,):
        raise ValueError("pose must be [qx qy qz qw tx ty tz]")
    return _eng().test_pose(_corr(corr), float(thr), pose, int(min_inliers))


def guided_match(kp_src, desc_src, kp_dst, desc_dst, pose, K_src, K_dst, size_src, size_dst, max_points=100):
    """-> (matches [(src, dst, value)] as guidedMatching returns them, all matches [n, 2], adapted ratios [n])."""
    r = _eng().guided_match(kp_src, desc_src, kp_dst, desc_dst, pose, K_src, K_dst, size_src, size_dst, 45, max_points)
    return r["selected"], r["matches"], r["ratios"]


def match_features(desc_src, desc_dst):
    """-> (matches [n, 2] (queryIdx, trainIdx), ratios [n]) as matchFeatures stores them (sorted by ratio)."""
    return _eng().match_features(desc_src, desc_dst)
