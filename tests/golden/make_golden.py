"""Generates tests/golden/*.npz — golden vectors for the OpenCV-owned stages of the hot path, produced by the
cv2 wheel of THIS container (opencv-python-headless 4.13.0).  The reference (C++) cannot be built or imported
here, and has no tests of its own (SURVEY §4), so the pins are its third-party dependency's observable behaviour
at the reference's call sites (pose_graph_builder.h:1013-1020, :1037-1044).  Run:  python tests/golden/make_golden.py
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from helpers import two_view, two_view_keypoints  # noqa: E402

cv2.setNumThreads(1)
rng = np.random.default_rng(2024)

# --- cv::RNG (MWC) through cv2.randu-free route: the legacy RANSAC's first sample is observable (App. B.2)
# --- cv::SVD::compute(5x9, FULL_UV)  (null-space basis incl. the RNG-seeded completion)
Q = rng.standard_normal((24, 5, 9))
W = np.empty((24, 5)); VT = np.empty((24, 9, 9))
for k in range(24):
    w, u, vt = cv2.SVDecomp(Q[k], flags=cv2.SVD_FULL_UV)
    W[k], VT[k] = w.ravel(), vt
# --- cv::SVD::solveZ on 3x3
B = rng.standard_normal((24, 3, 3))
Z = np.stack([cv2.SVDecomp(B[k])[2][-1] for k in range(24)])
# --- cv::invert (LU) 10x10
A = rng.standard_normal((12, 10, 10))
AI = np.stack([cv2.invert(A[k])[1] for k in range(12)])
# --- cv::solvePoly degree 10
C = rng.standard_normal((24, 11))
R = np.stack([cv2.solvePoly(C[k].reshape(1, -1))[1].reshape(10, 2) for k in range(24)])
np.savez_compressed(os.path.join(HERE, "cv_linear_algebra.npz"), Q=Q, W=W, VT=VT, B=B, Z=Z, A=A, AI=AI, C=C, R=R)

# --- five-point kernel: cv2.findEssentialMat on exactly 5 points returns ALL solutions, in order (App. B.6)
P5 = np.empty((120, 5, 4)); counts = np.zeros(120, dtype=np.int32); sols = np.zeros((120, 10, 3, 3))
for k in range(120):
    c, _, _ = two_view(5, 0.4 if k % 3 == 0 else 0.0, rng)
    P5[k] = c
    E, _ = cv2.findEssentialMat(c[:, :2].copy(), c[:, 2:].copy(), np.eye(3), cv2.RANSAC, 0.99, 1.0)
    n = 0 if E is None else E.shape[0] // 3
    counts[k] = n
    if n:
        sols[k, :n] = E.reshape(n, 3, 3)
np.savez_compressed(os.path.join(HERE, "cv_five_point.npz"), P5=P5, counts=counts, sols=sols)

# --- legacy findEssentialMat(RANSAC, 0.99, DBL_MAX): "first solution of the first sample" (App. B.2), incl. k<5, k==5
cases = []
for n in (3, 4, 5, 6, 7, 20, 57, 300, 1000):
    for rep in range(3):
        c, _, _ = two_view(n, 0.3, rng)
        E, mask = cv2.findEssentialMat(c[:, :2].copy(), c[:, 2:].copy(), np.eye(3), cv2.RANSAC, 0.99, np.finfo(np.float64).max)
        cases.append((c, None if E is None else E.copy(), None if mask is None else mask.ravel().copy()))
np.savez_compressed(os.path.join(HERE, "cv_legacy_ransac.npz"), n=len(cases),
                    **{f"c{i}": cs[0] for i, cs in enumerate(cases)},
                    **{f"E{i}": (cs[1] if cs[1] is not None else np.zeros((0, 3))) for i, cs in enumerate(cases)},
                    **{f"m{i}": (cs[2] if cs[2] is not None else np.zeros(0, dtype=np.uint8)) for i, cs in enumerate(cases)})

# --- USAC_MAGSAC black box (fallback call site): accept/reject + inlier count + E on a few scenes (statistical pin)
us = []
for n, rho in ((300, 0.3), (1000, 0.4), (2000, 0.4), (2000, 0.7), (500, 1.0)):
    c, Rg, tg = two_view(n, rho, rng)
    thr = 0.4 / 800.0
    E, mask = cv2.findEssentialMat(c[:, :2].copy(), c[:, 2:].copy(), np.eye(3), cv2.USAC_MAGSAC, 0.99, thr)
    us.append((c, E[:3].copy() if E is not None else np.zeros((3, 3)), mask.ravel().copy(), Rg, tg))
np.savez_compressed(os.path.join(HERE, "cv_usac_magsac.npz"), n=len(us),
                    **{f"c{i}": u[0] for i, u in enumerate(us)}, **{f"E{i}": u[1] for i, u in enumerate(us)},
                    **{f"m{i}": u[2] for i, u in enumerate(us)}, **{f"R{i}": u[3] for i, u in enumerate(us)},
                    **{f"t{i}": u[4] for i, u in enumerate(us)})

# --- matchFeatures (feature_utils.h:103-210): BFMatcher(NORM_L2SQR) 2-NN both ways, 0.90 ratio test, mutual check,
#     survivors sorted by ratio -> (ratio, query, train) on the descriptors of tests/test_oracle_features.py
mf = {}
for n, seed in ((200, 0), (900, 1)):
    d = two_view_keypoints(n, np.random.default_rng(seed))
    fw = cv2.BFMatcher(cv2.NORM_L2SQR).knnMatch(d["desc_src"], d["desc_dst"], 2)
    bw = cv2.BFMatcher(cv2.NORM_L2SQR).knnMatch(d["desc_dst"], d["desc_src"], 2)
    good = []
    for i, m in enumerate(fw):
        if len(m) < 2 or len(bw[m[0].trainIdx]) < 2:
            continue
        if m[0].distance < 0.90 * m[1].distance and m[0].queryIdx == bw[m[0].trainIdx][0].trainIdx:
            good.append((m[0].distance / m[1].distance, i, m[0].trainIdx))
    good.sort()
    mf[f"ratio_{n}_{seed}"] = np.array([g[0] for g in good])
    mf[f"query_{n}_{seed}"] = np.array([g[1] for g in good], dtype=np.int32)
    mf[f"train_{n}_{seed}"] = np.array([g[2] for g in good], dtype=np.int32)
np.savez_compressed(os.path.join(HERE, "cv_match_features.npz"), **mf)
print("golden vectors written to", HERE, "with cv2", cv2.__version__)
