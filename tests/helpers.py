"""Shared synthetic two-view data for the tests (seeded; no dependency on /root/reference)."""
import numpy as np


def rodrigues(v):
    th = np.linalg.norm(v)
    if th < 1e-12:
        return np.eye(3)
    k = v / th
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def quat_from_rot(R):
    t = np.trace(R)
    if t > 0:
        s = np.sqrt(t + 1.0) * 2
        q = np.array([(R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s, 0.25 * s])
    else:
        i = int(np.argmax(np.diag(R)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = np.sqrt(R[i, i] - R[j, j] - R[k, k] + 1.0) * 2
        q = np.zeros(4)
        q[i] = 0.25 * s
        q[3] = (R[k, j] - R[j, k]) / s
        q[j] = (R[j, i] + R[i, j]) / s
        q[k] = (R[k, i] + R[i, k]) / s
    return q / np.linalg.norm(q)


def two_view(n, outlier_ratio, rng, f=800.0, noise_px=0.5):
    """n normalised correspondences [x1 y1 x2 y2] of a random relative pose, `outlier_ratio` of them random.
    Returns (corr, R, t) with x2 ~ R x1 + t."""
    X = rng.standard_normal((n, 3)) + np.array([0, 0, 6.0])
    R = rodrigues(rng.uniform(-0.3, 0.3, 3))
    t = rng.standard_normal(3)
    t /= np.linalg.norm(t)
    x1 = X[:, :2] / X[:, 2:]
    X2 = X @ R.T + t
    x2 = X2[:, :2] / X2[:, 2:]
    x1 = x1 + rng.standard_normal((n, 2)) * noise_px / f
    x2 = x2 + rng.standard_normal((n, 2)) * noise_px / f
    no = int(n * outlier_ratio)
    x2[:no] = rng.uniform(-0.8, 0.8, (no, 2))
    p = rng.permutation(n)
    return np.ascontiguousarray(np.hstack([x1, x2])[p]), R, t


def pose_qt(R, t):
    return np.concatenate([quat_from_rot(R), t])


def perturbed_pose(R, t, rng, rot_sigma=1e-4, t_sigma=1e-4):
    Rp = rodrigues(rng.standard_normal(3) * rot_sigma) @ R
    tp = t + rng.standard_normal(3) * t_sigma
    return pose_qt(Rp, tp)


def two_view_keypoints(n, rng, f=800.0, w=1600, h=1200, noise_px=0.3, desc_noise=0.05, extra=0.3):
    """Pixel keypoints (float32) + 128-d float32 descriptors of n shared 3-D points seen by two cameras, plus `extra`*n
    unrelated keypoints per view, each view in its own shuffled order.  Returns dict(kp_src, desc_src, kp_dst, desc_dst,
    pose (T_dst_src as q,t), K, size, truth[src index] = dst index or -1)."""
    X = rng.standard_normal((n, 3)) * np.array([1.5, 1.0, 1.0]) + np.array([0, 0, 7.0])
    R = rodrigues(rng.uniform(-0.25, 0.25, 3))
    t = rng.standard_normal(3) * 0.8
    K = np.array([[f, 0, w / 2.0], [0, f, h / 2.0], [0, 0, 1.0]])
    base = rng.standard_normal((n, 128))
    base /= np.linalg.norm(base, axis=1, keepdims=True)

    def view(Xc):
        uv = (Xc[:, :2] / Xc[:, 2:]) * f + np.array([w / 2.0, h / 2.0]) + rng.standard_normal((n, 2)) * noise_px
        d = base + rng.standard_normal((n, 128)) * desc_noise
        m = int(extra * n)
        uv = np.vstack([uv, rng.uniform([0, 0], [w, h], (m, 2))])
        de = rng.standard_normal((m, 128))
        d = np.vstack([d, de / np.linalg.norm(de, axis=1, keepdims=True)])
        p = rng.permutation(n + m)
        inv = np.empty(n + m, dtype=np.int64)
        inv[p] = np.arange(n + m)
        return uv[p].astype(np.float32), d[p].astype(np.float32), inv  # inv[original] = position in the view

    kp_s, d_s, inv_s = view(X)
    kp_d, d_d, inv_d = view(X @ R.T + t)
    truth = np.full(len(kp_s), -1, dtype=np.int64)
    truth[inv_s[:n]] = inv_d[:n]
    return dict(kp_src=kp_s, desc_src=d_s, kp_dst=kp_d, desc_dst=d_d, pose=pose_qt(R, t), K=K, size=(w, h), truth=truth)


def intrinsics(f, size):
    """K = [f 0 w/2; 0 f h/2; 0 0 1], the camera the reference builds for every view (pose_graph_builder.h:284-286)."""
    return np.array([[f, 0.0, size[0] / 2.0], [0.0, f, size[1] / 2.0], [0.0, 0.0, 1.0]])


def _project(K, X):
    return (X @ K.T)[:, :2] / X[:, 2:]


def _inside(uv, size):
    return (uv[:, 0] >= 0) & (uv[:, 0] < size[0]) & (uv[:, 1] >= 0) & (uv[:, 1] < size[1])


def two_view_keypoints_posed(n, rng, R, t, K_src, K_dst, size_src, size_dst, noise_px=0.3, desc_noise=0.05, extra=0.3,
                             dim=128, depth=7.0):
    """two_view_keypoints with a given relative pose (x_dst ~ R x_src + t) and each view's own intrinsics and image size.
    The n shared points lie in front of both cameras and project inside both images (before the keypoint noise); the
    `extra`*n unrelated keypoints per view are uniform in that view's image.  Returns two_view_keypoints' dict with
    K_src / K_dst and size_src / size_dst in place of K and size."""
    R, t = np.asarray(R, dtype=np.float64), np.asarray(t, dtype=np.float64)
    K_src, K_dst = np.asarray(K_src, dtype=np.float64), np.asarray(K_dst, dtype=np.float64)
    X = np.zeros((0, 3))
    for _ in range(200):
        if len(X) >= n:
            break
        C = rng.standard_normal((4 * n, 3)) * np.array([1.5, 1.0, 1.0]) + np.array([0, 0, depth])
        C2 = C @ R.T + t
        ok = (C[:, 2] > 0.5) & (C2[:, 2] > 0.5) & _inside(_project(K_src, C), size_src) & _inside(_project(K_dst, C2), size_dst)
        X = np.vstack([X, C[ok]])
    assert len(X) >= n, "the two cameras do not share enough of the point cloud"
    X = X[:n]
    base = rng.standard_normal((n, dim))
    base /= np.linalg.norm(base, axis=1, keepdims=True)

    def view(Xc, K, size):
        uv = _project(K, Xc) + rng.standard_normal((n, 2)) * noise_px
        d = base + rng.standard_normal((n, dim)) * desc_noise
        m = int(extra * n)
        uv = np.vstack([uv, rng.uniform([0, 0], size, (m, 2))])
        de = rng.standard_normal((m, dim))
        d = np.vstack([d, de / np.linalg.norm(de, axis=1, keepdims=True)])
        p = rng.permutation(n + m)
        inv = np.empty(n + m, dtype=np.int64)
        inv[p] = np.arange(n + m)
        return uv[p].astype(np.float32), d[p].astype(np.float32), inv

    kp_s, d_s, inv_s = view(X, K_src, size_src)
    kp_d, d_d, inv_d = view(X @ R.T + t, K_dst, size_dst)
    truth = np.full(len(kp_s), -1, dtype=np.int64)
    truth[inv_s[:n]] = inv_d[:n]
    return dict(kp_src=kp_s, desc_src=d_s, kp_dst=kp_d, desc_dst=d_d, pose=pose_qt(R, t), K_src=K_src, K_dst=K_dst,
                size_src=tuple(size_src), size_dst=tuple(size_dst), truth=truth)


# (focal length px, (width, height)): landscape, portrait, small, large and odd sizes (w/2 or h/2 not an integer).  The
# focal lengths are exact in binary, so thr_px / ((f + f + f + f) / 4) == thr_px / f.
CAMERAS = ((1200.0, (1601, 1199)), (450.0, (640, 480)), (2400.0, (3000, 4000)), (912.5, (1200, 1600)),
           (1636.25, (2048, 1535)), (700.0, (1023, 767)))


def per_view_camera_scene(n_views=12, seed=0, cameras=CAMERAS, group=3, n_points=1500, kp_max=1200, dim=128, noise_px=0.2,
                          desc_noise=0.01, distractor_ratio=0.2, radius=6.0, arc=np.pi, with_matches=False,
                          outlier_ratio=0.25):
    """A scene in scene.py's dict layout in which each view has its own camera: view v uses cameras[(v // group) %
    len(cameras)], so neighbouring views of one group share a camera and neighbours across groups do not.  Cameras on a
    ring arc looking at a Gaussian blob, as scene.make_descriptor_scene; view v keeps at most kp_max keypoints: points that
    project inside its image (projected with its own K, plus noise_px), plus distractor_ratio of unrelated keypoints, in
    its own shuffled order, each with a `dim`-d descriptor (a unit vector per point plus desc_noise per dimension).
    with_matches adds m_offset / matches for every pair: its shared points in random order, outlier_ratio of them with a
    wrong destination keypoint.  gt_point[sum K] holds each keypoint's 3-D point (-1 for distractors)."""
    rng = np.random.default_rng(seed)
    V = n_views
    cam_of = [cameras[(v // group) % len(cameras)] for v in range(V)]
    pts = rng.standard_normal((n_points, 3))
    base = rng.standard_normal((n_points, dim))
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    ang = np.arange(V) * (arc / V) + rng.uniform(-0.2, 0.2, V) * (arc / V)
    elev = rng.uniform(-0.2, 0.2, V)
    rad = radius * (1.0 + rng.uniform(-0.1, 0.1, V))
    cam = np.stack([rad * np.cos(ang) * np.cos(elev), rad * np.sin(ang) * np.cos(elev), rad * np.sin(elev)], 1)
    Rw = np.empty((V, 3, 3))
    for v in range(V):
        z = rng.standard_normal(3) * 0.15 - cam[v]
        z /= np.linalg.norm(z)
        x = np.cross(z, [0.0, 0.0, 1.0])
        x /= np.linalg.norm(x)
        Rw[v] = np.stack([x, np.cross(z, x), z])  # rows: camera axes in world coordinates (world -> camera)
    tw = -np.einsum("vij,vj->vi", Rw, cam)
    kps, descs, pids = [], [], []
    for v in range(V):
        f, size = cam_of[v]
        Xc = pts @ Rw[v].T + tw[v]
        uv = _project(intrinsics(f, size), Xc)
        vis = np.flatnonzero((Xc[:, 2] > 0.5) & _inside(uv, size))
        n_real = min(len(vis), int(round(kp_max * (1.0 - distractor_ratio))))
        real = np.sort(rng.choice(vis, n_real, replace=False))
        m = int(round(n_real * distractor_ratio / (1.0 - distractor_ratio)))
        de = rng.standard_normal((m, dim))
        xy = np.vstack([uv[real] + rng.standard_normal((n_real, 2)) * noise_px, rng.uniform([0.0, 0.0], size, (m, 2))])
        d = np.vstack([base[real] + rng.standard_normal((n_real, dim)) * desc_noise, de / np.linalg.norm(de, axis=1, keepdims=True)])
        pid = np.concatenate([real, np.full(m, -1)])
        order = rng.permutation(len(pid))
        kps.append(xy[order].astype(np.float32)); descs.append(d[order].astype(np.float32)); pids.append(pid[order])
    view_dir = Rw[:, 2, :]
    sim = np.round(np.minimum(np.clip(view_dir @ view_dir.T, 0.0, 0.999), 0.999), 3)
    sim = np.round((sim + sim.T) / 2.0, 3)
    np.fill_diagonal(sim, 1.0)
    iu, ju = np.triu_indices(V, 1)
    counts = np.array([len(k) for k in kps])
    sc = dict(focal=np.array([c[0] for c in cam_of]), size=np.array([c[1] for c in cam_of], dtype=np.float64), sim=sim,
              kp_offset=np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64), kp=np.concatenate(kps).reshape(-1, 2),
              desc=np.concatenate(descs).reshape(-1, dim), pair_views=np.stack([iu, ju], 1).astype(np.uint32),
              gt_q=np.array([quat_from_rot(R) for R in Rw]), gt_t=tw.copy(), gt_R=Rw.copy(),
              gt_point=np.concatenate(pids).astype(np.int64))
    if with_matches:
        mo, rows = [0], []
        for s, d in zip(iu, ju):
            ps, pd = pids[s], pids[d]
            where_d = {int(p): k for k, p in enumerate(pd) if p >= 0}
            m = np.array([(k, where_d[int(p)]) for k, p in enumerate(ps) if p >= 0 and int(p) in where_d], dtype=np.int64).reshape(-1, 2)
            m = m[rng.permutation(len(m))]
            bad = rng.random(len(m)) < outlier_ratio
            m[bad, 1] = rng.integers(0, len(pd), int(bad.sum()))
            rows.append(m)
            mo.append(mo[-1] + len(m))
        sc["m_offset"] = np.array(mo, dtype=np.uint64)
        sc["matches"] = np.concatenate(rows).astype(np.uint32).reshape(-1, 2)
    return sc


# ---- pose-path regimes the two_view / make_scene generators never produce ----------------------------------------------
REGIME_KINDS = ("wide_fov", "off_centre", "forward", "pure_rotation", "tiny_baseline", "planar", "duplicated", "identical",
                "outliers", "nonfinite", "focal_zero")
REGIME_SIZES = (5, 6, 9, 19, 20, 21, 2047, 2048, 2049, 4097, 11264, 11265)
REGIME_OUTLIER_RATIOS = (0.0, 0.05, 0.5, 0.85, 1.0)
REGIME_THRESHOLDS = (1e-5, 1e-4, 5e-4, 2e-3, 1e-2)  # per-pair thr_norm across three decades (thr_px 0.4 at f 40 000 .. 40)


def _view_rows(X, R, t, noise, rng):
    """Normalised [x1 y1 x2 y2] rows of the 3-D points X (camera 1) seen by camera 2 (X2 = R X + t), plus noise."""
    x1 = X[:, :2] / X[:, 2:]
    X2 = X @ R.T + t
    x2 = X2[:, :2] / X2[:, 2:]
    c = np.hstack([x1, x2])
    return c + rng.standard_normal(c.shape) * noise


def regime_pair(kind, n, rng, outlier_ratio=0.3, thr=5e-4):
    """One seeded pair of the given regime kind with n rows -> dict(corr [n, 4], thr, R, t, good (a pose near the truth as
    q,t), bad (a wrong pose), outliers (rows replaced by random ones)).  The kinds:
      wide_fov       normalised coordinates up to about +-2.5 (a focal length of 0.2 x the image width)
      off_centre     destination camera turned by ~0.9 rad: the destination rows sit far from the principal point
      forward        motion along the optical axis: the epipole lies inside both images
      pure_rotation  t = 0 exactly
      tiny_baseline  |t| = 1e-6
      planar         every point on one plane
      duplicated     50 distinct rows, each repeated n / 50 times (n a multiple of 50)
      identical      one row repeated n times
      outliers       two_view-like geometry with outlier_ratio of the rows replaced by random ones
      nonfinite      rows with NaN, +inf and -inf coordinates among finite ones
      focal_zero     what createCorrespondenceMatrix makes of a view with focal length 0.0: +-inf / NaN rows, thr = inf"""
    noise = 0.5 / 800.0
    R = rodrigues(rng.uniform(-0.2, 0.2, 3))
    t = rng.standard_normal(3)
    t /= np.linalg.norm(t)
    X = rng.standard_normal((n, 3)) + np.array([0.0, 0.0, 6.0])
    n_out = 0
    if kind == "wide_fov":
        z = rng.uniform(4.0, 8.0, n)
        X = np.stack([rng.uniform(-2.4, 2.4, n) * z, rng.uniform(-2.4, 2.4, n) * z, z], 1)
        t = t * 0.3
        R = rodrigues(rng.uniform(-0.05, 0.05, 3))
        noise = 0.5 / 200.0
    elif kind == "off_centre":
        R = rodrigues(np.array([0.5, -0.9, 0.05]))
        t = np.array([0.8, -0.3, 0.2])
    elif kind == "forward":
        R = rodrigues(rng.uniform(-0.02, 0.02, 3))
        t = np.array([0.03, -0.02, -1.0])
    elif kind == "pure_rotation":
        t = np.zeros(3)
    elif kind == "tiny_baseline":
        t = t * 1e-6
    elif kind == "planar":
        xy = rng.uniform(-2.0, 2.0, (n, 2))
        X = np.stack([xy[:, 0], xy[:, 1], 6.0 + 0.3 * xy[:, 0] - 0.2 * xy[:, 1]], 1)
    corr = _view_rows(X, R, t, noise, rng)
    if kind == "duplicated":
        assert n % 50 == 0
        corr = np.tile(corr[:50], (n // 50, 1))[rng.permutation(n)]
    elif kind == "identical":
        corr = np.repeat(corr[:1], n, 0)
    elif kind == "outliers":
        n_out = int(round(n * outlier_ratio))
        corr[:n_out, 2:] = rng.uniform(-0.8, 0.8, (n_out, 2))
        corr = corr[rng.permutation(n)]
    elif kind == "nonfinite":
        bad = rng.choice(n, max(1, n // 10), replace=False)
        vals = np.array([np.nan, np.inf, -np.inf])
        for k, i in enumerate(bad):
            corr[i, k % 4] = vals[k % 3]
    elif kind == "focal_zero":
        # ((double)kp - c) / 0.0 per coordinate: +-inf, or NaN where the key point sits on the principal point
        sgn = np.sign(rng.standard_normal((n, 4)))
        sgn[rng.random((n, 4)) < 0.05] = 0.0
        with np.errstate(divide="ignore", invalid="ignore"):
            corr = sgn / 0.0
        thr = np.inf
    good = perturbed_pose(R, t, rng)
    bad = pose_qt(rodrigues(np.array([0.0, 0.6, 0.0])), np.array([1.0, 0.0, 0.0]))
    return dict(corr=np.ascontiguousarray(corr), thr=float(thr), R=R, t=t, good=good, bad=bad, n_outliers=n_out)


def hypotheses_for(i, good, bad):
    """0, 1 or 3 hypotheses for the i-th pair of a set (as test_gpu_k1_stream.py): none; a good or a bad one; good, bad,
    good or bad, good, bad (the last one decides)."""
    k = (0, 1, 3)[i % 3]
    first_good = (i // 3) % 2 == 0
    return [good if (first_good if j % 2 == 0 else not first_good) else bad for j in range(k)]


def lo_fixed_point_bound(corr):
    """The largest of the 45 sums  sum_rows |a_r a_q| 2^40  of the fallback's LO refit (a = [x2x1 x2y1 x2 y2x1 y2y1 y2 x1
    y1 1]) over every finite row: an upper bound of the int64 accumulators whatever rows the model makes inliers.  Rows
    with a non-finite coordinate never enter the sums (their Sampson residual is NaN under every E)."""
    c = corr[np.isfinite(corr).all(1)]
    x1, y1, x2, y2 = c.T
    a = np.abs(np.stack([x2 * x1, x2 * y1, x2, y2 * x1, y2 * y1, y2, x1, y1, np.ones(len(c))], 1))
    return float((a.T @ a).max() * 2.0 ** 40) if len(c) else 0.0


# Fallback termination edges: (seed, N, outlier ratio) of two_view(N, ratio, default_rng(seed)) at thr_norm 0.4 / 800,
# picked by a one-off scan with oracle.fallback, keyed by the iteration count they end at: one iteration, both sides of
# K5's 16-iteration batch edges, both sides of the 125-iteration chunk edge and one past the second, and "rejected", which
# runs all 1 000 iterations and keeps a model of fewer than 20 inliers.
TERMINATION_EDGES = (  # (label, iterations, seed, N, outlier ratio, noise_px)
    ("one", 1, 0, 100, 0.0, 0.05),
    ("batch16", 16, 0, 100, 0.23, 0.05),
    ("batch17", 17, 0, 100, 0.25, 0.05),
    ("batch32", 32, 3, 100, 0.32, 0.05),
    ("batch33", 33, 0, 100, 0.24, 0.1),
    ("chunk124", 124, 2, 200, 0.48, 0.1),
    ("chunk125", 125, 2, 200, 0.49, 0.05),
    ("chunk126", 126, 11, 60, 0.1, 0.5),
    ("chunk251", 251, 0, 300, 0.12, 0.5),
    ("rejected", 1000, 6, 60, 0.36, 0.5),
)
TERMINATION_THR = 0.4 / 800.0


def termination_pairs():
    """[(label, expected iterations, corr, thr)] of TERMINATION_EDGES plus an all-NaN pair, which runs all 1 000 iterations
    with models that keep no inlier.  (No input the scan tried ends the fallback without any model: identical, collinear,
    constant-coordinate and zero-motion rows all give the five-point solver solutions to score.)"""
    out = [(lab, it, two_view(n, ratio, np.random.default_rng(seed), noise_px=noise)[0], TERMINATION_THR)
           for lab, it, seed, n, ratio, noise in TERMINATION_EDGES]
    out.append(("no_inlier", 1000, np.full((50, 4), np.nan), TERMINATION_THR))
    return out


def first_finite_pair():
    """A pair whose hypothesis passes the in-traversal test and makes every row an inlier (k = N = 100), with the first
    sample of the legacy RANSAC (its ranks depend on k only) replaced by five rows 1e-9 apart: the five-point solver
    returns a solution for them, but no finite one, so K2 has to keep sampling.  -> (corr, thr, hypothesis, first sample)."""
    from oracle import pgo_oracle as O

    c, R, t = two_view(100, 0.0, np.random.default_rng(5), noise_px=0.05)
    sample = O.find_essential_ransac_inf(c)[3].astype(np.int64)  # the first sample: it succeeds on the clean pair
    c[sample] = c[sample[0]] + np.random.default_rng(0).standard_normal((5, 4)) * 1e-9
    return c, TERMINATION_THR, pose_qt(R, t), sample


def regime_set():
    """The regime pairs of the pose-path tests: [(label, corr, thr, hypotheses)].  Every geometric kind at every size of
    REGIME_SIZES, the row-pattern kinds at a few sizes, every outlier ratio; thresholds cycle through REGIME_THRESHOLDS."""
    rng = np.random.default_rng(2024)
    specs = [(k, n, 0.3) for k in ("wide_fov", "off_centre", "forward", "pure_rotation", "tiny_baseline", "planar", "nonfinite")
             for n in REGIME_SIZES]
    specs += [("duplicated", 500, 0.0), ("duplicated", 1000, 0.0), ("identical", 5, 0.0), ("identical", 21, 0.0),
              ("identical", 500, 0.0), ("focal_zero", 5, 0.0), ("focal_zero", 300, 0.0)]
    specs += [("outliers", n, r) for r in REGIME_OUTLIER_RATIOS for n in (21, 2048, 4097)]
    out = []
    for i, (kind, n, ratio) in enumerate(specs):
        p = regime_pair(kind, n, rng, ratio, REGIME_THRESHOLDS[i % len(REGIME_THRESHOLDS)])
        out.append((f"{kind}-{n}-{ratio}", p["corr"], p["thr"], hypotheses_for(i, p["good"], p["bad"])))
    return out
