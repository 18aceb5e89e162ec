"""Synthetic scene generator + binary container (SURVEY App. D).

Replaces the reference's on-disk inputs (1DSfM `list_with_focals.txt`, `image_data.h5`, `keypoints.h5`,
`correspondences.h5`, similarity-matrix text; utils.h:122-182, feature_utils.h:27-133,
imagesimilarity_graph.h:108-171), none of which can be read here (no HDF5, no images).

A scene is a dict of numpy arrays:
  focal[V] f64, size[V,2] f64 (width,height), sim[V,V] f64 (3 decimals, diag 1.0, never 1.0 off-diag),
  kp_offset[V+1] u64, kp[sum K,2] f32 pixel keypoints (cv::KeyPoint.pt is float),
  pair_views[P,2] u32 (src<dst as the similarity queue emits them), m_offset[P+1] u64,
  matches[sum N,2] u32 (srcIdx,dstIdx) in the order matchFeatures would emit (sorted by ratio = shuffled),
  gt_q[V,4]/gt_t[V,3] world->camera ground truth (accuracy reporting only).
A descriptor scene (make_descriptor_scene; the reference's keypoints.h5) has desc[sum K,dim] f32 row-aligned with kp and
no matches until they are computed (Engine.register_scene_descriptors fills m_offset, matches and ratios[sum N] f64).
"""
import struct

import numpy as np

MAGIC = b"PGISCN01"
MAGIC_V2 = b"PGISCN02"  # + descriptors, matches and ratios optional


def _rot_look_at(cam_pos, target, up=np.array([0.0, 0.0, 1.0])):
    z = target - cam_pos
    z = z / np.linalg.norm(z)
    x = np.cross(z, up)
    x = x / np.linalg.norm(x)
    y = np.cross(z, x)
    return np.stack([x, y, z])  # rows = camera axes in world coords  (world->camera rotation)


def make_scene(n_views=50, n_corr=1000, outlier_ratio=0.3, seed=0, n_points=4000, focal=800.0, width=1600.0,
               height=1200.0, noise_px=0.5, radius=6.0, overlap_knn=None, overlap_outlier_ratio=None,
               max_pairs=None, arc=2.0 * np.pi):
    """Cameras on a ring (arc radians) looking at a Gaussian blob; every view detects all n_points (noisy,
    FP32).  Every i<j pair gets n_corr matches, `outlier_ratio` of them wrong.  If overlap_knn is given,
    only pairs within that ring distance share points (others are 100 % outliers; SURVEY §8d cfg 4)."""
    rng = np.random.default_rng(seed)
    V = n_views
    pts = rng.standard_normal((n_points, 3))
    ang = np.arange(V) * (arc / V) + rng.uniform(-0.2, 0.2, V) * (arc / V)
    elev = rng.uniform(-0.25, 0.25, V)
    rad = radius * (1.0 + rng.uniform(-0.15, 0.15, V))
    cam = np.stack([rad * np.cos(ang) * np.cos(elev), rad * np.sin(ang) * np.cos(elev), rad * np.sin(elev)], 1)
    Rw = np.stack([_rot_look_at(cam[v], rng.standard_normal(3) * 0.15) for v in range(V)])
    tw = -np.einsum("vij,vj->vi", Rw, cam)
    # keypoints: view v stores point pid at index perm[v][pid]
    kp = np.empty((V, n_points, 2), dtype=np.float32)
    perm = np.empty((V, n_points), dtype=np.uint32)
    for v in range(V):
        Xc = pts @ Rw[v].T + tw[v]
        uv = focal * Xc[:, :2] / Xc[:, 2:3] + np.array([width / 2.0, height / 2.0])
        uv = uv + rng.standard_normal(uv.shape) * noise_px
        p = rng.permutation(n_points).astype(np.uint32)
        perm[v] = p
        kp[v, p] = uv.astype(np.float32)
    view_dir = Rw[:, 2, :]
    sim = np.clip(view_dir @ view_dir.T, 0.0, 0.999)
    sim = np.round(sim, 3)
    sim = np.minimum(sim, 0.999)
    sim = (sim + sim.T) / 2.0
    sim = np.round(sim, 3)
    np.fill_diagonal(sim, 1.0)

    iu, ju = np.triu_indices(V, 1)
    if max_pairs is not None and len(iu) > max_pairs:
        # keep the most similar pairs (what a similarity threshold would do); ties by queue order
        s = sim[iu, ju]
        order = np.lexsort((-ju, -iu, -s))[:max_pairs]
        order.sort()
        iu, ju = iu[order], ju[order]
    P = len(iu)
    pair_views = np.stack([iu, ju], 1).astype(np.uint32)
    N = n_corr
    m_offset = (np.arange(P + 1, dtype=np.uint64) * np.uint64(N))
    matches = np.empty((P * N, 2), dtype=np.uint32)
    # per pair: N distinct point ids = (a + b k) mod n_points, b odd & coprime (n_points power-of-two friendly
    # is not required: we pick b from primes not dividing n_points)
    primes = np.array([p for p in (7919, 6007, 4099, 3001, 2003, 1009, 911, 727, 523, 317) if n_points % p], dtype=np.int64)
    chunk = max(1, (1 << 24) // max(N, 1))
    ring = np.minimum((ju - iu) % V, (iu - ju) % V)
    for c0 in range(0, P, chunk):
        c1 = min(P, c0 + chunk)
        n = c1 - c0
        a = rng.integers(0, n_points, (n, 1))
        b = primes[rng.integers(0, len(primes), (n, 1))]
        ids = (a + b * np.arange(N)[None, :]) % n_points
        rho = np.full((n, 1), outlier_ratio)
        if overlap_knn is not None:
            far = ring[c0:c1, None] > overlap_knn
            rho = np.where(far, 1.0, overlap_outlier_ratio if overlap_outlier_ratio is not None else outlier_ratio)
        is_out = rng.random((n, N)) < rho
        wrong = (ids + 1 + rng.integers(0, n_points - 1, (n, N))) % n_points
        dst_ids = np.where(is_out, wrong, ids)
        src = np.take_along_axis(perm[iu[c0:c1]], ids, 1)
        dst = np.take_along_axis(perm[ju[c0:c1]], dst_ids, 1)
        matches[c0 * N:c1 * N, 0] = src.reshape(-1)
        matches[c0 * N:c1 * N, 1] = dst.reshape(-1)
    # ground truth as quaternions (x,y,z,w)
    gt_q = np.empty((V, 4))
    for v in range(V):
        gt_q[v] = _quat_from_rot(Rw[v])
    return dict(focal=np.full(V, focal), size=np.tile(np.array([width, height]), (V, 1)), sim=sim,
                kp_offset=(np.arange(V + 1, dtype=np.uint64) * np.uint64(n_points)), kp=kp.reshape(-1, 2),
                pair_views=pair_views, m_offset=m_offset, matches=matches, gt_q=gt_q, gt_t=tw.copy(),
                gt_R=Rw.copy())


def _quat_from_rot(R):
    t = np.trace(R)
    if t > 0:
        s = np.sqrt(t + 1.0) * 2
        return np.array([(R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s, 0.25 * s])
    i = int(np.argmax(np.diag(R)))
    j, k = (i + 1) % 3, (i + 2) % 3
    s = np.sqrt(R[i, i] - R[j, j] - R[k, k] + 1.0) * 2
    q = np.zeros(4)
    q[i] = 0.25 * s
    q[3] = (R[k, j] - R[j, k]) / s
    q[j] = (R[j, i] + R[i, j]) / s
    q[k] = (R[k, i] + R[i, k]) / s
    return q


def relative_gt(scene, src, dst):
    """Ground-truth T_dst_src = T_dst_world * T_world_src as (R, t)."""
    Rs, Rd = scene["gt_R"][src], scene["gt_R"][dst]
    ts, td = scene["gt_t"][src], scene["gt_t"][dst]
    R = Rd @ Rs.T
    return R, td - R @ ts


def pair_correspondences(scene, p, thr_px=0.4):
    """createCorrespondenceMatrix (pose_graph_builder.h:864-938) for pair index p, in numpy — used by tests
    to feed single pairs through the C-ABI.  (x - w_src/2)/f_src for BOTH images (SURVEY §0.8)."""
    src, dst = (int(x) for x in scene["pair_views"][p])
    m = scene["matches"][int(scene["m_offset"][p]):int(scene["m_offset"][p + 1])]
    ks = scene["kp"][int(scene["kp_offset"][src]):int(scene["kp_offset"][src + 1])]
    kd = scene["kp"][int(scene["kp_offset"][dst]):int(scene["kp_offset"][dst + 1])]
    f = scene["focal"][src]
    c = scene["size"][src] / 2.0
    a = ks[m[:, 0]].astype(np.float64)
    b = kd[m[:, 1]].astype(np.float64)
    corr = np.concatenate([(a - c) / f, (b - c) / f], 1)
    return np.ascontiguousarray(corr), thr_px / ((f + f + f + f) / 4.0)


CONFIGS = {
    # BASELINE.json configs / SURVEY §8d table; seeds = config index
    "cfg1_50v": dict(n_views=50, n_corr=1000, outlier_ratio=0.3, seed=1),
    "cfg2_300v": dict(n_views=300, n_corr=2000, outlier_ratio=0.3, seed=2),
    "cfg3_1000v": dict(n_views=1000, n_corr=2000, outlier_ratio=0.4, seed=3),
    "cfg4_sparse": dict(n_views=300, n_corr=2000, outlier_ratio=0.7, seed=4, overlap_knn=6, overlap_outlier_ratio=0.7),
    "cfg5_5000v": dict(n_views=5000, n_corr=4000, outlier_ratio=0.4, seed=5, max_pairs=2_000_000),
}


def make_descriptor_scene(n_views=12, kp_range=(600, 2500), dim=128, seed=0, n_points=None, kp_counts=None, focal=800.0,
                          width=1600.0, height=1200.0, noise_px=0.5, desc_noise=0.05, distractor_ratio=0.3, radius=6.0,
                          arc=2.0 * np.pi, visible_half_angle=0.5 * np.pi):
    """Keypoints and descriptors of every view, no matches (what matchFeatures starts from).  Cameras on a ring as in
    make_scene.  Every 3-D point faces a random azimuth and is detectable only from cameras within visible_half_angle of
    it, so overlap falls with the ring distance and far pairs end below kMinimumPointNumber.  View v keeps kp_counts[v]
    keypoints (default: uniform in kp_range): a random subset of its detectable points plus distractor_ratio of unrelated
    keypoints, in its own shuffled order.  A point's descriptor is a unit vector plus per-view Gaussian noise (desc_noise
    per dimension, as tests/helpers.two_view_keypoints); a distractor's is an unrelated unit vector.  gt_point[sum K] holds
    the 3-D point of each keypoint (-1 for distractors).  Uses its own RNG stream: make_scene is unaffected."""
    rng = np.random.default_rng(seed)
    V = n_views
    counts = (np.asarray(kp_counts, dtype=np.int64) if kp_counts is not None
              else rng.integers(int(kp_range[0]), int(kp_range[1]) + 1, V))
    assert len(counts) == V
    if n_points is None:
        n_points = max(64, 2 * int(counts.max()) if V else 64)
    pts = rng.standard_normal((n_points, 3))
    facing = rng.uniform(0.0, 2.0 * np.pi, n_points)
    base = rng.standard_normal((n_points, dim))
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    ang = np.arange(V) * (arc / max(V, 1)) + rng.uniform(-0.2, 0.2, V) * (arc / max(V, 1))
    elev = rng.uniform(-0.25, 0.25, V)
    rad = radius * (1.0 + rng.uniform(-0.15, 0.15, V))
    cam = np.stack([rad * np.cos(ang) * np.cos(elev), rad * np.sin(ang) * np.cos(elev), rad * np.sin(elev)], 1)
    Rw = np.stack([_rot_look_at(cam[v], rng.standard_normal(3) * 0.15) for v in range(V)]) if V else np.zeros((0, 3, 3))
    tw = -np.einsum("vij,vj->vi", Rw, cam)
    kps, descs, pids = [], [], []
    for v in range(V):
        dphi = np.abs((facing - ang[v] + np.pi) % (2.0 * np.pi) - np.pi)
        vis = np.flatnonzero(dphi < visible_half_angle)
        n_real = min(len(vis), int(round(counts[v] * (1.0 - distractor_ratio))))
        real = rng.choice(vis, n_real, replace=False) if n_real else np.zeros(0, dtype=np.int64)
        m = int(counts[v]) - n_real
        Xc = pts[real] @ Rw[v].T + tw[v]
        uv = focal * Xc[:, :2] / Xc[:, 2:3] + np.array([width / 2.0, height / 2.0]) + rng.standard_normal((n_real, 2)) * noise_px
        d = base[real] + rng.standard_normal((n_real, dim)) * desc_noise
        de = rng.standard_normal((m, dim))
        de /= np.linalg.norm(de, axis=1, keepdims=True)
        uv = np.vstack([uv, rng.uniform([0.0, 0.0], [width, height], (m, 2))])
        d = np.vstack([d, de])
        pid = np.concatenate([real, np.full(m, -1)])
        order = rng.permutation(int(counts[v]))
        kps.append(uv[order].astype(np.float32)); descs.append(d[order].astype(np.float32)); pids.append(pid[order])
    view_dir = Rw[:, 2, :]
    sim = np.round(np.minimum(np.clip(view_dir @ view_dir.T, 0.0, 0.999), 0.999), 3)
    sim = np.round((sim + sim.T) / 2.0, 3)
    np.fill_diagonal(sim, 1.0)
    iu, ju = np.triu_indices(V, 1)
    gt_q = np.array([_quat_from_rot(Rw[v]) for v in range(V)]).reshape(V, 4)
    return dict(focal=np.full(V, focal), size=np.tile(np.array([width, height]), (V, 1)), sim=sim,
                kp_offset=np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64),
                kp=np.concatenate(kps).reshape(-1, 2) if V else np.zeros((0, 2), dtype=np.float32),
                desc=np.concatenate(descs).reshape(-1, dim) if V else np.zeros((0, dim), dtype=np.float32),
                pair_views=np.stack([iu, ju], 1).astype(np.uint32), gt_q=gt_q, gt_t=tw.copy(), gt_R=Rw.copy(),
                gt_point=np.concatenate(pids).astype(np.int64) if V else np.zeros(0, dtype=np.int64))


def save_scene(path, scene):
    """Binary container of SURVEY App. D: header + arrays, little-endian.  A scene with descriptors is written as
    version 2 (PGISCN02: the version-1 header plus dim and which of matches / ratios follow, then desc and those); any
    other scene as version 1, byte for byte as before."""
    V, P = len(scene["focal"]), len(scene["pair_views"])
    if "desc" in scene:
        desc = np.ascontiguousarray(scene["desc"], dtype="<f4")
        has_m = "matches" in scene and "m_offset" in scene
        has_r = has_m and "ratios" in scene
        M = len(scene["matches"]) if has_m else 0
        with open(path, "wb") as f:
            f.write(MAGIC_V2)
            f.write(struct.pack("<QQQQQQ", V, P, len(scene["kp"]), M, desc.shape[1], int(has_m) | int(has_r) << 1))
            for key, dt in (("focal", "<f8"), ("size", "<f8"), ("sim", "<f8"), ("kp_offset", "<u8"), ("kp", "<f4"),
                            ("pair_views", "<u4")):
                f.write(np.ascontiguousarray(scene[key], dtype=dt).tobytes())
            f.write(desc.tobytes())
            if has_m:
                f.write(np.ascontiguousarray(scene["m_offset"], dtype="<u8").tobytes())
                f.write(np.ascontiguousarray(scene["matches"], dtype="<u4").tobytes())
            if has_r:
                f.write(np.ascontiguousarray(scene["ratios"], dtype="<f8").tobytes())
        return
    with open(path, "wb") as f:
        f.write(MAGIC)
        f.write(struct.pack("<QQQQ", V, P, len(scene["kp"]), len(scene["matches"])))
        for key, dt in (("focal", "<f8"), ("size", "<f8"), ("sim", "<f8"), ("kp_offset", "<u8"), ("kp", "<f4"),
                        ("pair_views", "<u4"), ("m_offset", "<u8"), ("matches", "<u4")):
            f.write(np.ascontiguousarray(scene[key], dtype=dt).tobytes())


def load_scene(path):
    with open(path, "rb") as f:
        magic = f.read(8)
        assert magic in (MAGIC, MAGIC_V2), "not a PGI scene container"

        def rd(dt, shape):
            n = int(np.prod(shape))
            return np.frombuffer(f.read(n * np.dtype(dt).itemsize), dtype=dt).reshape(shape).copy()

        if magic == MAGIC_V2:
            V, P, K, M, D, flags = struct.unpack("<QQQQQQ", f.read(48))
            sc = dict(focal=rd("<f8", (V,)), size=rd("<f8", (V, 2)), sim=rd("<f8", (V, V)), kp_offset=rd("<u8", (V + 1,)),
                      kp=rd("<f4", (K, 2)), pair_views=rd("<u4", (P, 2)), desc=rd("<f4", (K, D)))
            if flags & 1:
                sc["m_offset"], sc["matches"] = rd("<u8", (P + 1,)), rd("<u4", (M, 2))
            if flags & 2:
                sc["ratios"] = rd("<f8", (M,))
            return sc
        V, P, K, M = struct.unpack("<QQQQ", f.read(32))
        return dict(focal=rd("<f8", (V,)), size=rd("<f8", (V, 2)), sim=rd("<f8", (V, V)),
                    kp_offset=rd("<u8", (V + 1,)), kp=rd("<f4", (K, 2)), pair_views=rd("<u4", (P, 2)),
                    m_offset=rd("<u8", (P + 1,)), matches=rd("<u4", (M, 2)))


# ---- the reference's two plain-text inputs (the HDF5 caches cannot be read here: no HDF5 in this image) ------------------
def load_1dsfm_image_list(path):
    """load1DSfMImageList (utils.h:120-182) without the image-size pass: every line of `list_with_focals.txt` is
    `images/<name> <flag> <focal>`; the name drops its first 7 characters (utils.h:149), the third token is the focal
    length (std::atof, :154).  A line without a third token keeps an indeterminate focal length in the reference; it is
    reported as 0.0 here.  Returns (names, focal[V])."""
    names, focal = [], []
    with open(path) as f:
        for line in f:  # the reference counts and keeps every line, also empty ones (:137-170)
            tok = line.split()
            names.append(tok[0][7:] if tok else "")
            try:
                focal.append(float(tok[2]) if len(tok) > 2 else 0.0)
            except ValueError:
                focal.append(0.0)  # std::atof of a non-number
    return names, np.asarray(focal, dtype=np.float64)


def load_similarity_matrix(path, n_views):
    """SimilarityTable::loadFromFile (imagesimilarity_graph.h:108-171): one whitespace-separated row per line; the file must
    have exactly n_views rows of n_views values (the reference logs and returns false otherwise: ValueError here).  The
    similarity-ordered pair queue the reference builds while reading (:141-157) is built by pgb_create from the returned
    matrix.  Returns sim[V, V] float64."""
    rows = []
    with open(path) as f:
        for line in f:
            vals = []
            for tok in line.split():
                try:
                    vals.append(float(tok))
                except ValueError:
                    break  # `ss >> value` stops at the first token that is not a number
            rows.append(vals)
    if len(rows) != n_views or any(len(r) != n_views for r in rows):
        raise ValueError("%s has different size than the initialised similarity map (%d views)" % (path, n_views))
    return np.asarray(rows, dtype=np.float64)


def save_similarity_matrix(path, sim):
    with open(path, "w") as f:
        for row in np.asarray(sim):
            f.write(" ".join(repr(float(x)) for x in row) + "\n")
