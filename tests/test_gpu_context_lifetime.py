"""Lifetime of the engine context's device memory: a context that shares another's pairs reads the owner's
registration and stops reading it once it registers its own, and a context gives back everything it allocated when it
is closed, whichever entry points it used."""
import numpy as np
import pytest
import torch

from helpers import pose_qt, two_view, two_view_keypoints
from pose_graph_initialization_b200 import Engine
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import ADJ_ENTRY_DTYPE, QUERY_DTYPE, WAVE_FALLBACK, WAVE_PATH

pytestmark = pytest.mark.gpu


def _dense_pairs(sc, thr_px=0.4):
    parts = [S.pair_correspondences(sc, p, thr_px) for p in range(len(sc["pair_views"]))]
    offset = np.zeros(len(parts) + 1, dtype=np.uint64)
    offset[1:] = np.cumsum([len(c) for c, _ in parts])
    return np.concatenate([c for c, _ in parts]), offset, np.array([t for _, t in parts])


def test_a_shared_context_sees_the_owners_registration():
    sc = S.make_scene(n_views=8, n_corr=300, outlier_ratio=0.3, seed=41, n_points=900)
    owner, borrower = Engine(device=0), Engine(device=0, background=True)
    try:
        owner.register_scene(sc, 0.4)
        borrower.share_pairs(owner)
        pids = np.arange(12, dtype=np.uint32)
        flags = WAVE_PATH | WAVE_FALLBACK
        v_own, m_own = owner.run_wave(pids, flags=flags, want_masks=True)
        v_bor, m_bor = borrower.run_wave(pids, flags=flags, want_masks=True)
        assert v_own["accepted"].any() and m_own.any()
        assert v_bor.tobytes() == v_own.tobytes() and m_bor.tobytes() == m_own.tobytes()
        shared = [owner.read_pair(p) for p in (0, 7)]
        assert all(np.array_equal(borrower.read_pair(p)[0], c) for p, (c, _) in zip((0, 7), shared))

        other = S.make_scene(n_views=5, n_corr=200, outlier_ratio=0.2, seed=42, n_points=600)
        corr, offset, thr = _dense_pairs(other)
        borrower.register_pairs(corr, offset, thr)
        for p, (c, t) in zip((0, 7), shared):
            c2, t2 = owner.read_pair(p)
            assert c2.tobytes() == c.tobytes() and t2 == t
        v2, m2 = owner.run_wave(pids, flags=flags, want_masks=True)
        assert v2.tobytes() == v_own.tobytes() and m2.tobytes() == m_own.tobytes()
        c0, t0 = borrower.read_pair(0)
        assert c0.tobytes() == corr[: int(offset[1])].tobytes() and t0 == thr[0]
    finally:
        borrower.close()
        owner.close()


def _big_scene(base, rows=1 << 25, n_big=32):
    """base plus n_big pairs of views 0 and 1 with rows correspondences in all: 32 bytes each on the device (1 GiB)."""
    sc = dict(base)
    k0 = int(base["kp_offset"][1] - base["kp_offset"][0])
    k1 = int(base["kp_offset"][2] - base["kp_offset"][1])
    i = np.arange(rows, dtype=np.uint64)
    big = np.stack([i % k0, (7 * i) % k1], 1).astype(np.uint32)
    end = int(base["m_offset"][-1])
    sc["pair_views"] = np.concatenate([base["pair_views"], np.tile(np.array([[0, 1]], dtype=np.uint32), (n_big, 1))])
    sc["m_offset"] = np.concatenate([base["m_offset"], end + (rows // n_big) * np.arange(1, n_big + 1, dtype=np.uint64)])
    sc["matches"] = np.concatenate([base["matches"], big])
    return sc


def _one_cycle(big, desc_scene, inputs):
    eng = Engine(device=0)
    try:
        eng.register_scene(big, 0.4)
        verdicts, masks = eng.run_wave(np.arange(8, dtype=np.uint32), want_masks=True)
        assert len(verdicts) == 8 and masks.any()
        eng.register_scene_descriptors(desc_scene)
        assert int(desc_scene["m_offset"][-1]) > 0

        V = 8
        eng.graph_init(np.full((V, V), 0.5))
        entries = np.zeros(4, dtype=ADJ_ENTRY_DTYPE)
        for k, (v, idx, nxt) in enumerate(((0, 0, 1), (1, 0, 0), (1, 1, 2), (2, 0, 1))):
            entries[k] = (v, idx, nxt, 0, 0.5)
        counts = np.array([1, 2, 1, 0, 0, 0, 0, 0], dtype=np.uint32)
        eng.graph_apply(entries, counts, counts)
        res, _ = eng.graph_search(np.array([(0, 2, 0, 0)], dtype=QUERY_DTYPE))
        assert len(res) == 1

        d = inputs["keypoints"]
        eng.guided_match(d["kp_src"], d["desc_src"], d["kp_dst"], d["desc_dst"], d["pose"], d["K"], d["K"], d["size"], d["size"])
        m, _ = eng.match_features(d["desc_src"], d["desc_dst"])
        assert len(m) > 0
        corr, E = inputs["corr"], inputs["E"]
        eng.estimate_pose(corr, 0.4 / 800.0)
        eng.dbg_sampson(corr, E)
        eng.dbg_five_point(corr[:5, :2].reshape(1, 10), corr[:5, 2:].reshape(1, 10))
        eng.dbg_pose_from_essential(E, corr)
        eng.fp64_peak()
    finally:
        eng.close()


def test_contexts_give_their_memory_back(oracle):
    base = S.make_scene(n_views=6, n_corr=300, outlier_ratio=0.3, seed=43, n_points=900)
    big = _big_scene(base)
    desc_scene = S.make_descriptor_scene(6, kp_range=(200, 500), seed=44, n_points=400)
    rng = np.random.default_rng(45)
    corr, R, t = two_view(400, 0.3, rng)
    inputs = dict(keypoints=two_view_keypoints(300, rng), corr=corr, E=oracle.essential_from_pose(pose_qt(R, t)))
    torch.cuda.init()
    _one_cycle(big, dict(desc_scene), inputs)  # warm-up: loads the kernels and sizes the driver's own pools
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(6):
        _one_cycle(big, dict(desc_scene), inputs)
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free0 - free1 < 512 << 20, (free0, free1)
