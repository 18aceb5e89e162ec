"""Descriptor scenes on the CPU: make_descriptor_scene (deterministic, ragged, some pairs below kMinimumPointNumber, and
make_scene's stream untouched), the version-2 container carrying descriptors / matches / ratios while version-1 files
load as before, and two gloo ranks that each match only the pairs they own (stand-in engine matching with
oracle.match_features), all-gather the per-pair counts into the global m_offset and commit what one rank commits."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _small(seed=7):
    from pose_graph_initialization_b200 import scene as S
    return S.make_descriptor_scene(8, kp_range=(120, 400), seed=seed, n_points=500)


def _oracle_full(sc):
    from oracle import pgo_oracle as O
    ko = sc["kp_offset"].astype(np.int64)
    res = [O.match_features(sc["desc"][ko[s]:ko[s + 1]], sc["desc"][ko[d]:ko[d + 1]]) for s, d in sc["pair_views"]]
    full = dict(sc)
    full["m_offset"] = np.concatenate([[0], np.cumsum([len(m) for m, _ in res])]).astype(np.uint64)
    full["matches"] = np.concatenate([m for m, _ in res]).reshape(-1, 2).astype(np.uint32)
    full["ratios"] = np.concatenate([r for _, r in res])
    return full


def test_descriptor_scene_is_deterministic_ragged_and_has_weak_pairs(oracle):
    from pose_graph_initialization_b200 import scene as S

    a, b = _small(), _small()
    assert set(a) == set(b) and "matches" not in a and "m_offset" not in a
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["desc"], _small(8)["desc"])
    k = np.diff(a["kp_offset"].astype(np.int64))
    assert len(np.unique(k)) > 4 and k.sum() == len(a["kp"]) == len(a["desc"]) == len(a["gt_point"])
    assert a["desc"].dtype == np.float32 and a["desc"].shape[1] == 128 and a["kp"].dtype == np.float32
    assert len(a["pair_views"]) == 28 and a["sim"].shape == (8, 8)
    full = _oracle_full(a)
    n = np.diff(full["m_offset"].astype(np.int64))
    assert (n < 50).any() and (n >= 50).any()  # some pairs fall below kMinimumPointNumber, others pass
    # the matches are mostly the same 3-D point seen twice
    ko = a["kp_offset"].astype(np.int64)
    good = total = 0
    for p, (s, d) in enumerate(a["pair_views"]):
        m = full["matches"][full["m_offset"][p]:full["m_offset"][p + 1]].astype(np.int64)
        ps, pd = a["gt_point"][ko[s] + m[:, 0]], a["gt_point"][ko[d] + m[:, 1]]
        good += int(((ps == pd) & (ps >= 0)).sum())
        total += len(m)
    assert good > 0.9 * total
    # 64 dimensions and explicit counts
    c = S.make_descriptor_scene(3, dim=64, seed=1, kp_counts=[0, 1, 5])
    assert c["desc"].shape == (6, 64) and list(c["kp_offset"]) == [0, 0, 1, 6]


def test_make_scene_is_unchanged_by_the_descriptor_generator():
    from pose_graph_initialization_b200 import scene as S

    a = S.make_scene(n_views=5, n_corr=60, outlier_ratio=0.3, seed=3, n_points=200)
    _small()
    b = S.make_scene(n_views=5, n_corr=60, outlier_ratio=0.3, seed=3, n_points=200)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_container_round_trip_of_descriptors(tmp_path, oracle):
    from pose_graph_initialization_b200 import scene as S

    sc = _small()
    p = str(tmp_path / "d.pgi")
    S.save_scene(p, sc)
    back = S.load_scene(p)
    assert set(back) == {"focal", "size", "sim", "kp_offset", "kp", "pair_views", "desc"}
    for k in back:
        assert np.array_equal(np.asarray(sc[k]), back[k]), k
    full = _oracle_full(sc)
    S.save_scene(p, full)
    back = S.load_scene(p)
    for k in ("desc", "m_offset", "matches", "ratios", "kp", "pair_views"):
        assert np.asarray(full[k]).tobytes() == back[k].astype(np.asarray(full[k]).dtype).tobytes(), k
    # a scene without descriptors is still written as version 1, byte for byte as before
    old = S.make_scene(n_views=4, n_corr=30, outlier_ratio=0.3, seed=2, n_points=100)
    q = str(tmp_path / "o.pgi")
    S.save_scene(q, old)
    raw = open(q, "rb").read()
    assert raw[:8] == b"PGISCN01"
    V, P, K, M = 4, 6, 400, 180
    assert len(raw) == 8 + 32 + V * 8 + V * 16 + V * V * 8 + (V + 1) * 8 + K * 8 + P * 8 + (P + 1) * 8 + M * 8
    back = S.load_scene(q)
    assert set(back) == {"focal", "size", "sim", "kp_offset", "kp", "pair_views", "m_offset", "matches"}
    for k in back:
        assert np.array_equal(np.asarray(old[k]), back[k]), k


class StandInEngine:
    """register_scene_descriptors with oracle.match_features (tests only); records which pairs it matched."""

    def __init__(self):
        self.matched = []

    def register_scene_descriptors(self, scene, thr_px=0.4):
        full = _oracle_full(scene)
        self.matched.extend(map(tuple, np.asarray(scene["pair_views"]).tolist()))
        for k in ("m_offset", "matches", "ratios"):
            scene[k] = full[k]
        return full["m_offset"]

    def register_scene(self, scene, thr_px=0.4):
        raise AssertionError("a descriptor scene is registered by matching it")


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT); sys.path.insert(0, HERE)
    import torch.distributed as dist

    from oracle import pgo_oracle as O
    from oracle_engine import OracleEngine
    from pose_graph_initialization_b200 import builder as B

    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sc = _small(9)
    P = len(sc["pair_views"])
    pgb = B.PoseGraphBuilder(kSimilarityThreshold_=0.0, scene=sc, overlap_fallback=False, rank=rank, world_size=world)
    stand_in = StandInEngine()
    pgb.engine = stand_in
    pgb.prepare()
    # only the owned pairs were matched; the global m_offset is every rank's
    assert stand_in.matched == [tuple(v) for v in sc["pair_views"][rank::world].tolist()]
    assert "matches" not in sc and len(sc["m_offset"]) == P + 1
    full = _oracle_full(sc)
    assert np.array_equal(sc["m_offset"], full["m_offset"])
    assert np.array_equal(pgb._sub["matches"], B.shard_scene(full, rank, world)["matches"])
    # the wave loop of the multi-rank host on the global m_offset, verdicts for owned positions only
    eng = OracleEngine(O, full)
    host = B.HostBuilder(sc, similarity_threshold=0.0, host_threads=2, lazy_fallback=False)
    mine_ids = np.arange(rank, P, world)
    mine = np.zeros(len(mine_ids), dtype=B.VERDICT_DTYPE)
    for k, p in enumerate(mine_ids):
        mine[k] = eng.verdict(int(p), None, path=False, fallback=True)
    parts = B.allgather_verdicts(mine, [len(range(r, P, world)) for r in range(world)])
    allv = np.zeros(P, dtype=B.VERDICT_DTYPE)
    for r in range(world):
        allv[r::world] = parts[r]
    host.set_fallback_verdicts(allv)
    host.set_partition(rank, world)
    while host.remaining() > 0:
        items = host.next_wave(16)
        status = host.wave_status()
        while status != B.WAVE_DONE:
            if status == B.WAVE_NEED_GPU:
                host.commit_wave(eng.run_items(items[items["need_gpu"] > 0], path=True, fallback=False))
            else:
                host.import_records(B.allreduce_records(host.export_records()))
            status = host.wave_status()
            if status != B.WAVE_DONE:
                items = host.next_wave(16)
    edges = host.edges()
    olog, ostats = O.run_scene(full, sim_threshold=0.0)
    committed = olog[olog["committed"] > 0]
    ok = (len(edges) == ostats["edges"] > 0 and np.array_equal(edges["src"], committed["src"])
          and np.array_equal(edges["dst"], committed["dst"]) and np.array_equal(edges["q"], committed["q"])
          and np.array_equal(edges["score"], committed["score"]))
    ret[rank] = (bool(ok), edges.tobytes())
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_match_their_own_pairs_and_commit_the_sequential_graph():
    world = 2
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0
    assert ret[0][0] and ret[1][0] and ret[0][1] == ret[1][1]
