"""Batched descriptor matching on the device (K9, pgi_register_scene_descriptors): every pair's matches and ratio bits equal
oracle.match_features (at full size too, where pgi_match_features must agree), the registration built from the device-resident matches equals the one
built from the oracle's, and PoseGraphBuilder on a keypoints + descriptors scene commits what the sequential oracle
commits on the same scene matched by oracle.match_features."""
import multiprocessing as mp
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S
from pose_graph_initialization_b200.engine import Engine, PgiError

pytestmark = pytest.mark.gpu


def _oracle_pair(args):
    from oracle import pgo_oracle as O
    return O.match_features(*args)


def oracle_matches(sc):
    """oracle.match_features of every pair (a process pool: the numpy restatement takes seconds per pair)."""
    ko = sc["kp_offset"].astype(np.int64)
    jobs = [(sc["desc"][ko[s]:ko[s + 1]], sc["desc"][ko[d]:ko[d + 1]]) for s, d in sc["pair_views"]]
    with ProcessPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1)), mp_context=mp.get_context("fork")) as ex:
        res = list(ex.map(_oracle_pair, jobs, chunksize=1))
    n = np.array([len(m) for m, _ in res], dtype=np.int64)
    full = dict(sc)
    full["m_offset"] = np.concatenate([[0], np.cumsum(n)]).astype(np.uint64)
    full["matches"] = np.concatenate([m for m, _ in res]).reshape(-1, 2).astype(np.uint32)
    full["ratios"] = np.concatenate([r for _, r in res]).astype(np.float64)
    return full


def edge_case_scene(dim, seed):
    """~12 views, 600-2 500 keypoints (not multiples of the 128-row tiles), one view with no keypoint, one with one, and
    one whose descriptors are small integers (exact distance ties)."""
    counts = np.array([1537, 0, 2431, 1, 611, 1999, 1280, 2500, 703, 1025, 129, 1871])
    sc = S.make_descriptor_scene(len(counts), dim=dim, seed=seed, kp_counts=counts)
    ko = sc["kp_offset"].astype(np.int64)
    v = 4
    sc["desc"][ko[v]:ko[v + 1]] = np.round(sc["desc"][ko[v]:ko[v + 1]] * 3.0)
    return sc


@pytest.fixture(scope="module", params=[128, 64])
def matched(request):
    sc = edge_case_scene(request.param, seed=40 + request.param)
    ref = oracle_matches(sc)
    eng = Engine(device=0)
    dev = dict(sc)
    mo = eng.register_scene_descriptors(dev, 0.4)
    yield sc, ref, dev, eng, mo
    eng.close()


def test_matches_and_ratio_bits_equal_the_oracle(matched):
    sc, ref, dev, eng, mo = matched
    assert np.array_equal(mo, ref["m_offset"])
    assert np.array_equal(dev["matches"], ref["matches"])
    assert dev["ratios"].tobytes() == ref["ratios"].tobytes()
    n = np.diff(mo.astype(np.int64))
    assert (n == 0).any() and (n > 0).any()  # the 0- and 1-keypoint views' pairs are empty, others are not
    st = eng.stats()
    ko = sc["kp_offset"].astype(np.int64)
    k = np.diff(ko)
    assert st["dist_evals"] == int(sum(k[s] * k[d] for s, d in sc["pair_views"]))
    assert st["match_pairs"] == len(sc["pair_views"]) and st["match_rows"] == int(mo[-1]) and st["ms_match"] > 0


def test_registration_from_device_matches(matched):
    sc, ref, dev, eng, mo = matched
    for p in range(len(sc["pair_views"])):
        corr, thr = eng.read_pair(p)
        rc, rthr = S.pair_correspondences(ref, p, 0.4)
        assert np.array_equal(corr, rc) and thr == rthr, p


def test_matches_equal_the_oracle_at_full_size():
    sc = S.make_descriptor_scene(40, kp_range=(4000, 4000), seed=41)
    eng = Engine(device=0)
    dev = dict(sc)
    mo = eng.register_scene_descriptors(dev, 0.4).astype(np.int64)
    rng = np.random.default_rng(0)
    pairs = rng.choice(len(sc["pair_views"]), 60, replace=False)
    ref = oracle_matches(dict(sc, pair_views=sc["pair_views"][pairs]))
    ro = ref["m_offset"].astype(np.int64)
    ko = sc["kp_offset"].astype(np.int64)
    for k, p in enumerate(pairs):
        s, d = sc["pair_views"][p]
        m, r = eng.match_features(sc["desc"][ko[s]:ko[s + 1]], sc["desc"][ko[d]:ko[d + 1]])
        for got_m, got_r in ((dev["matches"][mo[p]:mo[p + 1]], dev["ratios"][mo[p]:mo[p + 1]]), (m, r)):
            assert np.array_equal(got_m, ref["matches"][ro[k]:ro[k + 1]]), p
            assert got_r.tobytes() == ref["ratios"][ro[k]:ro[k + 1]].tobytes(), p
    eng.close()


@pytest.mark.parametrize("prefetch", [True, False])
def test_descriptor_scene_graph_identity(oracle, prefetch):
    sc = S.make_descriptor_scene(10, kp_range=(500, 900), seed=43)
    ref = oracle_matches(sc)
    olog, ostats = oracle.run_scene(ref, sim_threshold=0.0)
    assert ostats["edges"] > 0 and (np.diff(ref["m_offset"].astype(np.int64)) < 50).any()  # some below kMinimumPointNumber
    dsc = dict(sc)
    assert B.needs_matching(dsc)
    pgb = B.PoseGraphBuilder(kCoreNumber_=4, kSimilarityThreshold_=0.0, scene=dsc, prefetch_fallback=prefetch,
                             overlap_fallback=prefetch, wave_size=16, fallback_wave=32)
    graph = pgb.run()
    assert np.array_equal(dsc["matches"], ref["matches"]) and np.array_equal(dsc["m_offset"], ref["m_offset"])
    plog = pgb.log
    assert len(plog) == len(olog)
    for f in ("src", "dst", "pairIndex", "visible", "hadPath", "testPassed", "branch", "committed", "testCount",
              "inlierNumber", "nCorr", "touchedNodes", "E", "q", "t", "score"):
        assert np.array_equal(plog[f], olog[f]), f
    committed = olog[olog["committed"] > 0]
    assert graph.numEdges() == ostats["edges"]
    assert np.array_equal(graph.edges["src"], committed["src"]) and np.array_equal(graph.edges["dst"], committed["dst"])
    assert np.array_equal(graph.edges["q"], committed["q"]) and np.array_equal(graph.edges["t"], committed["t"])
    assert np.array_equal(graph.edges["score"], committed["score"])
    pgb.close()


def test_bad_descriptor_inputs_are_rejected():
    sc = S.make_descriptor_scene(4, kp_range=(50, 80), seed=44)
    eng = Engine(device=0)
    bad = dict(sc, desc=np.ascontiguousarray(sc["desc"][:, :96]))
    with pytest.raises(PgiError, match="64 or 128"):
        eng.register_scene_descriptors(bad, 0.4)
    d = sc["desc"].copy()
    d[7, 3] = np.nan
    with pytest.raises(PgiError, match="non-finite"):
        eng.register_scene_descriptors(dict(sc, desc=d), 0.4)
    d[7, 3] = np.inf
    with pytest.raises(PgiError, match="non-finite"):
        eng.register_scene_descriptors(dict(sc, desc=d), 0.4)
    pv = sc["pair_views"].copy()
    pv[1, 1] = 4
    with pytest.raises(PgiError, match="out of range"):
        eng.register_scene_descriptors(dict(sc, pair_views=pv), 0.4)
    # the context is still usable after the rejections
    good = dict(sc)
    eng.register_scene_descriptors(good, 0.4)
    assert int(good["m_offset"][-1]) == len(good["matches"])
    eng.close()
