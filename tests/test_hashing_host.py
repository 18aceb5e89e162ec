"""Epipolar-hashing mode on the CPU: the C++ oracle's Tracklets (oracle/pgo_tracklets.hpp) against the Python restatement,
and the product's sequential hashing loop (pgb_run_hashing) against the oracle host's hashing branch
(pgo_run_scene_hashing).  The engine is a stand-in built on the oracle, behind the four function pointers the product
passes pgi_submit_wave, pgi_wait_wave, pgi_register_extra_pairs and pgi_guided_match_views through."""
import ctypes as C

import numpy as np
import pytest

from oracle import pgo_hashing
from oracle.pgo_tracklets import Tracklets as PyTracklets
from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S

CFG = dict(similarity_threshold=0.0, minimum_inlier_number=20, minimum_point_number=50, maximum_search_depth=5,
           traversal_heuristics_weight=0.8)
LOG_FIELDS = ("src", "dst", "pairIndex", "visible", "hadPath", "testPassed", "branch", "committed", "testCount",
              "inlierNumber", "nCorr", "touchedNodes", "E", "q", "t", "score")


# ---- the oracle's C++ Tracklets against oracle/pgo_tracklets.py -------------------------------------------------------
_TRACKLET_HARNESS = r"""
#include <cstdint>
#include <cstdio>
#include "pgo_tracklets.hpp"
// stdin: ops "a src dst n  s0 d0 m0 ..." (add) and "g src dst max" (getCorrespondences); stdout: one line per g
int main()
{
    pgo::Tracklets t;
    char op;
    while (std::scanf(" %c", &op) == 1) {
        if (op == 'a') {
            size_t s, d, n;
            std::scanf("%zu %zu %zu", &s, &d, &n);
            std::vector<std::pair<size_t, size_t>> m(n);
            std::vector<uint8_t> mask(n);
            for (size_t i = 0; i < n; i++) {
                unsigned k;
                std::scanf("%zu %zu %u", &m[i].first, &m[i].second, &k);
                mask[i] = (uint8_t)k;
            }
            t.add(s, d, m, mask);
        } else {
            size_t s, d, mx;
            std::scanf("%zu %zu %zu", &s, &d, &mx);
            for (const auto &r : t.getCorrespondences(s, d, mx)) std::printf("%zu %zu ", std::get<0>(r), std::get<1>(r));
            std::printf("| %zu\n", t.trackCount());
        }
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def tracklet_harness(tmp_path_factory):
    import os
    import subprocess

    d = tmp_path_factory.mktemp("tracklets")
    src = d / "h.cpp"
    src.write_text(_TRACKLET_HARNESS)
    exe = d / "h"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", inc, "-o", str(exe), str(src)])
    return str(exe)


@pytest.mark.parametrize("seed,views,points,adds,per_add", [(0, 6, 12, 60, 8), (1, 12, 40, 200, 30), (2, 4, 5, 80, 6),
                                                            (3, 30, 400, 300, 120)])
def test_oracle_cpp_tracklets_equal_the_python_restatement(tracklet_harness, seed, views, points, adds, per_add):
    import subprocess

    rng = np.random.default_rng(seed)
    ref = PyTracklets(views)
    ops, expected = [], []

    def query(a, b, mx):
        got = ref.getCorrespondences(a, b, mx)
        ops.append(f"g {a} {b} {mx}")
        expected.append(" ".join(f"{x} {y}" for x, y, _ in got) + (" " if got else "") + f"| {len(ref.tmpTracks)}")

    # the first add numbers (view, point) 0 — the "number 0 means not numbered" quirk; repeated views in one track come
    # from random histories over few points
    for k in range(adds):
        s, d = (int(x) for x in rng.choice(views, 2, replace=False))
        n = int(rng.integers(1, per_add + 1))
        m = np.stack([rng.integers(0, points, n), rng.integers(0, points, n)], 1)
        mask = (rng.random(n) < 0.8).astype(np.uint8)
        ref.add(s, d, [tuple(int(x) for x in r) for r in m], list(mask))
        ops.append(f"a {s} {d} {n} " + " ".join(f"{a} {b} {c}" for (a, b), c in zip(m, mask)))
        if k % 5 == 0:
            a, b = (int(x) for x in rng.choice(views, 2, replace=False))
            for mx in (0, 3, 5000):  # maximum + 1 rows come back when more tracks are shared
                query(a, b, mx)
    for a in range(views):
        for b in range(views):
            if a != b:
                query(a, b, 2)
    out = subprocess.run([tracklet_harness], input="\n".join(ops) + "\n", capture_output=True, text=True, check=True)
    assert out.stdout.splitlines() == expected
    assert any(len(e.split("|")[0].split()) == 2 * 4 for e in expected if e)  # some query returned maximum + 1 = 4 rows


# ---- pgb_run_hashing against pgo_run_scene_hashing --------------------------------------------------------------------
def cpu_matches(scene):
    """A deterministic mutual-nearest-neighbour ratio matcher (numpy): the CPU tests only need the same match list on
    both sides, not matchFeatures' exact rows (those are the device's, tests/test_gpu_match_scene.py)."""
    kpo, desc = scene["kp_offset"].astype(np.int64), scene["desc"].astype(np.float64)
    mo, rows = [0], []
    for s, d in scene["pair_views"]:
        a, b = desc[kpo[s]:kpo[s + 1]], desc[kpo[d]:kpo[d + 1]]
        D = (a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * a @ b.T
        fw = np.argsort(D, 1, kind="stable")[:, :2]
        bw = np.argmin(D, 0)
        i = np.arange(len(a))
        best, second = D[i, fw[:, 0]], D[i, fw[:, 1]]
        ok = (best < 0.81 * second) & (bw[fw[:, 0]] == i)
        order = np.argsort(best[ok] / second[ok], kind="stable")
        m = np.stack([i[ok], fw[ok, 0]], 1)[order]
        rows.append(m)
        mo.append(mo[-1] + len(m))
    scene["m_offset"] = np.array(mo, dtype=np.uint64)
    scene["matches"] = np.ascontiguousarray(np.vstack(rows), dtype=np.uint32)
    return scene


class StandInEngine:
    """pgi_* stand-ins over the oracle: createCorrespondenceMatrix, the in-traversal test, estimatePose with its inlier mask,
    guidedMatching.  Holds the scene's pairs and the extra pairs like a context does."""

    def __init__(self, oracle, scene, thr_px=0.4, min_inliers=20):
        self.o, self.sc, self.thr_px, self.min_inliers = oracle, scene, thr_px, min_inliers
        self.extra, self.pending = [], None
        self.calls = dict(extra=0, waves=0, extra_waves=0, guided=0)
        kpo = scene["kp_offset"].astype(np.int64)
        self.kp = [scene["kp"][kpo[v]:kpo[v + 1]] for v in range(len(kpo) - 1)]
        self.desc = [scene["desc"][kpo[v]:kpo[v + 1]] for v in range(len(kpo) - 1)]
        self._make_callbacks()

    def corr(self, src, dst, matches):
        f = float(self.sc["focal"][src])
        cx, cy = self.sc["size"][src] / 2.0
        return self.o.create_correspondences(self.kp[src], self.kp[dst], matches, f, f, cx, cy, self.thr_px)

    def K(self, v):
        f, (w, h) = float(self.sc["focal"][v]), self.sc["size"][v]
        return np.array([[f, 0.0, w / 2.0], [0.0, f, h / 2.0], [0.0, 0.0, 1.0]])

    def _make_callbacks(self):
        sc = self.sc

        @C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32))
        def register_extra(_e, n, pv, mo, m):
            self.calls["extra"] += 1
            self.extra = []
            for p in range(n):
                rows = np.array([[m[2 * i], m[2 * i + 1]] for i in range(mo[p], mo[p + 1])], dtype=np.uint32).reshape(-1, 2)
                self.extra.append(self.corr(pv[2 * p], pv[2 * p + 1], rows))
            return 0

        @C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.c_uint32)
        def submit(_e, n, pair_id, hoff, hyp, flags):
            assert n == 1 and flags & (B.WAVE_FALLBACK | 4)
            self.calls["waves"] += 1
            pid = int(pair_id[0])
            if flags & 16:
                self.calls["extra_waves"] += 1
                corr, thr = self.extra[pid]
            else:
                s, d = (int(x) for x in sc["pair_views"][pid])
                corr, thr = self.corr(s, d, sc["matches"][int(sc["m_offset"][pid]):int(sc["m_offset"][pid + 1])])
            v = np.zeros(1, dtype=B.VERDICT_DTYPE)[0]
            v["q"] = [0, 0, 0, 1]
            guesses = []
            if hoff[1] > hoff[0]:
                h = np.array([hyp[k] for k in range(7)])
                ok, cnt = self.o.test_pose(corr, h, 1.5 * thr, 5)
                v["n_hypotheses"], v["test_passed"], v["test_count"] = 1, ok, cnt
                if ok:
                    guesses = [h]
            r = self.o.estimate_pose(corr, thr, guesses, self.min_inliers)
            v["accepted"], v["branch"] = r["success"], r["branch"] if r["success"] else 0
            v["inlier_count"], v["n_corr"], v["E"] = r["inlier_number"], len(corr), r["E"].reshape(9)
            if r["success"]:
                v["q"], v["t"] = r["pose"][:4], r["pose"][4:]
            self.pending = (v, r["mask"].astype(np.uint8))
            return 0

        @C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p)
        def wait(_e, out, masks):
            v, mask = self.pending
            C.memmove(out, np.array([v]).ctypes.data, B.VERDICT_DTYPE.itemsize)
            if masks and len(mask):
                C.memmove(masks, mask.ctypes.data, len(mask))
            return 0

        @C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_double), C.c_int32, C.c_uint32,
                     C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.POINTER(C.c_uint32))
        def guided(_e, src, dst, pose, bins, max_points, m_out, v_out, n_out):
            self.calls["guided"] += 1
            g = self.o.guided_match(self.kp[src], self.desc[src], self.kp[dst], self.desc[dst], np.array([pose[k] for k in range(7)]),
                                    self.K(src), self.K(dst), sc["size"][src], sc["size"][dst], bins, max_points)
            k = len(g["selected_matches"])
            for i in range(k):
                m_out[2 * i], m_out[2 * i + 1] = int(g["selected_matches"][i, 0]), int(g["selected_matches"][i, 1])
                v_out[i] = float(g["selected_ratios"][i])
            n_out[0] = k
            return 0

        self.fns = (submit, wait, register_extra, guided)


def hashing_scene(n_views, seed):
    sc = S.make_descriptor_scene(n_views=n_views, kp_range=(500, 900), dim=64, seed=seed, arc=np.pi,
                                 visible_half_angle=0.6 * np.pi)
    return cpu_matches(sc)


@pytest.fixture(scope="module", params=[(12, 3), (24, 4)], ids=["12v", "24v"])
def scene(request):
    return hashing_scene(*request.param)


def assert_same_run(plog, pedges, psrc, olog, oedges, osrc):
    assert len(plog) == len(olog)
    for f in LOG_FIELDS:
        assert np.array_equal(plog[f], olog[f]), f
    assert len(pedges) == len(oedges)
    for f in ("src", "dst", "q", "t", "score"):
        assert np.array_equal(pedges[f], oedges[f]), f
    assert np.array_equal(psrc["source"], osrc["source"]) and np.array_equal(psrc["guided_rows"], osrc["guided_rows"])


def assert_both_branches_ran(src, log):
    ran = src["source"] != B.MATCH_SKIPPED
    quick = src["source"] == B.MATCH_QUICK
    assert quick.sum() >= 0.2 * ran.sum(), (quick.sum(), ran.sum())
    assert np.any(quick & (log["committed"] > 0) & (src["guided_rows"] > 0))      # a guided add
    assert np.any((src["source"] == B.MATCH_FULL) & (log["committed"] > 0))      # a full-match add


@pytest.mark.parametrize("path_finding", [True, False], ids=["path", "nopath"])
def test_hashing_loop_matches_the_oracle_host(oracle, scene, path_finding):
    olog, oedges, osrc = pgo_hashing.run_scene_hashing(scene, sim_threshold=0.0, use_path_finding=path_finding)
    eng = StandInEngine(oracle, scene)
    host = B.HostBuilder(scene, host_threads=1, lazy_fallback=True, use_path_finding=path_finding, **CFG)
    rc, st = host.run_hashing(scene["matches"], *eng.fns, None)
    assert rc == 0
    plog, psrc = host.log(), host.match_sources()
    assert_same_run(plog, host.edges(), psrc, olog, oedges, osrc)
    assert_both_branches_ran(psrc, plog)
    s = st.as_dict()
    assert s["positions"] == len(plog) and s["quick_matched"] == np.count_nonzero(psrc["source"] == B.MATCH_QUICK)
    assert s["full_matched"] == np.count_nonzero(psrc["source"] == B.MATCH_FULL)
    assert s["guided_calls"] == eng.calls["guided"] and s["guided_rows"] == int(psrc["guided_rows"].sum())
    assert s["tracklet_adds"] == int(plog["committed"].sum())
    assert eng.calls["extra"] == eng.calls["extra_waves"] == s["quick_matched"]
    if path_finding:
        assert plog["hadPath"].any()
    # a second call on a finished builder has nothing left to run; a builder driven by waves is refused
    assert host.run_hashing(scene["matches"], *eng.fns, None)[0] == 0 and len(host.log()) == len(plog)


def test_run_hashing_rejects_a_builder_driven_by_waves(oracle):
    from oracle_engine import OracleEngine

    sc = hashing_scene(8, 6)
    host = B.HostBuilder(sc, host_threads=1, lazy_fallback=True, **CFG)
    items = host.next_wave(4)
    host.commit_wave(OracleEngine(oracle, sc).run_items(items[items["need_gpu"] > 0]))
    eng = StandInEngine(oracle, sc)
    assert host.run_hashing(sc["matches"], *eng.fns, None)[0] == -1
