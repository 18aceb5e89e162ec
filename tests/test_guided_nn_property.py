"""pgi_guided_nn.h (the best / second-best state K10 merges across the lanes of a warp) compiled for the host: random bins with
many exact ties, DBL_MAX descriptor distances and inf / NaN / boundary gate values, cut into random runs of consecutive
entries merged in random grouping (order kept), must give exactly what the reference's sequential loop gives.  The harness
also checks that the variant which takes `second` as the true second-smallest distance disagrees with the loop, so the test
would catch that mistake.  And the builder's ValueErrors of guided_match_edges, which need no device."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "pose_graph_initialization_b200", "csrc", "pgi_guided_nn.h")

HARNESS = r"""
#include "%s"
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>
using namespace pgi;
struct Seq { double best, second; int bestIndex, countSnn; };
// the reference's loop (matcher.h:362-384), restated without the header
static Seq seqLoop(const std::vector<double> &d2, const std::vector<double> &acc) {
    Seq r{DBL_MAX, DBL_MAX, -1, 0};
    for (size_t k = 0; k < d2.size(); k++) {
        if (d2[k] >= 0.75 * 0.75) continue;
        r.countSnn += 1;
        if (acc[k] < r.best) { r.second = r.best; r.best = acc[k]; r.bestIndex = (int)(100 + k); }
    }
    return r;
}
static bool same(const GuidedNn &a, const Seq &b) {
    return !memcmp(&a.best, &b.best, 8) && !memcmp(&a.second, &b.second, 8) && a.bestIndex == b.bestIndex && a.count == b.countSnn;
}
int main() {
    std::mt19937_64 g(77);
    long lists = 0, merges = 0, secondDiffers = 0, nanGate = 0, noneFound = 0;
    for (int trial = 0; trial < 20000; trial++) {
        const int n = (int)(g() %% 200);
        const int levels = 1 + (int)(g() %% 8);  // few distinct values: exact ties everywhere
        std::vector<double> d2(n), acc(n);
        for (int k = 0; k < n; k++) {
            const unsigned r = (unsigned)(g() %% 100);
            d2[k] = r < 5 ? NAN : r < 10 ? INFINITY : r < 15 ? 0.75 * 0.75 : r < 20 ? std::nextafter(0.75 * 0.75, 0.0)
                  : (double)(g() %% 100) / 50.0;
            const unsigned q = (unsigned)(g() %% 100);
            acc[k] = q < 8 ? DBL_MAX : q < 12 ? INFINITY : (double)(g() %% levels) * 0.5;
        }
        const Seq seq = seqLoop(d2, acc);
        noneFound += seq.bestIndex < 0;
        // the candidates' states, one per entry, cut into runs of consecutive entries at random points
        std::vector<GuidedNn> st;
        GuidedNn run = guidedEmpty();
        for (int k = 0; k < n; k++) {
            if (!(d2[k] >= 0.75 * 0.75)) { guidedPush(run, acc[k], 100 + k); nanGate += std::isnan(d2[k]); }
            if (g() %% 4 == 0) { st.push_back(run); run = guidedEmpty(); }
        }
        st.push_back(run);
        while (st.size() > 1) {  // merge a random neighbour pair, earlier run first: any grouping, order kept
            const size_t a = g() %% (st.size() - 1);
            st[a] = guidedMerge(st[a], st[a + 1]);
            st.erase(st.begin() + a + 1);
            merges++;
        }
        if (!same(st[0], seq)) {
            printf("mismatch trial %%d: %%a %%a %%d %%d vs %%a %%a %%d %%d\n", trial, st[0].best, st[0].second, st[0].bestIndex,
                   st[0].count, seq.best, seq.second, seq.bestIndex, seq.countSnn);
            return 1;
        }
        // the true second-smallest distance among the candidates (below DBL_MAX) differs from the loop's `second` often
        std::vector<double> c;
        for (int k = 0; k < n; k++) if (!(d2[k] >= 0.75 * 0.75) && acc[k] < DBL_MAX) c.push_back(acc[k]);
        std::sort(c.begin(), c.end());
        const double trueSecond = c.size() >= 2 ? c[1] : DBL_MAX;
        secondDiffers += memcmp(&trueSecond, &seq.second, 8) != 0;
        lists++;
    }
    printf("ok %%ld %%ld %%ld %%ld %%ld\n", lists, merges, secondDiffers, nanGate, noneFound);
    return 0;
}
"""


def test_merged_runs_equal_the_sequential_loop(tmp_path):
    src = tmp_path / "h.cpp"
    src.write_text(HARNESS % HEADER)
    exe = tmp_path / "h"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-o", str(exe), str(src)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    tag, lists, merges, second_differs, nan_gate, none = r.stdout.split()
    assert tag == "ok" and int(lists) == 20000 and int(merges) > 100_000
    # the true second minimum is a different quantity on thousands of lists: computing it would fail the comparison
    assert int(second_differs) > 1000 and int(nan_gate) > 1000 and int(none) > 100


def test_guided_match_edges_value_errors():
    from pose_graph_initialization_b200 import builder as B
    from pose_graph_initialization_b200 import scene as S

    sc = S.make_descriptor_scene(n_views=4, kp_range=(20, 30), dim=64, seed=1)
    nodesc = {k: v for k, v in sc.items() if k != "desc"}
    with pytest.raises(ValueError, match="desc"):
        B.PoseGraphBuilder(scene=nodesc).guided_match_edges()
    with pytest.raises(ValueError, match="world_size"):
        B.PoseGraphBuilder(scene=sc, world_size=2).guided_match_edges()
    with pytest.raises(ValueError, match="no pose graph"):
        B.PoseGraphBuilder(scene=sc).guided_match_edges()
