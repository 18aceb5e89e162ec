"""pgi_nn2.h (the 2-NN state K9 merges across lanes, warps and CTAs) compiled for the host: random distance rows with many
exact ties, NaN and values >= FLT_MAX, cut into random index subsets merged in random order and grouping, must give
exactly what the sequential strict-`<` scan over ascending indices gives (the scan of the reference and oracle.match_features).
And the 64-bit survivor key (ratio bits << 32 | query) must sort like (ratio, query)."""
import os
import struct
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "pose_graph_initialization_b200", "csrc", "pgi_nn2.h")

HARNESS = r"""
#include "%s"
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>
using namespace pgi;
static bool same(const Nn2 &a, const Nn2 &b) { return !memcmp(&a.d1, &b.d1, 4) && !memcmp(&a.d2, &b.d2, 4) && a.i1 == b.i1; }
int main() {
    std::mt19937_64 g(2024);
    long rows = 0, merges = 0, none = 0, ties = 0;
    for (int trial = 0; trial < 20000; trial++) {
        const int n = 1 + (int)(g() %% 300);
        const int levels = 1 + (int)(g() %% 12);  // few distinct values: exact ties everywhere
        std::vector<float> v(n);
        for (int i = 0; i < n; i++) {
            const unsigned r = (unsigned)(g() %% 100);
            if (r < 6) v[i] = NAN;
            else if (r < 10) v[i] = FLT_MAX;
            else if (r < 13) v[i] = INFINITY;
            else v[i] = (float)(g() %% levels) * 0.25f;
        }
        if (trial %% 7 == 0)  // rows with no finite neighbour at all
            for (int i = 0; i < n; i++) v[i] = g() %% 3 == 0 ? NAN : (g() %% 2 ? FLT_MAX : INFINITY);
        Nn2 seq = nn2Empty();
        for (int i = 0; i < n; i++) nn2Push(seq, v[i], (uint32_t)i);  // the reference scan
        none += seq.i1 == kNn2None;
        ties += seq.i1 != kNn2None && seq.d1 == seq.d2;
        // random partition into subsets (not contiguous), each scanned in ascending order, then merged in random order
        const int parts = 1 + (int)(g() %% std::min(n, 40));
        std::vector<Nn2> st(parts, nn2Empty());
        for (int i = 0; i < n; i++) nn2Push(st[g() %% parts], v[i], (uint32_t)i);
        std::shuffle(st.begin(), st.end(), g);
        while (st.size() > 1) {  // random pairs, random operand order: any grouping
            const size_t a = g() %% st.size();
            size_t b = g() %% (st.size() - 1);
            if (b >= a) b++;
            const Nn2 m = (g() %% 2) ? nn2Merge(st[a], st[b]) : nn2Merge(st[b], st[a]);
            st[std::min(a, b)] = m;
            st.erase(st.begin() + std::max(a, b));
            merges++;
        }
        if (!same(st[0], seq)) {
            printf("mismatch trial %%d: %%a %%a %%u vs %%a %%a %%u\n", trial, st[0].d1, st[0].d2, st[0].i1, seq.d1, seq.d2, seq.i1);
            return 1;
        }
        rows++;
    }
    printf("ok %%ld %%ld %%ld %%ld\n", rows, merges, none, ties);
    return 0;
}
"""


def test_partial_2nn_states_merge_to_the_sequential_scan(tmp_path):
    src = tmp_path / "h.cpp"
    src.write_text(HARNESS % HEADER)
    exe = tmp_path / "h"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-o", str(exe), str(src)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    tag, rows, merges, none, ties = r.stdout.split()
    assert tag == "ok" and int(rows) == 20000 and int(merges) > 100_000 and int(none) > 100 and int(ties) > 1000


def test_match_key_sorts_like_ratio_then_query():
    rng = np.random.default_rng(5)
    n = 20000
    # ratios as K9 forms them: float32 d1 / d2 with d1 < 0.9 d2, plenty of equal ratios and zeros
    d2 = rng.integers(1, 50, n).astype(np.float32)
    d1 = np.floor(rng.uniform(0, 0.9, n) * d2).astype(np.float32)
    ratio = d1 / d2
    ratio[::17] = 0.0
    query = rng.permutation(1 << 20)[:n].astype(np.uint32)
    bits = ratio.view(np.uint32).astype(np.uint64)
    key = (bits << np.uint64(32)) | query.astype(np.uint64)
    by_key = np.argsort(key, kind="stable")
    by_value = np.lexsort((query, ratio.astype(np.float64)))
    assert np.array_equal(by_key, by_value)
    # the high word is the float's bit pattern (what __float_as_uint gives on the device)
    assert struct.unpack("<I", struct.pack("<f", float(ratio[1])))[0] == int(bits[1])
    assert len(np.unique(key)) == n
