"""Epipolar-hashing mode (PoseGraphBuilder(kUseEpipolarHashing_=True), the exact sequential loop pgb_run_hashing) on
descriptor scenes of 100 and 300 views with 2 000-4 000 keypoints per view, 128 dimensions.

Per scene it reports: the hashing pass (positions/s over the wall time of run(), which ends in a device synchronise), the
share of positions matched quickly from the tracklets, the time split of pgb_hashing_stats (A*, engine, guided matching,
tracklets); the same scene's default run() without hashing for comparison; and the device time per call of
pgi_guided_match_views against pgi_guided_match (K10 on one pair) on the same (pair, pose) cases, from the CUDA events the
engine records around the launches (pgi_stats.ms_guided), averaged over many calls.  The script exits non-zero if the two
entry points select different rows on any case.  Registration (K9 matching) is outside both timed
passes.  The card's name, power limit and SM clock are read in the same call and are part of the result.

    python scripts/hashing_bench.py [--views 100 300] [--guided-calls 200] [--out profiles/hashing_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pose_graph_initialization_b200 import builder as B  # noqa: E402
from pose_graph_initialization_b200 import scene as S  # noqa: E402


def smi(fields):
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout
    return [x.strip() for x in out.strip().splitlines()[0].split(",")]


def guided_device_time(pgb, sc, n_calls, seed):
    """Mean device time per call (ms) of pgi_guided_match_views and of pgi_guided_match on the same cases, and whether their
    selected rows are equal on every case."""
    eng = pgb.engine
    ko = sc["kp_offset"].astype(np.int64)
    rng = np.random.default_rng(seed)
    committed = pgb.host.edges()
    pick = rng.integers(0, len(committed), n_calls)
    cases = [(int(committed["src"][i]), int(committed["dst"][i]), np.concatenate([committed["q"][i], committed["t"][i]])) for i in pick]

    def K(v):
        f, (w, h) = float(sc["focal"][v]), sc["size"][v]
        return np.array([[f, 0.0, w / 2.0], [0.0, f, h / 2.0], [0.0, 0.0, 1.0]])

    out, rows = {}, {}
    for name in ("views", "single_pair"):
        s0, d0, qt0 = cases[0]
        eng.guided_match_views(s0, d0, qt0)  # warm
        before = eng.stats()
        t0 = time.perf_counter()
        rows[name] = got = []
        for s, d, qt in cases:
            if name == "views":
                got.append(eng.guided_match_views(s, d, qt))
            else:
                got.append(eng.guided_match(sc["kp"][ko[s]:ko[s + 1]], sc["desc"][ko[s]:ko[s + 1]], sc["kp"][ko[d]:ko[d + 1]],
                                            sc["desc"][ko[d]:ko[d + 1]], qt, K(s), K(d), sc["size"][s], sc["size"][d])["selected"])
        wall = time.perf_counter() - t0
        after = eng.stats()
        calls = after["guided_calls"] - before["guided_calls"]
        out[name] = dict(calls=int(calls), device_ms_per_call=(after["ms_guided"] - before["ms_guided"]) / max(calls, 1),
                         wall_ms_per_call=wall / len(cases) * 1e3,
                         h2d_bytes_per_call=(after["h2d_bytes"] - before["h2d_bytes"]) / len(cases))
    out["rows_equal"] = rows["views"] == rows["single_pair"]
    return out


def bench_scene(views, guided_calls, seed):
    t0 = time.perf_counter()
    sc = S.make_descriptor_scene(views, kp_range=(2000, 4000), dim=128, seed=seed)
    gen_s = time.perf_counter() - t0
    pgb = B.PoseGraphBuilder(kUseEpipolarHashing_=True, scene=sc)
    t0 = time.perf_counter()
    pgb.prepare()  # K9 matching + registration + resident descriptors: not part of the timed pass
    prep_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    g = pgb.run()
    hashing_s = time.perf_counter() - t0
    st = pgb.hashing_stats
    src = pgb.match_sources
    ran = int(np.count_nonzero(src["source"] != B.MATCH_SKIPPED))
    guided = guided_device_time(pgb, sc, guided_calls, seed)
    res = dict(views=views, keypoints_range=[2000, 4000], dim=128, pairs=len(sc["pair_views"]), matches=int(sc["m_offset"][-1]),
               scene_gen_s=round(gen_s, 2), prepare_s=prep_s, hashing_pass_s=hashing_s, positions=int(st["positions"]),
               positions_per_s=st["positions"] / hashing_s, verified_positions=ran,
               verified_positions_per_s=ran / hashing_s, quick_matched=int(st["quick_matched"]),
               full_matched=int(st["full_matched"]), quick_share_of_verified=st["quick_matched"] / max(ran, 1),
               guided_calls=int(st["guided_calls"]), guided_rows=int(st["guided_rows"]),
               tracklet_adds=int(st["tracklet_adds"]), edges=int(g.numEdges()),
               split_s=dict(astar=st["sec_astar"], engine=st["sec_engine"], guided=st["sec_guided"],
                            tracklets=st["sec_tracklets"]),
               guided_single_pair=guided)
    pgb.close()
    # the same scene (matches already in it) without hashing: the default speculative-wave pass
    ref = B.PoseGraphBuilder(scene=sc)
    ref.prepare()
    t0 = time.perf_counter()
    g2 = ref.run()
    res["default_pass_s"] = time.perf_counter() - t0
    res["default_positions_per_s"] = len(ref.log) / res["default_pass_s"]
    res["default_edges"] = int(g2.numEdges())
    ref.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, nargs="*", default=[100, 300])
    ap.add_argument("--guided-calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("hashing_bench needs a GPU")
    name, power, clk, max_clk = smi("name,power.limit,clocks.sm,clocks.max.sm")
    res = dict(gpu=name, power_limit_w=float(power), sm_clock_mhz_at_start=float(clk), max_sm_clock_mhz=float(max_clk),
               scenes=[bench_scene(v, a.guided_calls, seed=200 + i) for i, v in enumerate(a.views)])
    res["sm_clock_mhz_at_end"] = float(smi("clocks.sm")[0])
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not all(s["guided_single_pair"]["rows_equal"] for s in res["scenes"]):
        sys.exit("pgi_guided_match_views and pgi_guided_match select different rows")


if __name__ == "__main__":
    main()
