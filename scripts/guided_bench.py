"""Batched guided matching (K10: PoseGraphBuilder.guided_match_edges / pgi_guided_match_pairs) against the one-pair-per-call
loop (pgi_guided_match_views, K10 on one pair per call) on the 300-view descriptor scene of hashing_bench.py (2 000-4 000 keypoints, 128-D).

(a) Batched throughput: the scene runs in the default wave mode, then guided_match_edges() matches every committed edge at
    its own pose with max_points 100 and 0: K10 device time from the CUDA events the engine records around each chunk
    (pgi_stats.ms_guided_pairs), wall time of the call (it ends in a device synchronise), pairs/s and descriptor
    distances/s.  The single-pair loop runs on >= 300 evenly spaced edges and is scaled to all edges, as match_bench.py
    does; the rows of every compared edge must equal the batch's.
(b) Single-pair latency: pgi_guided_match_pairs on a batch of one pair against pgi_guided_match_views on the same cases
    (device time per call from the events).  The script exits non-zero if any rows differ.

A share of peak is guided_dist_evals x 2 * dim FP64 operations (the gate arithmetic is not counted) over the K10 device
time, against the non-fused FP64 rate pgi_dbg_fp64_peak measures in the same call.  Registration and matching (K9) are
outside every timed window.  The card's name, power limit and SM clock are read in the same call.

    python scripts/guided_bench.py [--views 300] [--sample 300] [--repeats 3] [--out profiles/r05_guided_bench.json]
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


def batched(pgb, max_points, repeats, dim, fp64_tflops):
    eng = pgb.engine
    pgb.guided_match_edges(max_points=max_points)  # warm: module load, scratch allocation
    best = None
    for _ in range(repeats):
        before = eng.stats()
        t0 = time.perf_counter()
        off, m, v = pgb.guided_match_edges(max_points=max_points)
        wall = time.perf_counter() - t0
        after = eng.stats()
        ms = after["ms_guided_pairs"] - before["ms_guided_pairs"]
        pairs = after["guided_pairs"] - before["guided_pairs"]
        evals = after["guided_dist_evals"] - before["guided_dist_evals"]
        r = dict(max_points=max_points, pairs=int(pairs), rows=int(off[-1]), chunks=int(after["guided_chunks"] - before["guided_chunks"]),
                 k10_device_ms=ms, wall_ms=wall * 1e3, pairs_per_s_device=pairs / (ms / 1e3), pairs_per_s_wall=pairs / wall,
                 dist_evals=int(evals), dist_evals_per_s_device=evals / (ms / 1e3),
                 fp64_share_of_nonfused_peak=evals * 2 * dim / (ms / 1e3) / (fp64_tflops * 1e12))
        if best is None or ms < best["k10_device_ms"]:
            best = r
        best.setdefault("device_ms_all_repeats", []).append(ms)
    return best, (off, m, v)


def views_loop(pgb, idx):
    """pgi_guided_match_views on the edges idx: (rows per edge, device ms, wall ms) of the loop."""
    eng = pgb.engine
    e = pgb.graph.edges
    qt = lambda i: np.concatenate([e["q"][i], e["t"][i]])
    eng.guided_match_views(int(e["src"][idx[0]]), int(e["dst"][idx[0]]), qt(idx[0]))  # warm
    before = eng.stats()
    rows = []
    t0 = time.perf_counter()
    for i in idx:
        rows.append(eng.guided_match_views(int(e["src"][i]), int(e["dst"][i]), qt(i), 45, pgb.max_points_hashing))
    wall = time.perf_counter() - t0
    after = eng.stats()
    return rows, after["ms_guided"] - before["ms_guided"], wall * 1e3


def single_pair(pgb, idx):
    """K10 on batches of one pair, each of the edges idx: device ms and wall ms of all calls."""
    eng = pgb.engine
    e = pgb.graph.edges
    one = lambda i: (np.array([[e["src"][i], e["dst"][i]]], dtype=np.uint32), np.concatenate([e["q"][i], e["t"][i]])[None])
    eng.guided_match_pairs(*one(idx[0]), 45, pgb.max_points_hashing)  # warm
    before = eng.stats()
    out = []
    t0 = time.perf_counter()
    for i in idx:
        out.append(eng.guided_match_pairs(*one(i), 45, pgb.max_points_hashing))
    wall = time.perf_counter() - t0
    after = eng.stats()
    return out, after["ms_guided_pairs"] - before["ms_guided_pairs"], wall * 1e3


def same_rows(sel, m, v):
    return len(sel) == len(m) and all(int(a) == int(x[0]) and int(b) == int(x[1]) and np.float64(r).tobytes() == np.float64(y).tobytes()
                                      for (a, b, r), x, y in zip(sel, m, v))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=300)
    ap.add_argument("--seed", type=int, default=201)  # hashing_bench.py's 300-view scene
    ap.add_argument("--sample", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("guided_bench needs a GPU")
    name, power, clk, max_clk = smi("name,power.limit,clocks.sm,clocks.max.sm")
    res = dict(gpu=name, power_limit_w=float(power), sm_clock_mhz_at_start=float(clk), max_sm_clock_mhz=float(max_clk))
    sc = S.make_descriptor_scene(a.views, kp_range=(2000, 4000), dim=128, seed=a.seed)
    pgb = B.PoseGraphBuilder(scene=sc)
    pgb.prepare()
    t0 = time.perf_counter()
    g = pgb.run()
    res.update(views=a.views, seed=a.seed, keypoints_range=[2000, 4000], dim=128, wave_pass_s=time.perf_counter() - t0,
               edges=int(g.numEdges()))
    fp64 = pgb.engine.fp64_peak(fused=False)
    res["fp64_nonfused_peak_tflops_measured"] = fp64
    res["batched"] = []
    batch100 = None
    for mp in (pgb.max_points_hashing, 0):
        r, out = batched(pgb, mp, a.repeats, 128, fp64)
        res["batched"].append(r)
        if mp:
            batch100 = out
    E = g.numEdges()
    idx = np.unique(np.linspace(0, E - 1, min(a.sample, E)).astype(np.int64))
    rows, views_ms, views_wall = views_loop(pgb, idx)
    off, m, v = batch100
    equal = [same_rows(rows[k], m[int(off[i]):int(off[i + 1])], v[int(off[i]):int(off[i + 1])]) for k, i in enumerate(idx)]
    res["views_loop"] = dict(edges_compared=len(idx), rows_equal_on_every_compared_edge=bool(all(equal)),
                             edges_differing=int(len(equal) - sum(equal)), device_ms=views_ms, wall_ms=views_wall,
                             device_ms_per_call=views_ms / len(idx), wall_ms_per_call=views_wall / len(idx),
                             device_ms_scaled_to_all_edges=views_ms / len(idx) * E, wall_ms_scaled_to_all_edges=views_wall / len(idx) * E)
    b = res["batched"][0]
    res["speedup_all_edges_device"] = res["views_loop"]["device_ms_scaled_to_all_edges"] / b["k10_device_ms"]
    res["speedup_all_edges_wall"] = res["views_loop"]["wall_ms_scaled_to_all_edges"] / b["wall_ms"]
    ones, k10_ms, k10_wall = single_pair(pgb, idx)
    equal1 = [same_rows(rows[k], o[1], o[2]) for k, o in enumerate(ones)]
    res["single_pair"] = dict(cases=len(idx), rows_equal=bool(all(equal1)), pairs_device_ms_per_call=k10_ms / len(idx),
                              views_device_ms_per_call=views_ms / len(idx), pairs_wall_ms_per_call=k10_wall / len(idx),
                              views_wall_ms_per_call=views_wall / len(idx))
    pgb.close()
    res["sm_clock_mhz_at_end"] = float(smi("clocks.sm")[0])
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not (res["views_loop"]["rows_equal_on_every_compared_edge"] and res["single_pair"]["rows_equal"]):
        sys.exit("batched rows differ from the single-pair rows")


if __name__ == "__main__":
    main()
