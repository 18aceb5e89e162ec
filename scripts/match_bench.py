"""Batched descriptor matching (K9, pgi_register_scene_descriptors) against the per-pair matcher (pgi_match_features, K9 on
one pair per call) on descriptor scenes of 300 views: 4 000 and 2 000 keypoints per view, 128 dimensions, all 44 850 pairs.

Per scene it reports: the batched call (matching + registration; the call ends in a device synchronise, so the host clock
around it is the call's time) with its K9 kernel time from CUDA events; the per-pair loop on a sample of pairs, scaled
to all pairs; that the sample's matches and ratio bits are equal in both; one PoseGraphBuilder pass on the matched
scene.  Rates: pairs/s, distance evaluations/s and algorithmic FP32 operations/s (3 non-fused operations per dimension
per distance, each distance counted once), the last also as a share of the FP32 instruction bound
(SMs x 128 lanes x the SM clock sampled during the batched call).  The card's name and power limit are part of the result.

    python scripts/match_bench.py [--loop-pairs 300] [--out profiles/match_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pose_graph_initialization_b200 import builder as B  # noqa: E402
from pose_graph_initialization_b200 import scene as S  # noqa: E402
from pose_graph_initialization_b200.engine import Engine  # noqa: E402


def smi(fields):
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout
    return [x.strip() for x in out.strip().splitlines()[0].split(",")]


class ClockSampler:
    """SM clock (MHz) sampled every 0.25 s while the timed call runs."""

    def __init__(self):
        self.samples, self.stop = [], threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                self.samples.append(float(smi("clocks.sm")[0]))
            except Exception:
                pass
            self.stop.wait(0.25)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join()


def bench_scene(eng, kp, loop_pairs, n_sms, seed):
    t0 = time.perf_counter()
    sc = S.make_descriptor_scene(300, kp_range=(kp, kp), seed=seed)
    gen_s = time.perf_counter() - t0
    P = len(sc["pair_views"])
    dim = sc["desc"].shape[1]
    eng.reset_stats()
    matched = dict(sc)
    with ClockSampler() as clk:
        t0 = time.perf_counter()
        eng.register_scene_descriptors(matched, 0.4)
        batched_s = time.perf_counter() - t0
    st = eng.stats()
    k9_s = st["ms_match"] / 1e3
    dist = int(st["dist_evals"])
    flops = 3.0 * dim * dist
    mhz = float(np.median(clk.samples)) if clk.samples else float("nan")
    bound = n_sms * 128 * mhz * 1e6
    # the per-pair loop on an evenly spaced sample of pairs, scaled per pair
    ko = sc["kp_offset"].astype(np.int64)
    mo = matched["m_offset"].astype(np.int64)
    sample = np.linspace(0, P - 1, min(loop_pairs, P)).astype(np.int64)
    args = [(sc["desc"][ko[s]:ko[s + 1]], sc["desc"][ko[d]:ko[d + 1]]) for s, d in sc["pair_views"][sample]]
    eng.match_features(*args[0])  # warm
    outs = []
    t0 = time.perf_counter()
    for a in args:
        outs.append(eng.match_features(*a))
    loop_s = (time.perf_counter() - t0) / len(sample) * P
    equal = all(np.array_equal(matched["matches"][mo[p]:mo[p + 1]], m) and
                matched["ratios"][mo[p]:mo[p + 1]].tobytes() == r.tobytes() for p, (m, r) in zip(sample, outs))
    # one full pass of the builder on the matched scene (matches present: no re-matching)
    pgb = B.PoseGraphBuilder(scene=matched)
    t0 = time.perf_counter()
    graph = pgb.run()
    pass_s = time.perf_counter() - t0
    pgb.close()
    return dict(views=300, keypoints=kp, dim=dim, pairs=P, scene_gen_s=round(gen_s, 2), matches=int(mo[-1]),
                pairs_below_50=int((np.diff(mo) < 50).sum()),
                batched_s=batched_s, k9_kernel_s=k9_s, k0_ms=st["ms_correspondences"], launches=int(st["launches"]),
                h2d_bytes=int(st["h2d_bytes"]), d2h_bytes=int(st["d2h_bytes"]), dist_evals=dist,
                pairs_per_s=P / batched_s, dist_evals_per_s=dist / batched_s, fp32_ops_per_s=flops / batched_s,
                fp32_ops_per_s_kernel=flops / k9_s, sm_clock_mhz=mhz, fp32_bound_ops_per_s=bound,
                fp32_share_of_bound_call=flops / batched_s / bound, fp32_share_of_bound_kernel=flops / k9_s / bound,
                loop_sample_pairs=int(len(sample)), loop_s_scaled=loop_s, speedup_vs_loop=loop_s / batched_s,
                sample_equal_to_loop=bool(equal), builder_pass_s=pass_s, edges=int(graph.numEdges()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loop-pairs", type=int, default=300)
    ap.add_argument("--out", default=None)
    ap.add_argument("--kp", type=int, nargs="*", default=[4000, 2000])
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("match_bench needs a GPU")
    name, power = smi("name,power.limit")
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    eng = Engine(device=0)
    warm = S.make_descriptor_scene(8, kp_range=(300, 900), seed=1)
    eng.register_scene_descriptors(warm, 0.4)
    res = dict(gpu=name, power_limit_w=float(power), sms=n_sms, max_sm_clock_mhz=float(smi("clocks.max.sm")[0]),
               scenes=[bench_scene(eng, kp, a.loop_pairs, n_sms, seed=100 + i) for i, kp in enumerate(a.kp)])
    eng.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
