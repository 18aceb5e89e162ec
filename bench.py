#!/usr/bin/env python
"""bench.py — pairs verified/s of the B200 hypothesis-verification path.  Default workload: BASELINE.json's
configs[2], the configuration its target is quoted on (synthetic 1,000-view scene, 499,500 pairs, 2,000
correspondences/pair, 40 % outliers, 32 GB of FP64 correspondences: fits one B200).

A "step" is one complete pass of the hot path over the scene: every queued pair goes through A* (K6 on the device,
small rounds on the host pool), in-traversal test + getInliers + five-point + E->(R,t) vote or the robust fallback
(K1-K5), and the sequential commit, producing the pose graph.  Every step runs prepare() — H2D of the compact scene
from PINNED host buffers + on-device createCorrespondenceMatrix — and then run():
  e2e    = the K (prepare + run) steps back to back, bracketed by barrier + synchronize (copies inside);
  value  = the K run() regions alone (inputs resident in HBM when each region starts), each bracketed by
           barrier + synchronize, summed.
CUDA events on the device, max over ranks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg3_1000v]
                    [--verify N] [--dump-tuples FILE] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ncu --set full on k5_fallback_score (profiles/): (dram__bytes_read + dram__bytes_write) / pairs of the launch
NCU_K5_DRAM_BYTES_PER_PAIR_LAUNCH = 164_500
# FP64 operations of one minimal five-point solve (K4a + K4b + K4c), counted by instrumenting the oracle's solver
# (tests/test_oracle_properties.py::test_five_point_flop_count keeps the figure honest): see DESIGN.md section 3
K4_FLOPS_PER_SOLVE = 60_000.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_scene(name):
    from pose_graph_initialization_b200 import scene as S
    return S.make_scene(**S.CONFIGS[name])


def scene_outlier_ratio(name):
    from pose_graph_initialization_b200 import scene as S
    return S.CONFIGS.get(name, {}).get("outlier_ratio")


def config_keys(name, scene):
    """The workload description both arms print (identical keys and values)."""
    P, n_corr = int(len(scene["pair_views"])), int(scene["m_offset"][1] - scene["m_offset"][0])
    return {"workload": name, "views": int(len(scene["focal"])), "pairs": P, "corr_per_pair": n_corr,
            "outlier_ratio": scene_outlier_ratio(name),
            "l2": "inputs (%.1f GB of FP64 correspondences) larger than the 126 MB L2" % (P * n_corr * 32 / 1e9)}


# ---- (pair, hypothesis) tuples: what the CPU legs replay ------------------------------------------------------
def tuple_fixture(name):
    return os.path.join(ROOT, "tests", "golden", "tuples_%s.npz" % name)


def tuples_from_log(log, n):
    """n evenly spaced queue positions that went through the per-pair pipeline, as (pair, hypothesis) tuples."""
    from pose_graph_initialization_b200.verify import verifiable_positions
    pos = verifiable_positions(log)
    if len(pos) > n:
        pos = pos[np.unique(np.linspace(0, len(pos) - 1, n).astype(np.int64))]
    lg = log[pos]
    return dict(position=pos.astype(np.int64), pair_id=lg["pairIndex"].astype(np.uint32), has_hyp=lg["hadPath"].astype(np.uint8),
                hyp=np.ascontiguousarray(lg["hyp"]), branch=lg["branch"].astype(np.uint8), committed=lg["committed"].astype(np.uint8),
                inlier_number=lg["inlierNumber"].astype(np.uint32), test_passed=lg["testPassed"].astype(np.uint8))


def load_tuples(name, scene):
    """Committed fixture of the config (written by `bench.py --dump-tuples` on a B200): evenly spaced queue positions
    of the sequential run with the hypothesis A* composed for each.  Without a fixture the pairs are replayed without
    hypothesis (every pair takes the fallback: a slower CPU arm; the line says so)."""
    path = tuple_fixture(name)
    if os.path.exists(path):
        d = np.load(path)
        return {k: d[k] for k in d.files}, "fixture tests/golden/%s (logged hypotheses of the sequential run)" % os.path.basename(path)
    P = len(scene["pair_views"])
    ids = np.unique(np.linspace(0, P - 1, min(P, 8192)).astype(np.int64)).astype(np.uint32)
    return dict(pair_id=ids, has_hyp=np.zeros(len(ids), dtype=np.uint8), hyp=np.zeros((len(ids), 7))), \
        "no tuple fixture for this config: every pair replayed without hypothesis (fallback branch only)"


def cpu_pipeline(scene, tup, sel, threads=0):
    """The oracle's per-pair pipeline (createCorrespondenceMatrix -> in-traversal test -> estimatePose: path branch or
    robust fallback -> E->(R,t) vote), worker-pulls-queue on all host threads, over the tuples `sel`.
    Only place besides tests/ and smoke() where oracle/ is executed."""
    from oracle import pgo_oracle as O
    O.build()
    t0 = time.perf_counter()
    r = O.scene_pipeline_batch(scene, tup["pair_id"][sel], tup["hyp"][sel], tup["has_hyp"][sel], 0.4, 20, threads)
    dt = time.perf_counter() - t0
    info = r["info"]
    return dict(pairs=int(len(sel)), seconds=dt, pairs_per_s=len(sel) / dt, cores=int(r["threads"]),
                path=int(((info[:, 0] > 0) & (info[:, 1] == 1)).sum()), fallback=int(((info[:, 0] > 0) & (info[:, 1] == 2)).sum()),
                rejected=int((info[:, 0] == 0).sum()))


CPU_NOTE = ("per-pair pipeline of processImages (PGB:553-627) on logged (pair, hypothesis) tuples; A* (~0.5 ms per pair on a "
            "host thread, <2 % of the per-pair CPU time) and the commit are not replayed")


def _cv2_usac_one(job):
    import cv2
    cv2.setNumThreads(1)
    c, thr = job
    E, mask = cv2.findEssentialMat(c[:, :2].copy(), c[:, 2:].copy(), np.eye(3), cv2.USAC_MAGSAC, 0.99, thr)
    return 0 if mask is None else int(mask.sum())


def cv2_yardstick(scene, n_pairs, workers):
    """Third-party yard-stick of SURVEY 8(d): the fallback call site's own library call, cv2.findEssentialMat(USAC_MAGSAC)
    from the cv2 wheel of this image, over a process pool of `workers` (fallback stage only: no E->(R,t) vote, no A*).
    Runs in a fresh child process (this one holds CUDA/NCCL threads) with a hard timeout; None if unavailable."""
    import tempfile
    from pose_graph_initialization_b200 import scene as S
    P = len(scene["pair_views"])
    ids = np.unique(np.linspace(0, P - 1, n_pairs).astype(np.int64))
    jobs = [S.pair_correspondences(scene, int(p), 0.4) for p in ids]
    try:
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "jobs.npz")
            np.savez(path, corr=np.stack([c for c, _ in jobs]) if len({len(c) for c, _ in jobs}) == 1 else
                     np.array([c for c, _ in jobs], dtype=object), thr=np.array([t for _, t in jobs]))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cv2-yardstick", path, "--workers", str(workers)],
                               capture_output=True, text=True, timeout=240)
        return json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 and r.stdout.strip() else None
    except Exception:
        return None


def cv2_yardstick_child(path, workers):
    import multiprocessing as mp
    try:
        import cv2
    except Exception:
        return 1
    d = np.load(path, allow_pickle=True)
    jobs = [(np.asarray(c, dtype=np.float64), float(t)) for c, t in zip(d["corr"], d["thr"])]
    with mp.get_context("fork").Pool(workers) as pool:
        pool.map(_cv2_usac_one, jobs[:workers])  # warm the workers
        t0 = time.perf_counter()
        inl = pool.map(_cv2_usac_one, jobs)
        dt = time.perf_counter() - t0
    emit({"pairs_per_s": len(jobs) / dt, "workers": workers, "pairs": len(jobs),
          "accepted": int(sum(1 for k in inl if k >= 20)),
          "what": "cv2 %s findEssentialMat(USAC_MAGSAC) only, process pool" % cv2.__version__})
    return 0


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU path (oracle port: the reference cannot be compiled in this image)
    timed on the host cores, all threads, on the same workload's tuple mix.  Rank 0 only."""
    if rank != 0:
        return
    scene = make_scene(args.config)
    cores = os.cpu_count() or 1
    tup, src = load_tuples(args.config, scene)
    n = len(tup["pair_id"])
    sample = min(n, args.cpu_sample or 128 * cores)  # ~4-8 s of all-core CPU work per step
    for w in range(args.warmup):
        cpu_pipeline(scene, tup, np.arange(w * cores, w * cores + cores) % n)
    tot_p, tot_s, last, mix = 0, 0.0, None, {"path": 0, "fallback": 0, "rejected": 0}
    for k in range(args.steps):
        # a different bounded slice of the evenly spaced tuples every step (stride keeps each slice evenly spaced)
        stride = max(1, n // sample)
        sel = (k + stride * np.arange(sample)) % n
        last = cpu_pipeline(scene, tup, sel)
        tot_p += last["pairs"]; tot_s += last["seconds"]
        for key in mix:
            mix[key] += last[key]
    v = tot_p / tot_s
    line = {
        "impl": "reference", "metric": "image_pairs_verified_per_sec", "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_keys(args.config, scene),
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": last["cores"], "kind": "port",
                         "sample": "%d tuples per step, %s; %s; branch mix of the timed tuples %s" % (sample, src, CPU_NOTE, mix)},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def emit(line):
    """Exactly one JSON line on the real stdout (NCCL/torch banners are diverted to stderr, see main)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


DUMP_BYTES = 64_000_000


def dump_outputs(path, edges, budget=DUMP_BYTES):
    """--dump-outputs: the pose graph the last timed step returned to its caller, its committed edges in commit order,
    as one float64 array per field of builder.EDGE_DTYPE (path/edges_<field>.npy) and the rows' positions in the edge
    list (edges_row.npy).  When the edges exceed `budget` bytes, a fixed seeded sample of rows, still in commit order."""
    fields = [f for f in edges.dtype.names if f != "pad"]
    row_bytes = 8 * (1 + sum(int(np.prod(edges.dtype[f].shape)) for f in fields))
    rows = np.arange(len(edges))
    if len(rows) * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(len(edges), budget // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "edges_row.npy"), rows.astype(np.float64))
    for f in fields:
        np.save(os.path.join(path, "edges_%s.npy" % f), edges[f][rows].astype(np.float64))


def verify_run(scene, log, n_tuples, replay_pairs):
    """--verify: the finished run against the CPU oracle at benchmark scale (pose_graph_initialization_b200/verify.py)."""
    from oracle import pgo_oracle as O
    from pose_graph_initialization_b200.verify import compare_tuples, verifiable_positions
    O.build()
    pos = verifiable_positions(log)
    if n_tuples > 0 and len(pos) > n_tuples:
        pos = pos[np.unique(np.linspace(0, len(pos) - 1, n_tuples).astype(np.int64))]
    tup = compare_tuples(O, scene, log, pos)
    t0 = time.perf_counter()
    rep = O.replay_scene(scene, log, max_pairs=replay_pairs)
    rep["seconds"] = time.perf_counter() - t0
    return {"tuples": tup, "host_replay": rep, "ok": tup["mismatches"] == 0 and rep["mismatches"] == 0,
            "what": "tuples: logged (pair, hypothesis) tuples through the oracle's per-pair pipeline, verdicts compared bit for bit; "
                    "host_replay: the oracle's sequential host (own queue, visibility table, A*) fed the logged verdicts, every "
                    "host-side decision and composed hypothesis compared (max_pairs=%d, 0 = whole queue)" % replay_pairs}


def main():
    global _REAL_STDOUT
    # keep stdout clean for the one-line contract: everything else this process (or NCCL) prints goes to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="cfg3_1000v")
    ap.add_argument("--step", default="batch", choices=("batch", "pass"),
                    help="what one step is: 'batch' (default) = 1/K of the queue, the K timed steps together are ONE complete pass "
                         "over the scene (the W warm-up steps are the first batches of an untimed pass run before); 'pass' = every "
                         "step is a complete pass (K + W passes)")
    ap.add_argument("--wave", type=int, default=0, help="queue positions per speculative wave (0 = default of the config)")
    ap.add_argument("--window", type=int, default=0, help="host re-search window (0 = library default)")
    ap.add_argument("--no-overlap", action="store_true", help="prefetch the fallback before the waves instead of concurrently")
    ap.add_argument("--cpu-sample", type=int, default=0, help="tuples in the cpu_baseline sample (0 = 256 x cores, ~10 s)")
    ap.add_argument("--fb-wave", type=int, default=1024, help="pairs per fallback prefetch wave")
    ap.add_argument("--fb-streams", type=int, default=2, help="background contexts running prefetch waves concurrently")
    ap.add_argument("--cv2-yardstick", default="", help=argparse.SUPPRESS)
    ap.add_argument("--workers", type=int, default=1, help=argparse.SUPPRESS)
    ap.add_argument("--lazy", action="store_true", help="run the fallback lazily inside the waves instead of prefetching it")
    ap.add_argument("--device-search", action="store_true", help="A* rounds on the device (K6) beside the host thread pool (default: host pool only)")
    ap.add_argument("--search-min-batch", type=int, default=64, help="device search: rounds with fewer searches stay on the host pool")
    ap.add_argument("--verify", type=int, default=-1, help="after the timed steps, check the last run against the CPU oracle: "
                    "N evenly spaced tuples (0 = every pair) + sequential host replay; exit code 3 on any mismatch")
    ap.add_argument("--verify-replay", type=int, default=-1, help="queue positions replayed by the oracle host (-1 = whole queue up to 400 views, else 20000; 0 = whole queue)")
    ap.add_argument("--dump-tuples", default="", help="write N evenly spaced (pair, hypothesis) tuples of the last run (npz)")
    ap.add_argument("--dump-n", type=int, default=8192)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the pose graph of the last step as float64 .npy files under DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm builds no pose graph")
    if args.cv2_yardstick:  # child mode of cv2_yardstick(): no torch, no CUDA
        sys.exit(cv2_yardstick_child(args.cv2_yardstick, args.workers))

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from pose_graph_initialization_b200 import builder as B

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the hot path has no CPU implementation (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        group = dist.group.WORLD

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scene = make_scene(args.config)  # same seed on every rank => identical scene
    if args.wave <= 0:
        args.wave = B.default_wave_size(len(scene["focal"]), world, args.device_search)
    # the step's host inputs live in PINNED memory (every step copies them host->device).  With several ranks only the
    # rank's own shard of the matches is registered, so only the shard is pinned (the full 8 GB list of the 1 000-view
    # scene stays pageable, and only rank 0 keeps it: its CPU legs replay pairs of the whole scene)
    def pin(d, keys):
        for key in keys:
            src = np.ascontiguousarray(d[key])
            pinned = torch.empty(src.nbytes, dtype=torch.uint8, pin_memory=True).numpy().view(src.dtype).reshape(src.shape)
            pinned[...] = src
            d[key] = pinned

    small = ("kp", "sim", "pair_views", "m_offset", "kp_offset", "focal", "size")
    shard = None
    if world == 1:
        pin(scene, ("matches",) + small)
    else:
        pin(scene, small)
        shard = B.shard_scene(scene, rank, world)
        pin(shard, ("matches", "pair_views", "m_offset"))
        if rank != 0:
            scene["matches"] = np.zeros((0, 2), dtype=np.uint32)
    P = len(scene["pair_views"])
    n_corr = int(scene["m_offset"][1] - scene["m_offset"][0])
    pgb = B.PoseGraphBuilder(kCoreNumber_=max(1, (os.cpu_count() or 1) // world),  # ranks share the box's cores
                             kSimilarityThreshold_=0.0, scene=scene, device=local_rank, wave_size=args.wave,
                             prefetch_fallback=not args.lazy, overlap_fallback=not args.no_overlap, research_window=args.window,
                             fallback_wave=args.fb_wave, prefetch_streams=args.fb_streams, gpu_search=args.device_search,
                             gpu_search_min_batch=args.search_min_batch, group=group, rank=rank, world_size=world)
    if shard is not None:
        pgb._sub = shard
    pgb.prepare()
    fp64_peak = pgb.engine.fp64_peak(fused=False)
    fp64_peak_fma = pgb.engine.fp64_peak(fused=True)

    K = args.steps
    batch_steps = args.step == "batch"
    batch = -(-P // K)  # queue positions per step in batch mode (cut at the next wave boundary)
    if batch_steps:
        # warm-up: one untimed pass driven exactly like the timed one; its first W batches are the warm-up steps
        if args.warmup > 0:
            for _ in pgb.run_in_batches(batch):
                pass
    else:
        for _ in range(args.warmup):
            pgb.run()
    pgb.reset_engine_stats()
    sampler = ClockSampler(local_rank)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    step_wall = {"e2e": [], "detail": []}
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    counters, timing, search_stats = None, None, None
    gen, graph = None, None
    for k in range(K):
        ts = time.perf_counter()
        evs[k][0].record()
        if not batch_steps or k == 0:
            pgb.prepare()      # H2D of the compact scene from pinned host buffers + K0 (synchronous)
        barrier()
        evs[k][1].record()
        tp = time.perf_counter()
        if not batch_steps:
            graph = pgb.run()  # inputs resident in HBM from here on
        else:
            if k == 0:
                gen = pgb.run_in_batches(batch)
            if gen is not None:
                try:
                    next(gen)          # the next `batch` queue positions of the pass
                    while k == K - 1:  # the last step ends with the pass, wherever the wave boundaries fell
                        next(gen)
                except StopIteration as done:
                    graph, gen = done.value, None
                    if k < K - 1:  # the remaining steps would be timed with nothing in them
                        sampler.stop()
                        raise SystemExit("--steps %d: the pass over %d queue positions ended in step %d (waves of %d "
                                         "positions); use fewer steps or a smaller --wave" % (K, P, k + 1, args.wave))
        barrier()
        evs[k][2].record()
        step_wall["e2e"].append(round((time.perf_counter() - ts) * 1e3, 1))
        if not batch_steps or (graph is not None and counters is None):  # (batch steps: once, when the pass is complete)
            step_wall["detail"].append({"prepare_ms": round((tp - ts) * 1e3, 1),
                                        **{kk: round(v * 1e3, 1) for kk, v in pgb.timing.items() if kk.endswith("_s")}})
            counters, timing, search_stats = pgb.counters, dict(pgb.timing), dict(getattr(pgb, "search_stats", {}) or {})
    n_edges = graph.numEdges()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    ms_e2e = evs[0][0].elapsed_time(evs[K - 1][2])
    ms_resident = sum(evs[k][1].elapsed_time(evs[k][2]) for k in range(K))
    st = pgb.engine_stats()
    log = pgb.log

    t = torch.tensor([ms_resident, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_resident, ms_e2e = float(t[0]), float(t[1])
    pairs_done = P if batch_steps else P * K  # batch steps: the K steps are one pass
    value = pairs_done / (ms_resident * 1e-3)
    e2e = pairs_done / (ms_e2e * 1e-3)

    # ---- K1 on full-size waves (HBM roofline probe): every local pair scored against one hypothesis ---------------
    # In the pipeline K1 only sees the hypotheses of a round (launch-latency bound); its bandwidth behaviour is measured
    # here on waves of 8192 pairs x 2000 rows (0.5 GB each, inputs larger than L2), at most 64 waves.
    eng = pgb.engine
    n_local = eng.n_pairs
    n_probe = min(n_local, 64 * 8192)
    ident = np.tile(np.array([0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0]), (8192, 1))
    def k1_pass():
        for s0 in range(0, n_probe, 8192):
            ids = np.arange(s0, min(n_probe, s0 + 8192), dtype=np.uint32)
            eng.run_wave(ids, np.arange(len(ids) + 1, dtype=np.uint32), ident[:len(ids)], flags=B.WAVE_PATH)
    k1_pass()
    eng.reset_stats()
    k1_pass()
    st_k1 = eng.stats()

    # ---- the fallback kernels on one wave with nothing else on the GPU: in the step several contexts overlap (wave loop,
    # two prefetch streams), so per-stage CUDA-event brackets there contain each other's kernels; the roofline's launch
    # durations — and the choice of the dominant kernel — come from this isolated wave of the same pairs (same launches:
    # 8 x (K4a, K4b, K4c, K5) + K3).  1776 pairs = 4 x 148 SMs x 3 resident K5 CTAs.
    fb_ids = np.arange(min(n_local, 1776), dtype=np.uint32)
    eng.run_wave(fb_ids, None, None, flags=B.WAVE_FALLBACK)
    eng.reset_stats()
    v_fb = eng.run_wave(fb_ids, None, None, flags=B.WAVE_FALLBACK)
    st_fb = eng.stats()
    it = np.sort(v_fb["iters"].astype(np.int64))  # iterations of the robust loop per pair (SURVEY 8d: report next to the rate)
    fb_iters = {"pairs": int(len(it)), "mean": float(it.mean()), "p10": int(it[len(it) // 10]), "median": int(it[len(it) // 2]),
                "p90": int(it[(len(it) * 9) // 10]), "max": int(it[-1]),
                "models_per_pair": st_fb["fallback_models"] / max(1, st_fb["fallback_pairs"])}
    iso = {"k4_fallback_solve": st_fb["ms_fallback_solve"], "k5_fallback_score": st_fb["ms_fallback_score"],
           "k3_decompose_vote": st_fb["ms_decompose"]}
    dominant = max(iso, key=iso.get)

    stages = {"k1_score_hypotheses": st["ms_score"], "k2_fivept_first_solution": st["ms_fivept"],
              "k4_fallback_solve": st["ms_fallback_solve"], "k5_fallback_score": st["ms_fallback_score"],
              "k3_decompose_vote": st["ms_decompose"], "k6_astar_search": float(search_stats.get("ms_search", 0.0)) * 1.0}
    hbm_peak, hbm_src = load_peaks()
    # K5: every scored model evaluates the Sampson residual of all N correspondences: 33 FP64 flops each (algorithmic)
    k5_flops = st_fb["fallback_models"] * n_corr * 33.0
    k5_t = st_fb["ms_fallback_score"] * 1e-3
    k5_launches = 8
    roof_k5 = {"kernel": "k5_fallback_score", "bound": "fp64", "achieved": k5_flops / k5_t / 1e12 if k5_t > 0 else 0.0,
               "peak": fp64_peak, "unit": "TFLOP/s",
               "traffic": NCU_K5_DRAM_BYTES_PER_PAIR_LAUNCH * len(fb_ids),
               # FP64 rows staged once per CTA + the (72 B FP64 + 48 B FP32) model records of the chunk's iterations
               "algorithmic_bytes_per_launch": int(len(fb_ids) * (
                   n_corr * 32 + 120.0 * st_fb["fallback_models"] / max(1, st_fb["fallback_pairs"] * 8))),
               "launches": k5_launches, "ms_per_launch": st_fb["ms_fallback_score"] / k5_launches,
               "timed_on": "one isolated %d-pair fallback wave after the timed region (in the step several contexts overlap and "
                           "their CUDA-event brackets contain each other's kernels)" % len(fb_ids),
               "peak_source": "measured live by pgi_dbg_fp64_peak: non-fused DMUL+DADD chains %.2f TFLOP/s (parity forbids FMA), "
                              "DFMA chains %.2f TFLOP/s; not in MEASURED_PEAKS.json.  `achieved` counts 33 algorithmic FP64 flops "
                              "per model x correspondence evaluation, most of which are certified in FP32 (DESIGN.md section 3)"
                              % (fp64_peak, fp64_peak_fma),
               "fp64_peak_nonfused_tflops": fp64_peak, "fp64_peak_dfma_tflops": fp64_peak_fma}
    roof_k5["frac"] = roof_k5["achieved"] / fp64_peak if fp64_peak > 0 else None
    k4_solves = float(st_fb["fallback_pairs"]) * float(it.mean())
    roof_k4 = {"kernel": "k4_fallback_solve", "bound": "fp64", "unit": "TFLOP/s", "peak": fp64_peak,
               "achieved": k4_solves * K4_FLOPS_PER_SOLVE / max(st_fb["ms_fallback_solve"] * 1e-3, 1e-9) / 1e12,
               "traffic": None, "launches": 24, "ms_per_launch": st_fb["ms_fallback_solve"] / 24,
               "timed_on": roof_k5["timed_on"], "peak_source": roof_k5["peak_source"],
               "flops_per_solve": K4_FLOPS_PER_SOLVE}
    roof_k4["frac"] = roof_k4["achieved"] / fp64_peak if fp64_peak > 0 else None
    # K1: 32 B per hypothesis x correspondence evaluation, measured on the full-size probe waves above
    k1_bytes = st_k1["corr_evals"] * 32.0
    k1_t = st_k1["ms_score"] * 1e-3
    roof_k1 = {"kernel": "k1_score_hypotheses", "bound": "hbm", "achieved": k1_bytes / k1_t / 1e9 if k1_t > 0 else 0.0,
               "peak": hbm_peak, "unit": "GB/s", "traffic": None,
               "peak_source": hbm_src + " (MEASURED_PEAKS.json hbm_gbs); probe: %d pairs x %d rows per pass, waves of 8192 pairs" % (n_probe, n_corr),
               "gcorr_evals_per_s": st_k1["corr_evals"] / k1_t / 1e9 if k1_t > 0 else 0.0}
    roof_k1["frac"] = roof_k1["achieved"] / hbm_peak
    roofline = dict(roof_k5 if dominant == "k5_fallback_score" else roof_k4 if dominant == "k4_fallback_solve" else roof_k5)
    roofline["dominant"] = roofline["kernel"]
    roofline["share_of_isolated_fallback_wave"] = iso[roofline["kernel"]] / max(sum(iso.values()), 1e-9)

    verify = None
    if args.verify >= 0 and rank == 0:
        replay = args.verify_replay if args.verify_replay >= 0 else (0 if len(scene["focal"]) <= 400 else 20000)
        verify = verify_run(scene, log, args.verify, replay)
    if args.dump_tuples and rank == 0:
        np.savez_compressed(args.dump_tuples, **tuples_from_log(log, args.dump_n))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, graph.edges)

    if rank == 0:
        cores = os.cpu_count() or 1
        tup = tuples_from_log(log, args.cpu_sample or 256 * cores)  # ~10 s of all-core CPU work
        cpu = cpu_pipeline(scene, tup, np.arange(len(tup["pair_id"])))
        n1 = min(len(tup["pair_id"]), 96)  # the same pipeline on ONE thread (SURVEY 8d: core_number = 1), ~3 s
        cpu1 = cpu_pipeline(scene, tup, np.unique(np.linspace(0, len(tup["pair_id"]) - 1, n1).astype(np.int64)), threads=1)
        yard = cv2_yardstick(scene, 8 * cores, cores)  # ~1-2 s
        line = {
            "metric": "image_pairs_verified_per_sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_resident / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_keys(args.config, scene),  # the workload: identical in both arms
            "run_config": {"wave": args.wave, "fallback": "lazy" if args.lazy else "prefetched",
                           "search": "host pool" if not args.device_search else "device (K6) + host pool, rounds below %d searches on the host pool alone" % args.search_min_batch,
                           "parallelism": "pairs sharded over %d rank(s), verdict exchange per wave round" % world},
            "step": ("%d queue positions (1/%d of the similarity-ordered queue, cut at the next wave boundary): the %d timed steps "
                     "are ONE complete pass over the scene, from the empty pose graph to the last committed edge; warm-up = an "
                     "untimed complete pass before" % (batch, K, K)) if batch_steps else "one complete pass over the scene",
            "timing": ("e2e: prepare (H2D + K0, in step 0) + the K batches back to back; value: the K batch regions (inputs "
                       "resident), each bracketed by barrier + synchronize; CUDA events, max over ranks") if batch_steps else
                      "e2e: K x (prepare + run) back to back; value: the K run() regions (inputs resident), each bracketed by "
                      "barrier + synchronize; CUDA events, max over ranks",
            "step_wall_ms": step_wall,
            "e2e": {"value": e2e, "unit": "pairs/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": int((st["h2d_bytes"] + search_stats.get("h2d_bytes", 0) * K) // K),
                    "d2h_bytes_per_step": int((st["d2h_bytes"] + search_stats.get("d2h_bytes", 0) * K) // K)},
            "gpu_launches": int(st["launches"] + search_stats.get("launches", 0) * K),
            "gcorr_evals_per_sec": {"path_hypotheses": st["corr_evals"] / (ms_resident * 1e-3) / 1e9,
                                    "fallback_models": st["fallback_models"] * n_corr / (ms_resident * 1e-3) / 1e9},
            "roofline": roofline, "roofline_k1_scoring": roof_k1, "roofline_k5_fallback": roof_k5, "roofline_k4_fallback": roof_k4,
            "gpu_stage_ms_per_step": {k: v / K for k, v in stages.items() if k != "k6_astar_search"} | {"k6_astar_search": stages["k6_astar_search"]},
            "gpu_stage_ms_note": "CUDA-event brackets per context; with the prefetch overlapping the waves the brackets of "
                                 "concurrent contexts include each other's kernels (sums exceed the step's GPU time)",
            "gpu_stage_ms_isolated_fallback_wave": {"pairs": int(len(fb_ids)), **iso},
            "host_s_per_pass": {k: timing.get(k) for k in ("prefetch_s", "waves_s", "total_s", "engine_s", "exchange_s", "host_s",
                                                            "wait_prefetch_s", "engine_rounds", "exchanges")},
            "host_s_per_step": {k: (timing.get(k) / K if batch_steps and timing.get(k) is not None else timing.get(k))
                                for k in ("prefetch_s", "waves_s", "total_s", "engine_s", "exchange_s", "host_s",
                                          "wait_prefetch_s", "engine_rounds", "exchanges")},
            "search_stats_last_step": search_stats,
            "host_counters": counters, "edges": int(n_edges), "wall_s": wall,
            "branch_mix": {k: int(counters[k]) for k in ("path_accepted", "fallback_accepted", "rejected", "skipped")},
            "cpu_baseline": {"value": cpu["pairs_per_s"], "unit": "pairs/s", "cores": cpu["cores"], "kind": "port",
                             "sample": "%d evenly spaced (pair, hypothesis) tuples of this run's log, %.1f s; %s; branch mix of the "
                                       "sample: %d path / %d fallback / %d rejected"
                                       % (cpu["pairs"], cpu["seconds"], CPU_NOTE, cpu["path"], cpu["fallback"], cpu["rejected"]),
                             "single_thread": {"value": cpu1["pairs_per_s"], "unit": "pairs/s", "pairs": cpu1["pairs"]},
                             "third_party_yardstick": yard},
            "fallback_iterations": fb_iters,
            "clocks": clocks,
        }
        if verify is not None:
            line["verify"] = verify
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if verify is not None and not verify["ok"]:
        sys.exit(3)


if __name__ == "__main__":
    main()
