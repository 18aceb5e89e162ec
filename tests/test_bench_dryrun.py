"""bench.py's GPU arm end to end on CPU with stand-ins for the CUDA pieces (tests/bench_dryrun.py): the control flow and
the arithmetic of the JSON line, for both step definitions.  The numbers mean nothing; the contract keys must be there."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("extra,passes", [(["--steps", "4", "--warmup", "2"], 1), (["--steps", "2", "--warmup", "1", "--step", "pass"], 2),
                                          (["--steps", "20", "--warmup", "5", "--verify", "50", "--wave", "8"], 1)])
def test_bench_main_dry_run(extra, passes):
    r = subprocess.run([sys.executable, os.path.join(HERE, "bench_dryrun.py"), "--config", "dry_24v", "--cpu-sample", "16", "--wave", "16", "--fb-wave", "32"] + extra,
                       capture_output=True, text=True, timeout=900)
    # --verify compares the stand-in engine's verdicts with the oracle: they cannot agree, bench.py must exit with 3
    assert r.returncode == (3 if "--verify" in extra else 0), r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    K = int(extra[1])
    assert d["steps"] == K and d["warmup"] == int(extra[3]) and d["n_gpus"] == 1 and d["edges"] == 276
    assert d["config"]["workload"] == "dry_24v" and "l2" in d["config"] and d["unit"] == "pairs/s"
    # value = pairs of the timed passes / their time
    assert abs(d["value"] - 276 * passes / (d["ms_per_step"] * K * 1e-3)) < 1e-6 * d["value"]
    for key in ("e2e", "roofline", "cpu_baseline", "gpu_launches", "clocks", "host_counters", "branch_mix", "run_config"):
        assert key in d
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] <= d["value"] * 1.0001
    assert d["roofline"]["kernel"] == d["roofline"]["dominant"]
    assert d["cpu_baseline"]["single_thread"]["value"] > 0
    assert len(d["step_wall_ms"]["e2e"]) == K
    if "--verify" in extra:
        assert d["verify"]["tuples"]["tuples"] == 50  # (stand-in verdicts cannot agree with the oracle; the plumbing ran)


def _dry_run(*extra):
    return subprocess.run([sys.executable, os.path.join(HERE, "bench_dryrun.py"), "--config", "dry_24v", "--cpu-sample", "16",
                           "--wave", "16", "--fb-wave", "32", "--warmup", "1"] + list(extra), capture_output=True, text=True, timeout=900)


def test_bench_refuses_steps_it_cannot_fill():
    """Every one of the --steps K timed steps carries queue positions: 18 waves of 16 cannot fill 20 steps."""
    r = _dry_run("--steps", "20")
    assert r.returncode != 0 and "ended in step 18" in r.stderr and not r.stdout.strip(), r.stderr[-3000:]
    r = _dry_run("--steps", "0")
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs writes the pose graph of the last timed step, one float64 array per edge field; the same arguments
    write the same arrays."""
    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        r = _dry_run("--steps", "3", "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-3000:]
        runs.append((json.loads(r.stdout.strip().splitlines()[-1]), {f: np.load(out / f) for f in os.listdir(out)}))
    (d, a), (_, b) = runs
    assert sorted(a) == ["edges_%s.npy" % f for f in ("branch", "dst", "inlier_number", "n_corr", "q", "row", "score", "src", "t")]
    assert all(x.dtype == np.float64 and len(x) == d["edges"] == 276 for x in a.values())
    assert a["edges_q.npy"].shape == (276, 4) and a["edges_t.npy"].shape == (276, 3)
    assert np.array_equal(a["edges_row.npy"], np.arange(276))
    assert (a["edges_branch.npy"] == 1).sum() == d["branch_mix"]["path_accepted"]
    assert (a["edges_branch.npy"] == 2).sum() == d["branch_mix"]["fallback_accepted"]
    assert all(np.array_equal(a[f], b[f]) for f in a)


def test_dump_outputs_samples_rows_beyond_the_budget(tmp_path):
    import bench
    from pose_graph_initialization_b200 import builder as B

    edges = np.zeros(1000, dtype=B.EDGE_DTYPE)
    edges["src"] = np.arange(1000)
    edges["score"] = np.linspace(0, 1, 1000)
    for k in range(2):
        bench.dump_outputs(str(tmp_path / str(k)), edges, budget=100 * 112)  # 112 B: 14 float64 per edge
    files = sorted(os.listdir(tmp_path / "0"))
    assert sum(os.path.getsize(tmp_path / "0" / f) - 128 for f in files) <= 100 * 112  # (128 B: .npy header)
    rows = np.load(tmp_path / "0" / "edges_row.npy")
    assert len(rows) == 100 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "0" / "edges_src.npy"), rows)
    assert np.array_equal(np.load(tmp_path / "0" / "edges_score.npy"), edges["score"][rows.astype(np.int64)])
    assert all(np.array_equal(np.load(tmp_path / "0" / f), np.load(tmp_path / "1" / f)) for f in files)


def test_bench_main_dry_run_two_ranks():
    """The same under torchrun with two ranks (gloo): shard pinning, batches bracketed by barriers, the record exchange and
    the prefetch gather of builder.py, max-over-ranks timing, one JSON line from rank 0."""
    port = 34500 + (os.getpid() % 2000)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(HERE, "bench_dryrun.py"), "--gpus", "2", "--config", "dry_24v",
                        "--cpu-sample", "16", "--wave", "16", "--fb-wave", "32", "--steps", "5", "--warmup", "2"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and d["steps"] == 5 and d["edges"] == 276
    assert d["host_s_per_pass"]["exchanges"] > 0
    assert abs(d["value"] - 276 / (d["ms_per_step"] * 5 * 1e-3)) < 1e-6 * d["value"]
