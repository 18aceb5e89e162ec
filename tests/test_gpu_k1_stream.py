"""K1 in its streaming form (persistent CTAs, cp.async.bulk tiles through shared memory) against the direct-load K1 and the
oracle: same test verdicts, counts, inlier bit masks (observable through the five-point sample K2 draws from them) and
final verdict records on full waves — ragged pair sizes, pairs longer than one tile, several hypotheses per pair, pairs
without hypothesis.  The wave selects the form: at least two pairs per SM and no byte masks take the streaming K1, a wave
that asks for byte masks takes the direct one."""
import numpy as np
import pytest
import torch

from helpers import perturbed_pose, pose_qt, two_view
from pose_graph_initialization_b200.engine import WAVE_PATH

pytestmark = pytest.mark.gpu


def test_streaming_k1_equals_direct_k1_and_oracle(engine, oracle):
    rng = np.random.default_rng(11)
    sizes = [0, 3, 5, 31, 32, 33, 250, 1023, 1024, 1025, 2000, 2500, 4097] + list(rng.integers(40, 2300, 400))
    corr, off, thr, hyps, hoff = [], [0], [], [], [0]
    for i, n in enumerate(sizes):
        c, R, t = two_view(max(n, 1), 0.3, rng)
        c = c[:n]
        corr.append(c)
        off.append(off[-1] + n)
        thr.append(0.4 / 800.0)
        k = i % 4  # 0..3 hypotheses: good ones, bad ones, and a good one followed by a bad one
        for j in range(k):
            good = (i + j) % 2 == 0
            hyps.append(perturbed_pose(R, t, rng) if good else pose_qt(np.eye(3), np.array([1.0, 0.0, 0.0])))
        hoff.append(hoff[-1] + k)
    corr = np.vstack(corr)
    ids = np.arange(len(sizes), dtype=np.uint32)
    assert len(ids) >= 2 * torch.cuda.get_device_properties(0).multi_processor_count  # a full wave: streaming K1
    engine.register_pairs(corr, np.array(off, dtype=np.uint64), np.array(thr))
    a = engine.run_wave(ids, np.array(hoff, dtype=np.uint32), np.array(hyps), flags=WAVE_PATH)
    b, _ = engine.run_wave(ids, np.array(hoff, dtype=np.uint32), np.array(hyps), flags=WAVE_PATH, want_masks=True)  # direct K1
    assert a.tobytes() == b.tobytes()
    assert a["test_passed"].sum() > 50 and (a["n_hypotheses"] > 0).sum() > (a["test_passed"] > 0).sum()
    # single-hypothesis pairs against the oracle's in-traversal test
    for i in range(1, len(sizes), 4):
        assert hoff[i + 1] - hoff[i] == 1
        c = corr[off[i]:off[i + 1]]
        ok, cnt = oracle.test_pose(c, hyps[hoff[i + 1] - 1], 1.5 * thr[i], 5)
        assert bool(a[i]["test_passed"]) == ok and int(a[i]["test_count"]) == cnt, i
