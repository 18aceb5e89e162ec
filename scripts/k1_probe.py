"""K1 throughput probe: 8 192 pairs x 2 000 correspondences (524 MB of FP64 rows, larger than L2), one hypothesis per
pair, PATH-only waves without byte masks, so K1 runs in its streaming form; prints the scoring time per wave (CUDA events
inside the engine) and GB/s."""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pose_graph_initialization_b200 import Engine  # noqa: E402

rng = np.random.default_rng(0)
n, N = 8192, 2000
corr = rng.uniform(-0.5, 0.5, (n * N, 4))
eng = Engine(device=0)
eng.register_pairs(corr, np.arange(n + 1, dtype=np.uint64) * N, np.full(n, 5e-4))
ident = np.tile(np.array([0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0]), (n, 1))
ids, hoff = np.arange(n, dtype=np.uint32), np.arange(n + 1, dtype=np.uint32)
for _ in range(3):
    eng.run_wave(ids, hoff, ident, flags=1)
eng.reset_stats()
reps = 10
for _ in range(reps):
    eng.run_wave(ids, hoff, ident, flags=1)
ms = eng.stats()["ms_score"] / reps
print(json.dumps(dict(tag=os.environ.get("TAG", ""), ms_per_wave=ms, gbs=n * N * 32 / ms / 1e6,
                      frac_of_6453=n * N * 32 / ms / 1e6 / 6453.7)))
