"""The host A*'s first expansion pass has three implementations picked from the CPU at load time: AVX-512, AVX2 and the
scalar loop that defines them (pgb_host.cpp).  PGB_NO_AVX512 / PGB_NO_AVX2 step down to the next one, so every path
that runs on some supported CPU also runs here; all three must commit the same graph, bit for bit.  Each run is a
fresh process because the dispatch is decided when the library is loaded."""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

RUN = """
import sys
sys.path[:0] = [{root!r}, {here!r}]
import numpy as np
from fake_verdicts import dense_scene, drive
from pose_graph_initialization_b200 import builder as B

sc = dense_scene(80, n_corr=2000, seed=7, ring_cameras=True)
host = B.HostBuilder(sc, host_threads=1, lazy_fallback=False, similarity_threshold=0.0, minimum_inlier_number=20,
                     minimum_point_number=50, maximum_search_depth=5, traversal_heuristics_weight=0.8,
                     use_path_finding=True)
drive(host, 64, 2000)
c = {{k: v for k, v in host.counters().items() if not k.startswith("sec_")}}  # all but the timings
np.savez({out!r}, log=host.log().view(np.uint8), edges=host.edges().view(np.uint8), names=list(c),
         counts=np.array(list(c.values()), dtype=np.uint64))
host.close()
"""


def _run(tmp_path, name, **env):
    out = str(tmp_path / (name + ".npz"))
    e = {k: v for k, v in os.environ.items() if k not in ("PGB_NO_AVX2", "PGB_NO_AVX512")}
    e.update(env)
    r = subprocess.run([sys.executable, "-c", RUN.format(root=ROOT, here=HERE, out=out)], env=e, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return np.load(out)


def test_expansion_paths_commit_the_same_graph(tmp_path):
    runs = [_run(tmp_path, "default"), _run(tmp_path, "avx2", PGB_NO_AVX512="1"),
            _run(tmp_path, "scalar", PGB_NO_AVX2="1", PGB_NO_AVX512="1")]
    ref = runs[0]
    c = dict(zip(ref["names"], ref["counts"]))
    assert c["path_accepted"] > 100 and c["astar_pushes"] > 0
    for r in runs[1:]:
        for k in ("log", "edges", "names", "counts"):
            assert r[k].tobytes() == ref[k].tobytes(), k
