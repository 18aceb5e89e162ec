"""K6 (device A*, pgi_graph_search) against the host A* of pgb_host.cpp — itself proven equal to the sequential
oracle host in tests/test_host_waves.py.  The device search must return the same path (hence the same composed
hypothesis, bit for bit), the same touched-node / pushed-node counts and the same set of expanded vertices for every
query, including queries that see predicted (overlay) edges of the open wave; then the committed graphs are equal."""
import os

import numpy as np
import pytest

from fake_verdicts import dense_scene, drive
from pose_graph_initialization_b200 import builder as B
from pose_graph_initialization_b200 import scene as S

pytestmark = pytest.mark.gpu

CFG = dict(similarity_threshold=0.0, minimum_inlier_number=20, minimum_point_number=50, maximum_search_depth=5,
           traversal_heuristics_weight=0.8, use_path_finding=True)


def _run(engine, sc, wave, backend, check, n_corr=2000, max_positions=None):
    os.environ["PGB_SEARCH_CHECK"] = "1" if check else "0"
    host = B.HostBuilder(sc, host_threads=4, lazy_fallback=False, **CFG)
    if backend:
        host.set_search_backend(engine, min_batch=1)
    drive(host, wave, n_corr, max_positions)
    out = host.log().copy(), host.edges().copy(), host.counters()
    host.close()
    os.environ.pop("PGB_SEARCH_CHECK", None)
    return out


@pytest.mark.parametrize("views,wave,decimals", [(40, 64, 3), (64, 128, 1), (120, 512, 3), (120, 2048, 1), (90, 300, 2)])
def test_device_search_equals_host_search(engine, views, wave, decimals):
    sc = dense_scene(views, seed=views + decimals, decimals=decimals)
    hlog, hedges, hc = _run(engine, sc, wave, backend=False, check=False)
    glog, gedges, gc = _run(engine, sc, wave, backend=True, check=True)
    assert gc["gpu_searches"] > 0
    assert gc["search_mismatches"] == 0
    assert gc["gpu_search_redo"] == 0
    assert len(glog) == len(hlog) and glog.tobytes() == hlog.tobytes()
    assert gedges.tobytes() == hedges.tobytes()
    assert gc["astar_pops"] == hc["astar_pops"] and gc["astar_pushes"] == hc["astar_pushes"]


def test_heap_overflow_is_repeated_on_the_host(engine):
    # a 2048-entry heap slab overflows on most searches of a 120-view graph: those are redone by the host, same graph
    sc = dense_scene(120, seed=4)
    hlog, hedges, hc = _run(engine, sc, 256, backend=False, check=False)
    os.environ["PGI_ASTAR_HEAP"] = "2048"
    try:
        glog, gedges, gc = _run(engine, sc, 256, backend=True, check=True)
    finally:
        os.environ.pop("PGI_ASTAR_HEAP", None)
    assert gc["gpu_search_redo"] > 0 and gc["search_mismatches"] == 0
    assert glog.tobytes() == hlog.tobytes() and gedges.tobytes() == hedges.tobytes()


def test_real_scene_with_device_search(oracle):
    # the complete product path (PoseGraphBuilder.run: device A* + verification kernels) against the sequential oracle
    from test_gpu_scene import run_and_compare

    sc = S.make_scene(n_views=16, n_corr=300, outlier_ratio=0.3, seed=31, n_points=900)
    os.environ["PGB_SEARCH_CHECK"] = "1"
    try:
        pgb, ostats = run_and_compare(oracle, sc, prefetch_fallback=True, wave_size=64, gpu_search=True, gpu_search_min_batch=1)
    finally:
        os.environ.pop("PGB_SEARCH_CHECK", None)
    assert pgb.counters["gpu_searches"] > 0 and pgb.counters["search_mismatches"] == 0
