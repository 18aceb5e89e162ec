"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes loader for the oracle's epipolar-hashing run (pgo_hashing.hpp / pgo_hashing_api.cpp).  The library is compiled on
first use with the flags of oracle/Makefile into a temporary directory keyed by the sources' hash, so the repository tree
is never written.  Only tests/ and scripts may import this module; the product package never does.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from .pgo_oracle import PAIRLOG_DTYPE

_HERE = os.path.dirname(os.path.abspath(__file__))
_FLAGS = ["-std=c++17", "-O3", "-ftree-vectorize", "-funroll-loops", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall",
          "-Wno-unused-variable", "-shared"]
_lib = None


def build():
    srcs = sorted(f for f in os.listdir(_HERE) if f.endswith((".hpp", ".cpp")))
    h = hashlib.sha256()
    for f in srcs:
        with open(os.path.join(_HERE, f), "rb") as fh:
            h.update(f.encode() + fh.read())
    out = os.path.join(tempfile.gettempdir(), f"pgo_hashing_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = out + f".{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++")] + _FLAGS + ["-o", tmp, os.path.join(_HERE, "pgo_hashing_api.cpp"),
                                                                          "-lpthread"])
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.pgo_run_scene_hashing.restype = C.c_void_p
        for n in ("pgo_hashing_pairlog_size", "pgo_hashing_log_count", "pgo_hashing_edge_count"):
            getattr(L, n).restype = C.c_uint64
            getattr(L, n).argtypes = [C.c_void_p] if n != "pgo_hashing_pairlog_size" else []
        L.pgo_hashing_free.argtypes = [C.c_void_p]
        L.pgo_hashing_copy.argtypes = [C.c_void_p] * 7
        _lib = L
    return _lib


def _a(x, dt):
    return np.ascontiguousarray(x, dtype=dt)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run_scene_hashing(scene, sim_threshold=0.0, thr_px=0.4, min_inliers=20, min_points=50, max_depth=5, weight=0.8,
                      use_path_finding=True, max_tracklets=5000, max_points_hashing=100, bin_number=45):
    """processImages with epipolar hashing, sequential.  scene: run_scene's keys plus desc[sum K, dim] f32.
    Returns (log, edges, sources): log as pgo_oracle.run_scene; edges (src, dst, q[4], t[3], score) in commit order;
    sources (source: 0 skipped / 1 quick / 2 full, guided_rows), one per log record."""
    L = lib()
    assert L.pgo_hashing_pairlog_size() == PAIRLOG_DTYPE.itemsize
    focal, size, sim = _a(scene["focal"], np.float64), _a(scene["size"], np.float64), _a(scene["sim"], np.float64)
    kpo, kp = _a(scene["kp_offset"], np.uint64), _a(scene["kp"], np.float32)
    desc = _a(scene["desc"], np.float32)
    pv, mo = _a(scene["pair_views"], np.uint32), _a(scene["m_offset"], np.uint64)
    mt = _a(scene["matches"], np.uint32).reshape(-1, 2)
    h = C.c_void_p(L.pgo_run_scene_hashing(
        C.c_uint64(len(focal)), _p(focal), _p(size), _p(sim), _p(kpo), _p(kp), _p(desc), C.c_int(desc.shape[1]),
        C.c_uint64(len(pv)), _p(pv), _p(mo), _p(mt), C.c_double(sim_threshold), C.c_double(thr_px), C.c_uint64(min_inliers),
        C.c_uint64(min_points), C.c_uint64(max_depth), C.c_double(weight), C.c_int(1 if use_path_finding else 0),
        C.c_uint64(max_tracklets), C.c_uint64(max_points_hashing), C.c_int(bin_number)))
    n, ne = int(L.pgo_hashing_log_count(h)), int(L.pgo_hashing_edge_count(h))
    log = np.zeros(n, dtype=PAIRLOG_DTYPE)
    src, rows = np.zeros(max(n, 1), dtype=np.uint8), np.zeros(max(n, 1), dtype=np.uint32)
    es, ed, ev = np.zeros(max(ne, 1), dtype=np.uint32), np.zeros(max(ne, 1), dtype=np.uint32), np.zeros((max(ne, 1), 8))
    L.pgo_hashing_copy(h, _p(log) if n else None, _p(src), _p(rows), _p(es), _p(ed), _p(ev))
    L.pgo_hashing_free(h)
    edges = np.zeros(ne, dtype=[("src", np.uint32), ("dst", np.uint32), ("q", np.float64, (4,)), ("t", np.float64, (3,)),
                                ("score", np.float64)])
    edges["src"], edges["dst"] = es[:ne], ed[:ne]
    edges["q"], edges["t"], edges["score"] = ev[:ne, :4], ev[:ne, 4:7], ev[:ne, 7]
    sources = np.zeros(n, dtype=[("source", np.uint8), ("guided_rows", np.uint32)])
    sources["source"], sources["guided_rows"] = src[:n], rows[:n]
    return log, edges, sources
