"""ORACLE of connected-component segmentation (test infrastructure, not product code).

Compiles tests/cpp/segment_oracle.cpp — the serial restatement of extractConnectedComponents
(clustering/connected_component_extraction.hpp:162-265) — into a temporary directory on first use, and feeds it
neighbour lists from the oracle's kNN back ends (oracle.RefKnn = the reference's nanoflann where oracle/_ref was built,
oracle.BruteKnn otherwise) or from any (offsets, idx, d2) CSR the caller already has.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "segment_oracle.cpp")
_lib = None

FLT_MAX = float(np.finfo(np.float32).max)
EVALUATORS = {"always_true": 0, "points": 1, "normals": 2, "colors": 3, "points_normals": 4, "points_colors": 5,
              "normals_colors": 6, "points_normals_colors": 7}


def lib():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha1(f.read()).hexdigest()[:12]
        so = os.path.join(tempfile.gettempdir(), f"cb_segment_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            env = dict(os.environ)
            env.pop("CXX", None)
            tmp = so + f".{os.getpid()}"
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", _SRC,
                                   "-o", tmp], env=env)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_connected_components.restype = C.c_size_t
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def neighbour_lists(pts, k, radius2, knn):
    """KDTree::search(points.col(u), nh) for every u, as CSR (offsets [n + 1], idx, d2). The neighbourhood encoding is
    cb_cloud_segment's: k > 0 kNN (within radius2 when radius2 > 0), k == 0 radius2 > 0 radius, else empty."""
    pts = np.ascontiguousarray(pts, np.float32)
    n = pts.shape[0]
    if n == 0 or (k == 0 and not radius2 > 0):
        return np.zeros(n + 1, np.uint64), np.zeros(0, np.int64), np.zeros(0, np.float32)
    if k > 0:
        idx, d2, cnt = knn.neighborhoods(pts, k, float(radius2) if radius2 > 0 else FLT_MAX)
    else:
        _, _, cnt = knn.neighborhoods(pts, 0, float(radius2), stride=1)
        idx, d2, cnt = knn.neighborhoods(pts, 0, float(radius2), stride=max(1, int(cnt.max())))
    keep = np.arange(idx.shape[1])[None, :] < cnt[:, None].astype(np.int64)
    offsets = np.zeros(n + 1, np.uint64)
    offsets[1:] = np.cumsum(cnt, dtype=np.uint64)
    return offsets, np.ascontiguousarray(idx[keep], np.int64), np.ascontiguousarray(d2[keep], np.float32)


def connected_components(n, lists, evaluator="always_true", max_distance=0.0, max_angle=0.0, color_thresh=0.0,
                         min_size=1, max_size=2**64 - 1, seeds=None, normals=None, colors=None):
    """The serial reference loop over `lists` = (offsets, idx, d2). Returns (labels, offsets, points, m) like
    cilantro_b200.capi.segment."""
    off, idx, d2 = (np.ascontiguousarray(lists[0], np.uint64), np.ascontiguousarray(lists[1], np.int64),
                    np.ascontiguousarray(lists[2], np.float32))
    sd = None if seeds is None else np.ascontiguousarray(seeds, np.uint64)
    nr = None if normals is None else np.ascontiguousarray(normals, np.float32)
    cl = None if colors is None else np.ascontiguousarray(colors, np.float32)
    labels = np.empty(max(n, 1), np.uint64)
    seg_off = np.zeros(n + 1, np.uint64)
    seg_pts = np.empty(max(n, 1), np.uint64)
    kind = EVALUATORS[evaluator] if isinstance(evaluator, str) else int(evaluator)
    m = lib().orc_connected_components(C.c_size_t(n), _p(off), _p(idx), _p(d2), _p(sd),
                                       C.c_size_t(0 if sd is None else sd.shape[0]), C.c_int(kind),
                                       C.c_float(max_distance), C.c_float(max_angle), C.c_float(color_thresh),
                                       _p(nr), _p(cl), C.c_uint64(int(min_size)), C.c_uint64(int(max_size)),
                                       _p(labels), _p(seg_off), _p(seg_pts))
    return (labels[:n].astype(np.int64), seg_off[: m + 1].astype(np.int64), seg_pts[: int(seg_off[m])].astype(np.int64),
            int(m))


def segment(pts, knn, k=0, radius2=0.0, **kw):
    """neighbour_lists + connected_components: what ConnectedComponentExtraction3f::segment computes."""
    pts = np.ascontiguousarray(pts, np.float32)
    return connected_components(pts.shape[0], neighbour_lists(pts, k, radius2, knn), **kw)
