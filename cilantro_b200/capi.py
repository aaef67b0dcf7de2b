"""ctypes binding of libcilantro_b200.so (the C ABI declared in include/cilantro_b200.h).

This is harness plumbing for tests/ and bench.py: every call goes through the exported C entry
points, exactly as a cgo / JNI / C++ caller would. There is no Python compute path and no CPU
fallback: loading fails loudly if the shared library is missing, and cb_context_create fails if no
CUDA device is present.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CILANTRO_B200_LIB", os.path.join(_HERE, "libcilantro_b200.so"))

CB_OK = 0


class CbError(RuntimeError):
    pass


class IcpParams(C.Structure):
    _fields_ = [
        ("metric", C.c_int32),
        ("max_iter", C.c_int32),
        ("tol", C.c_float),
        ("max_d2", C.c_float),
        ("w_pt", C.c_float),
        ("w_pl", C.c_float),
        ("max_opt_iter", C.c_int32),
        ("opt_tol", C.c_float),
        ("T_init", C.c_float * 12),
        ("flush_l2", C.c_int32),
        ("timing", C.c_int32),
        ("search_dir", C.c_int32),
        ("require_reciprocal", C.c_int32),
        ("one_to_one", C.c_int32),
        ("host_loop", C.c_int32),
        ("inlier_fraction", C.c_double),
        ("pt_weight_kind", C.c_int32),
        ("pl_weight_kind", C.c_int32),
        ("pt_weight_coeff", C.c_float),
        ("pl_weight_coeff", C.c_float),
    ]


def rbf_coeff(sigma):
    """RBFKernelWeightEvaluator's coefficient, in float like the reference: -(0.5f) / (sigma * sigma)."""
    sg = np.float32(sigma)
    return float(np.float32(-0.5) / (sg * sg))


SEARCH_DIR = {"second_to_first": 0, "first_to_second": 1, "both": 2}


class IcpResult(C.Structure):
    _fields_ = [
        ("T", C.c_float * 12),
        ("iterations", C.c_int32),
        ("last_delta", C.c_float),
        ("converged", C.c_int32),
        ("num_corr", C.c_uint64),
        ("gpu_ms_total", C.c_double),
        ("gpu_ms_search", C.c_double),
        ("kernel_launches", C.c_uint64),
    ]


class KMeansResult(C.Structure):
    _fields_ = [("iterations", C.c_uint64), ("gpu_ms_total", C.c_double), ("kernel_launches", C.c_uint64)]


class RansacResult(C.Structure):
    _fields_ = [
        ("T", C.c_float * 12),
        ("iterations", C.c_uint64),
        ("num_inliers", C.c_uint64),
        ("best_iteration", C.c_uint64),
        ("gpu_ms_total", C.c_double),
        ("kernel_launches", C.c_uint64),
    ]


# every symbol include/cilantro_b200.h declares (tests/test_capi_host.py checks that the .so exports them and that this list matches the header)
EXPORTED = [
    "cb_last_error", "cb_version",
    "cb_context_create", "cb_context_destroy", "cb_context_synchronize", "cb_context_device_info",
    "cb_context_kernel_launches", "cb_context_flush_l2",
    "cb_comm_unique_id", "cb_context_init_comm", "cb_context_comm_info", "cb_comm_ipc_handle", "cb_comm_ipc_attach",
    "cb_comm_ipc_detach",
    "cb_cloud_create", "cb_cloud_create_pair", "cb_cloud_create_from_device", "cb_cloud_create_replicated", "cb_cloud_destroy", "cb_cloud_size", "cb_cloud_grid_info",
    "cb_cloud_estimate_normals", "cb_grid_downsample", "cb_cloud_grid_downsample", "cb_cloud_download",
    "cb_knn1_radius", "cb_knn_radius", "cb_radius_search", "cb_find_correspondences",
    "cb_icp_default_params", "cb_icp_create", "cb_icp_destroy", "cb_icp_estimate", "cb_icp_iteration_times",
    "cb_icp_correspondences", "cb_icp_residuals", "cb_icp_accumulate", "cb_icp_loop_cache",
    "cb_solve_kabsch_moments", "cb_solve_gauss_newton", "cb_solve_rotation", "cb_compose",
    "cb_kmeans_cluster", "cb_kmeans_assign", "cb_kmeans_seed_indices",
    "cb_ransac_score", "cb_ransac_residuals", "cb_ransac_rigid",
    "cb_mean_cov", "cb_pca", "cb_transform_points", "cb_cloud_segment",
]

_lib = None


def lib():
    """Load the shared library. Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CbError(
                f"{LIB_PATH} is missing: build it with `python -m cilantro_b200.build` "
                "(cilantro_b200 has no CPU / PyTorch fallback)")
        _lib = C.CDLL(LIB_PATH)
        _lib.cb_last_error.restype = C.c_char_p
        _lib.cb_version.restype = C.c_char_p
        _lib.cb_cloud_size.restype = C.c_size_t
        _lib.cb_context_kernel_launches.restype = C.c_uint64
        _lib.cb_context_kernel_launches.argtypes = [C.c_void_p]
    return _lib


def _check(rc):
    if rc < 0:
        raise CbError(f"cilantro_b200 error {rc}: {lib().cb_last_error().decode()}")
    return rc


def _f32(a, cols=3):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if cols is not None:
        assert a.ndim == 2 and a.shape[1] == cols, a.shape
    return a


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _T(T):
    return np.ascontiguousarray(T, dtype=np.float32).reshape(3, 4)


def identity():
    return np.hstack([np.eye(3, dtype=np.float32), np.zeros((3, 1), np.float32)])


class Context:
    def __init__(self, device=0):
        h = C.c_void_p()
        _check(lib().cb_context_create(C.c_int(device), C.byref(h)))
        self.h = h
        self.device = device
        self._children = weakref.WeakSet()  # clouds / icp objects must be destroyed before the context

    def _adopt(self, child):
        self._children.add(child)

    def close(self):
        if self.h:
            for child in list(self._children):
                child.close()
            lib().cb_context_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        _check(lib().cb_context_synchronize(self.h))

    def device_info(self):
        sm = C.c_int()
        hbm = C.c_size_t()
        name = C.create_string_buffer(64)
        _check(lib().cb_context_device_info(self.h, C.byref(sm), C.byref(hbm), name))
        return {"sm_count": sm.value, "hbm_bytes": hbm.value, "name": name.value.decode()}

    def kernel_launches(self):
        return int(lib().cb_context_kernel_launches(self.h))

    def flush_l2(self):
        _check(lib().cb_context_flush_l2(self.h))

    def init_comm(self, unique_id: bytes, rank: int, world: int):
        buf = C.create_string_buffer(unique_id, 128)
        _check(lib().cb_context_init_comm(self.h, buf, C.c_int(rank), C.c_int(world)))

    def ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        _check(lib().cb_comm_ipc_handle(self.h, buf))
        return buf.raw

    def ipc_attach(self, handles: bytes):
        buf = C.create_string_buffer(handles, len(handles))
        _check(lib().cb_comm_ipc_attach(self.h, buf))

    def ipc_detach(self):
        _check(lib().cb_comm_ipc_detach(self.h))

    def comm_info(self):
        r, w = C.c_int(), C.c_int()
        _check(lib().cb_context_comm_info(self.h, C.byref(r), C.byref(w)))
        return r.value, w.value


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _check(lib().cb_comm_unique_id(buf))
    return buf.raw


class Cloud:
    """Device-resident point set (+ optional normals); see cb_cloud_create."""

    def __init__(self, ctx, xyz=None, normals=None, index_offset=0, device_ptr=None, device_normals_ptr=None, n=None):
        self.ctx = ctx
        h = C.c_void_p()
        if device_ptr is not None:
            _check(lib().cb_cloud_create_from_device(ctx.h, C.c_void_p(device_ptr),
                                                     C.c_void_p(device_normals_ptr) if device_normals_ptr else None,
                                                     C.c_size_t(n), C.c_uint64(index_offset), C.byref(h)))
            self.n = n
        else:
            xyz = _f32(xyz)
            nrm = _f32(normals) if normals is not None else None
            if nrm is not None:
                assert nrm.shape == xyz.shape
            _check(lib().cb_cloud_create(ctx.h, _p(xyz), _p(nrm), C.c_size_t(xyz.shape[0]), C.c_uint64(index_offset),
                                         C.byref(h)))
            self.n = xyz.shape[0]
        self.h = h
        ctx._adopt(self)

    def close(self):
        if self.h:
            lib().cb_cloud_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def estimate_normals(self, k=0, radius2=0.0, view_point=None, use_current_as_ref=False, want_curvature=True,
                         want_cov=False, fetch=True):
        """cb_cloud_estimate_normals: kNN (k>0), kNN-in-radius (k>0, radius2>0) or radius (k=0) neighbourhoods.
        Stores the normals in the cloud; returns dict(normals, curvature, cov6, gpu_ms)."""
        n = self.n
        nrm = np.empty((n, 3), np.float32) if fetch else None
        curv = np.empty(n, np.float32) if (fetch and want_curvature) else None
        cov = np.empty((n, 6), np.float32) if (fetch and want_cov) else None
        vp = None if view_point is None else np.ascontiguousarray(view_point, np.float32).reshape(3)
        ms = C.c_float()
        _check(lib().cb_cloud_estimate_normals(self.ctx.h, self.h, C.c_int(k), C.c_float(radius2), _p(vp),
                                               C.c_int(int(use_current_as_ref)), _p(nrm), _p(curv), _p(cov), C.byref(ms)))
        return {"normals": nrm, "curvature": curv, "cov6": cov, "gpu_ms": ms.value}

    @classmethod
    def replicated(cls, ctx, xyz_block, normals_block, first_index, n_total):
        """cb_cloud_create_replicated: every rank passes its contiguous block; all of them get the whole cloud."""
        xb = _f32(xyz_block)
        nb = _f32(normals_block) if normals_block is not None else None
        h = C.c_void_p()
        _check(lib().cb_cloud_create_replicated(ctx.h, _p(xb), _p(nb), C.c_size_t(xb.shape[0]), C.c_uint64(first_index),
                                                C.c_size_t(n_total), C.byref(h)))
        return cls._wrap(ctx, h)

    @classmethod
    def _wrap(cls, ctx, handle):
        self = cls.__new__(cls)
        self.ctx = ctx
        self.h = handle
        self.n = int(lib().cb_cloud_size(handle))
        ctx._adopt(self)
        return self

    def grid_downsample(self, bin_size, min_points=1, order=0):
        """cb_cloud_grid_downsample: a new device-resident Cloud (points + normals if present); .gpu_ms = device time."""
        h = C.c_void_p()
        ms = C.c_float()
        _check(lib().cb_cloud_grid_downsample(self.ctx.h, self.h, C.c_float(bin_size), C.c_size_t(min_points),
                                              C.c_int(order), C.byref(h), C.byref(ms)))
        out = Cloud._wrap(self.ctx, h)
        out.gpu_ms = ms.value
        return out

    def download(self, normals=False):
        xyz = np.empty((self.n, 3), np.float32)
        nrm = np.empty((self.n, 3), np.float32) if normals else None
        _check(lib().cb_cloud_download(self.ctx.h, self.h, _p(xyz), _p(nrm)))
        return (xyz, nrm) if normals else xyz

    def grid_info(self):
        edge = C.c_float()
        dims = (C.c_int * 3)()
        occ = C.c_double()
        _check(lib().cb_cloud_grid_info(self.h, C.byref(edge), dims, C.byref(occ)))
        return {"cell_edge": edge.value, "dims": list(dims), "mean_occupancy": occ.value}


def cloud_pair(ctx, xyz_a, normals_a, xyz_b, normals_b, offset_a=0, offset_b=0):
    """cb_cloud_create_pair: two indexed Clouds; the second upload overlaps the first grid build."""
    xa, xb = _f32(xyz_a), _f32(xyz_b)
    na = _f32(normals_a) if normals_a is not None else None
    nb = _f32(normals_b) if normals_b is not None else None
    ha, hb = C.c_void_p(), C.c_void_p()
    _check(lib().cb_cloud_create_pair(ctx.h, _p(xa), _p(na), C.c_size_t(xa.shape[0]), C.c_uint64(offset_a), _p(xb), _p(nb),
                                      C.c_size_t(xb.shape[0]), C.c_uint64(offset_b), C.byref(ha), C.byref(hb)))
    return Cloud._wrap(ctx, ha), Cloud._wrap(ctx, hb)


def radius_search(ctx, ref, qry, radius2, T=None):
    """cb_radius_search: CSR (offsets [nq + 1], idx, d2) of all ref points with d2 < radius2 per query."""
    offsets = np.zeros(qry.n + 1, np.uint64)
    total = C.c_size_t()
    Tm = _T(T) if T is not None else None
    _check(lib().cb_radius_search(ctx.h, ref.h, qry.h, _p(Tm), C.c_float(radius2), _p(offsets), None, None,
                                  C.c_size_t(0), C.byref(total)))
    m = total.value
    idx = np.empty(m, np.int64)
    d2 = np.empty(m, np.float32)
    if m:
        _check(lib().cb_radius_search(ctx.h, ref.h, qry.h, _p(Tm), C.c_float(radius2), _p(offsets), _p(idx), _p(d2),
                                      C.c_size_t(m), C.byref(total)))
    return offsets.astype(np.int64), idx, d2


def grid_downsample(ctx, xyz, bin_size, normals=None, colors=None, min_points=1, order=0):
    """cb_grid_downsample on host arrays: returns (points, normals or None, colors or None)."""
    xyz = _f32(xyz)
    n = xyz.shape[0]
    nrm = _f32(normals) if normals is not None else None
    col = _f32(colors) if colors is not None else None
    o_xyz = np.empty((n, 3), np.float32)
    o_nrm = np.empty((n, 3), np.float32) if nrm is not None else None
    o_col = np.empty((n, 3), np.float32) if col is not None else None
    m = C.c_size_t()
    _check(lib().cb_grid_downsample(ctx.h, _p(xyz), _p(nrm), _p(col), C.c_size_t(n), C.c_float(bin_size),
                                    C.c_size_t(min_points), C.c_int(order), _p(o_xyz), _p(o_nrm), _p(o_col),
                                    C.byref(m)))
    m = m.value
    return o_xyz[:m].copy(), (o_nrm[:m].copy() if o_nrm is not None else None), (o_col[:m].copy() if o_col is not None else None)


def knn1_radius(ctx, ref, qry, T=None, max_d2=np.finfo(np.float32).max):
    idx = np.empty(qry.n, np.int64)
    d2 = np.empty(qry.n, np.float32)
    Tm = _T(T) if T is not None else None
    _check(lib().cb_knn1_radius(ctx.h, ref.h, qry.h, _p(Tm), C.c_float(max_d2), _p(idx), _p(d2)))
    return idx, d2


def knn_radius(ctx, ref, qry, k, T=None, max_d2=np.finfo(np.float32).max):
    idx = np.empty((qry.n, k), np.int64)
    d2 = np.empty((qry.n, k), np.float32)
    cnt = np.empty(qry.n, np.uint32)
    Tm = _T(T) if T is not None else None
    _check(lib().cb_knn_radius(ctx.h, ref.h, qry.h, _p(Tm), C.c_int(k), C.c_float(max_d2), _p(idx), _p(d2), _p(cnt)))
    return idx, d2, cnt


def find_correspondences(ctx, ref, qry, T=None, max_d2=1e-4):
    i1 = np.empty(qry.n, np.uint64)
    i2 = np.empty(qry.n, np.uint64)
    v = np.empty(qry.n, np.float32)
    cnt = C.c_size_t()
    Tm = _T(T) if T is not None else None
    _check(lib().cb_find_correspondences(ctx.h, ref.h, qry.h, _p(Tm), C.c_float(max_d2), _p(i1), _p(i2), _p(v),
                                         C.byref(cnt)))
    c = cnt.value
    return i1[:c].astype(np.int64), i2[:c].astype(np.int64), v[:c]


def transform_points(ctx, T, xyz):
    xyz = _f32(xyz)
    out = np.empty_like(xyz)
    _check(lib().cb_transform_points(ctx.h, _p(_T(T)), _p(xyz), C.c_size_t(xyz.shape[0]), _p(out)))
    return out


def icp_params(metric="p2p", max_iter=15, tol=1e-5, max_d2=1e-4, w_pt=0.0, w_pl=1.0, max_opt_iter=1, opt_tol=1e-5,
               T_init=None, flush_l2=False, timing=1, search_dir="second_to_first", inlier_fraction=1.0,
               require_reciprocal=False, one_to_one=False, host_loop=False, pt_rbf_sigma=None, pl_rbf_sigma=None):
    p = IcpParams()
    lib().cb_icp_default_params(C.byref(p))
    p.metric = 0 if metric == "p2p" else 1
    p.max_iter = int(max_iter)
    p.tol = tol
    p.max_d2 = max_d2
    p.w_pt, p.w_pl = w_pt, w_pl
    p.max_opt_iter = int(max_opt_iter)
    p.opt_tol = opt_tol
    Ti = identity() if T_init is None else _T(T_init)
    for i, v in enumerate(Ti.reshape(-1)):
        p.T_init[i] = float(v)
    p.flush_l2 = int(flush_l2)
    p.timing = int(timing)
    p.search_dir = SEARCH_DIR[search_dir] if isinstance(search_dir, str) else int(search_dir)
    p.inlier_fraction = float(inlier_fraction)
    p.require_reciprocal = int(require_reciprocal)
    p.one_to_one = int(one_to_one)
    p.host_loop = int(host_loop)
    if pt_rbf_sigma is not None:
        p.pt_weight_kind, p.pt_weight_coeff = 1, rbf_coeff(pt_rbf_sigma)
    if pl_rbf_sigma is not None:
        p.pl_weight_kind, p.pl_weight_coeff = 1, rbf_coeff(pl_rbf_sigma)
    return p


class Icp:
    """cb_icp_*: SimplePointToPointMetricRigidICP3f / SimpleCombinedMetricRigidICP3f."""

    def __init__(self, ctx, dst: Cloud, src: Cloud):
        self.ctx, self.dst, self.src = ctx, dst, src
        h = C.c_void_p()
        _check(lib().cb_icp_create(ctx.h, dst.h, src.h, C.byref(h)))
        self.h = h
        ctx._adopt(self)

    def close(self):
        if self.h:
            lib().cb_icp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def estimate(self, **kw):
        prm = kw.pop("params", None) or icp_params(**kw)
        res = IcpResult()
        _check(lib().cb_icp_estimate(self.h, C.byref(prm), C.byref(res)))
        times = np.zeros(max(res.iterations, 1), np.float64)
        n = lib().cb_icp_iteration_times(self.h, _p(times), C.c_int(times.shape[0]))
        return {
            "T": np.array(list(res.T), np.float32).reshape(3, 4),
            "iterations": int(res.iterations),
            "last_delta": float(res.last_delta),
            "converged": bool(res.converged),
            "num_corr": int(res.num_corr),
            "gpu_ms_total": float(res.gpu_ms_total),
            "gpu_ms_search": float(res.gpu_ms_search),
            "iter_ms": times[:max(n, 0)],
            "kernel_launches": int(res.kernel_launches),
        }

    def accumulate(self, T, **kw):
        prm = kw.pop("params", None) or icp_params(**kw)
        sums = np.zeros(28, np.float64)
        nv = _check(lib().cb_icp_accumulate(self.h, C.byref(prm), _p(_T(T)), _p(sums), C.c_int(28)))
        return sums[:nv]

    def correspondences(self):
        n = self.src.n + self.dst.n
        i1 = np.empty(n, np.uint64)
        i2 = np.empty(n, np.uint64)
        v = np.empty(n, np.float32)
        cnt = C.c_size_t()
        _check(lib().cb_icp_correspondences(self.h, _p(i1), _p(i2), _p(v), C.byref(cnt)))
        c = cnt.value
        return i1[:c].astype(np.int64), i2[:c].astype(np.int64), v[:c]

    def loop_cache(self):
        """cb_icp_loop_cache: (T_search 3x4, nearest dst index per source point or -1, queries searched by the last iteration)."""
        T = np.empty((3, 4), np.float32)
        near = np.empty(self.src.n, np.int64)
        cnt = C.c_uint64()
        _check(lib().cb_icp_loop_cache(self.h, _p(T), _p(near), C.byref(cnt)))
        return T, near, int(cnt.value)

    def residuals(self, T, **kw):
        prm = kw.pop("params", None) or icp_params(**kw)
        out = np.empty(self.src.n, np.float32)
        _check(lib().cb_icp_residuals(self.h, C.byref(prm), _p(_T(T)), _p(out)))
        return out


def solve_kabsch_moments(sums16):
    s = np.ascontiguousarray(sums16, np.float64)
    T = np.empty((3, 4), np.float32)
    ok = _check(lib().cb_solve_kabsch_moments(_p(s), _p(T)))
    return T, bool(ok)


def solve_gauss_newton(sums28, T_in=None):
    s = np.ascontiguousarray(sums28, np.float64)
    Ti = identity() if T_in is None else _T(T_in)
    To = np.empty((3, 4), np.float32)
    dn = C.c_float()
    _check(lib().cb_solve_gauss_newton(_p(s), _p(Ti), _p(To), C.byref(dn)))
    return To, dn.value


def solve_rotation(L):
    L = np.ascontiguousarray(L, np.float32).reshape(3, 3)
    R = np.empty((3, 3), np.float32)
    _check(lib().cb_solve_rotation(_p(L), _p(R)))
    return R


def compose(A, B):
    out = np.empty((3, 4), np.float32)
    _check(lib().cb_compose(_p(_T(A)), _p(_T(B)), _p(out)))
    return out


def kmeans_seed_indices(n, k, seed):
    out = np.empty(k, np.uint64)
    _check(lib().cb_kmeans_seed_indices(C.c_size_t(n), C.c_size_t(k), C.c_uint32(seed), _p(out)))
    return out.astype(np.int64)


def kmeans_assign(ctx, pts: Cloud, centroids, want_labels=True):
    cent = _f32(centroids)
    k = cent.shape[0]
    labels = np.empty(pts.n, np.uint64) if want_labels else None
    sums = np.empty((k, 3), np.float64)
    counts = np.empty(k, np.uint64)
    _check(lib().cb_kmeans_assign(ctx.h, pts.h, _p(cent), C.c_size_t(k), _p(labels), _p(sums), _p(counts)))
    return (labels.astype(np.int64) if want_labels else None), sums, counts.astype(np.int64)


def kmeans_cluster(ctx, pts: Cloud, centroids0, max_iter=100, tol=float(np.finfo(np.float32).eps), want_labels=True):
    cent = _f32(centroids0).copy()
    labels = np.empty(pts.n, np.uint64) if want_labels else None
    res = KMeansResult()
    _check(lib().cb_kmeans_cluster(ctx.h, pts.h, _p(cent), C.c_size_t(cent.shape[0]), C.c_size_t(max_iter),
                                   C.c_float(tol), _p(labels), C.byref(res)))
    return {
        "centroids": cent,
        "labels": labels.astype(np.int64) if want_labels else None,
        "iterations": int(res.iterations),
        "gpu_ms_total": float(res.gpu_ms_total),
        "kernel_launches": int(res.kernel_launches),
    }


def ransac_score(ctx, dst: Cloud, src: Cloud, T_h, thresh):
    T_h = np.ascontiguousarray(T_h, np.float32).reshape(-1, 3, 4)
    counts = np.empty(T_h.shape[0], np.uint32)
    _check(lib().cb_ransac_score(ctx.h, dst.h, src.h, _p(T_h), C.c_size_t(T_h.shape[0]), C.c_float(thresh), _p(counts)))
    return counts


def ransac_residuals(ctx, dst: Cloud, src: Cloud, T, thresh):
    res = np.empty(dst.n, np.float32)
    inl = np.empty(dst.n, np.uint64)
    cnt = C.c_size_t()
    _check(lib().cb_ransac_residuals(ctx.h, dst.h, src.h, _p(_T(T)), C.c_float(thresh), _p(res), _p(inl), C.byref(cnt)))
    return res, inl[:cnt.value].astype(np.int64)


def ransac_rigid(ctx, dst: Cloud, src: Cloud, seed, max_iter=100, thresh=0.01, inlier_count_thresh=None,
                 re_estimate=True):
    n = dst.n
    if inlier_count_thresh is None:
        inlier_count_thresh = n // 2 + n % 2
    res = RansacResult()
    inl = np.empty(n, np.uint64)
    resid = np.empty(n, np.float32)
    _check(lib().cb_ransac_rigid(ctx.h, dst.h, src.h, C.c_uint32(seed), C.c_size_t(inlier_count_thresh),
                                 C.c_size_t(max_iter), C.c_float(thresh), C.c_int(int(re_estimate)), C.byref(res),
                                 _p(inl), _p(resid)))
    return {
        "T": np.array(list(res.T), np.float32).reshape(3, 4),
        "iterations": int(res.iterations),
        "num_inliers": int(res.num_inliers),
        "best_iteration": int(res.best_iteration),
        "inliers": inl[: res.num_inliers].astype(np.int64),
        "residuals": resid,
        "gpu_ms_total": float(res.gpu_ms_total),
        "kernel_launches": int(res.kernel_launches),
    }


def mean_cov(ctx, pts: Cloud):
    mean = np.empty(3, np.float32)
    cov = np.empty((3, 3), np.float32)
    ok = _check(lib().cb_mean_cov(ctx.h, pts.h, _p(mean), _p(cov)))
    return mean, cov, bool(ok)


def pca(ctx, pts: Cloud):
    mean = np.empty(3, np.float32)
    cov = np.empty((3, 3), np.float32)
    ev = np.empty(3, np.float32)
    evec = np.empty((3, 3), np.float32)
    ok = _check(lib().cb_pca(ctx.h, pts.h, _p(mean), _p(cov), _p(ev), _p(evec)))
    return {"ok": bool(ok), "mean": mean, "cov": cov, "eigenvalues": ev, "eigenvectors": evec}


class SegmentParams(C.Structure):
    _fields_ = [
        ("k", C.c_int32),
        ("radius2", C.c_float),
        ("evaluator", C.c_int32),
        ("max_distance", C.c_float),
        ("max_angle", C.c_float),
        ("color_thresh", C.c_float),
        ("min_size", C.c_uint64),
        ("max_size", C.c_uint64),
    ]


SEGMENT_EVALUATORS = {"always_true": 0, "points": 1, "normals": 2, "colors": 3, "points_normals": 4,
                      "points_colors": 5, "normals_colors": 6, "points_normals_colors": 7}


def segment(ctx, cloud: Cloud, k=0, radius2=0.0, evaluator="always_true", max_distance=0.0, max_angle=0.0,
            color_thresh=0.0, min_size=1, max_size=2**64 - 1, seeds=None, normals=None, colors=None, want_ms=False):
    """cb_cloud_segment (ConnectedComponentExtraction3f::segment): returns (labels [n] int64, offsets [m + 1] int64,
    points [offsets[m]] int64, m), plus the stage times [total, neighbourhood + union, finalise] in ms when want_ms.
    seeds None = every point; normals None = the cloud's own."""
    n = cloud.n
    prm = SegmentParams(int(k), float(radius2), SEGMENT_EVALUATORS[evaluator] if isinstance(evaluator, str) else int(evaluator),
                        float(max_distance), float(max_angle), float(color_thresh), int(min_size), int(max_size))
    sd = None if seeds is None else np.ascontiguousarray(seeds, np.uint64)
    nr = None if normals is None else _f32(normals)
    cl = None if colors is None else _f32(colors)
    labels = np.empty(max(n, 1), np.uint64)
    offsets = np.zeros(n + 1, np.uint64)
    points = np.empty(max(n, 1), np.uint64)
    m = C.c_size_t()
    ms = np.zeros(3, np.float32)
    _check(lib().cb_cloud_segment(ctx.h, cloud.h, C.byref(prm), _p(sd), C.c_size_t(0 if sd is None else sd.shape[0]),
                                  _p(nr), _p(cl), _p(labels), _p(offsets), _p(points), C.byref(m), _p(ms) if want_ms else None))
    m = m.value
    out = (labels[:n].astype(np.int64), offsets[: m + 1].astype(np.int64), points[: int(offsets[m])].astype(np.int64), m)
    return out + (ms.astype(np.float64),) if want_ms else out
