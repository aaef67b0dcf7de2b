"""Generate tests/golden/ref_nanoflann.json and tests/golden/scan_crop.ply (committed fixtures).

The tests that pin the oracle and the CUDA path to the reference's own code compare against these two files, so they
run on any machine, with or without the reference's sources. Regenerate them where the reference's source tree is
available and oracle/_ref has been built from it (oracle/Makefile, target `ref`):

    python tests/golden/make_ref_golden.py <reference source tree>

ref_nanoflann.json holds what the reference's vendored nanoflann (oracle.RefKnn) and the restated loops driven by it
answer on the tests' seeded inputs: sha256 digests of the exact arrays, transforms as float32 values. A nearest-neighbour
index array is digested with its exact distance ties resolved to the lowest index (the rule of the brute-force
restatement and of the CUDA path; nanoflann keeps the first point its traversal meets), and the number of entries that
resolution changed is stored next to it.

scan_crop.ply holds the vertices of the reference's bundled scan examples/test_clouds/test.ply that fall inside a box of
whole 12 mm voxels, in file order and in the scan's own binary layout: downsampled at 12 mm it must give exactly the rows
of tests/golden/config1_cloud.npz listed in the JSON.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
JSON = os.path.join(HERE, "ref_nanoflann.json")
CROP = os.path.join(HERE, "scan_crop.ply")
FLT_MAX = np.float32(np.finfo(np.float32).max)
# the crop: 12 mm voxel keys floor(p * float32(1 / 0.012)) in [lo, hi) on every axis
CROP_LO, CROP_HI = (-72, 18, 72), (-54, 36, 90)


def load():
    with open(JSON) as f:
        return json.load(f)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def lowest_on_ties(knn, q, idx, d2, k=4):
    """idx with every exact tie of its squared distance resolved to the lowest index; and how many entries changed."""
    out = idx.copy()
    hit = np.flatnonzero(idx >= 0)
    ni, nd, _ = knn.neighborhoods(q[hit], k, FLT_MAX)
    tied = nd.view(np.uint32) == d2[hit, None].view(np.uint32)
    assert tied.any(axis=1).all() and not tied[:, -1].any(), "a tie wider than k"
    out[hit] = np.where(tied, ni, np.iinfo(np.int64).max).min(axis=1)
    return out, int((out != idx).sum())


def knn1_entry(knn, q, max_d2):
    idx, d2 = knn.query(q, max_d2)
    low, ties = lowest_on_ties(knn, q, idx, d2)
    return {"idx": sha(low), "d2": sha(d2), "ties": ties}


def read_ply(path):
    """(header bytes, structured vertex array) of a binary little-endian PLY in the scan's layout."""
    with open(path, "rb") as f:
        header = b""
        while not header.endswith(b"end_header\n"):
            header += f.readline()
        n = int([ln for ln in header.decode().splitlines() if ln.startswith("element vertex")][0].split()[-1])
        dt = np.dtype([("p", "<f4", 3), ("c", "u1", 3), ("n", "<f4", 3), ("radius", "<f4")])
        return header, np.frombuffer(f.read(n * dt.itemsize), dtype=dt, count=n)


def crop_keys(p):
    return np.floor(p * np.float32(1.0 / 0.012)).astype(np.int64)


def make_crop(orc, scan):
    header, v = read_ply(scan)
    k = crop_keys(v["p"])
    keep = np.all((k >= CROP_LO) & (k < CROP_HI), axis=1)
    crop = v[keep]
    with open(CROP, "wb") as f:
        f.write(header.replace(f"element vertex {v.shape[0]}\n".encode(), f"element vertex {crop.shape[0]}\n".encode()))
        f.write(crop.tobytes())
    # rows of the committed fixture (the whole scan downsampled at 12 mm) whose voxel lies in the box, in fixture order
    p, n = np.ascontiguousarray(v["p"]), np.ascontiguousarray(v["n"])
    _, rows = np.unique(crop_keys(p), axis=0, return_index=True)
    p12, n12, _ = orc.grid_downsample(p, 0.012, normals=n)
    fix = np.load(os.path.join(HERE, "config1_cloud.npz"))
    assert np.array_equal(p12.view(np.uint32), fix["points"].view(np.uint32))
    inside = np.all((crop_keys(p[rows]) >= CROP_LO) & (crop_keys(p[rows]) < CROP_HI), axis=1)
    # map order of the voxel keys = np.unique's lexicographic order, so fixture row r is the r-th unique key
    fixture_rows = np.flatnonzero(inside)
    cp, cn = np.ascontiguousarray(crop["p"]), np.ascontiguousarray(crop["n"])
    got_p, got_n, _ = orc.grid_downsample(cp, 0.012, normals=cn)
    assert np.array_equal(got_p.view(np.uint32), p12[fixture_rows].view(np.uint32))
    assert np.array_equal(got_n.view(np.uint32), n12[fixture_rows].view(np.uint32))
    return {"n_vertices": int(crop.shape[0]), "fixture_rows": fixture_rows.tolist(),
            "n_bins_5mm": int(orc.grid_downsample(cp, 0.005, normals=cn)[0].shape[0])}


def full_size_entry(orc, n, iters, kw, with_normals, noise):
    """tests/test_gpu_full_size.py::_full_size_parity: the restated ICP loop driven by the reference kd-tree."""
    from cilantro_b200 import synth

    dst, src, nrm, _ = synth.icp_pair(n, seed=1, noise=noise, with_normals=with_normals)
    knn = orc.RefKnn(dst)
    ref = orc.icp(dst, src, knn, dst_n=nrm, max_iter=iters, tol=0.0, accum_double=True, **kw)
    ref32 = orc.icp(dst, src, knn, dst_n=nrm, max_iter=iters, tol=0.0, accum_double=False, **kw)
    T = ref["T"]
    o1, o2, ov = orc.find_correspondences(T, src, knn, kw["max_d2"])
    low, ties = lowest_on_ties(knn, orc.transform_points(T, src[o2]), o1, ov)
    return {"iterations": ref["iterations"], "T": T.reshape(-1).tolist(), "num_corr": ref["num_corr"],
            "T_fp32_sums": ref32["T"].reshape(-1).tolist(), "num_corr_fp32_sums": ref32["num_corr"],
            "corr": {"n": int(o1.size), "first": sha(low), "second": sha(o2), "value": sha(ov), "ties": ties}}


def outlier_normals_entry(orc):
    """tests/test_gpu_knn.py::test_normals_with_isolated_outliers: covariances of k = 10 neighbourhoods from the reference
    kd-tree for the surface points and brute force (ascending (d2, index)) for the outliers, whose nearest surface points
    tie in fp32 d2; rows where the 10th and 11th neighbours tie are left out of the digest."""
    from cilantro_b200 import synth

    pts, _ = synth.surface_cloud(300_000, seed=8, noise=0.0005)
    rng = np.random.default_rng(9)
    outliers = (np.array([0.5, 0.5, 0.5]) + 3.0 * rng.standard_normal((25, 3))).astype(np.float32)
    cloud = np.vstack([pts, outliers]).astype(np.float32)
    knn = orc.RefKnn(cloud)
    idx, d2, cnt = knn.neighborhoods(cloud, 10, orc.FLT_MAX)
    bi, bd, bc = orc.BruteKnn(cloud).neighborhoods(outliers, 10, orc.FLT_MAX)
    m = pts.shape[0]
    assert np.array_equal(np.sort(d2[m:], axis=1).view(np.uint32), bd.view(np.uint32))
    idx[m:], cnt[m:] = bi, bc
    want = orc.estimate_normals(cloud, knn, k=10, view_point=[0.5, 0.5, 10.0], neighbors=(idx, cnt))
    tied = (np.diff(knn.neighborhoods(cloud, 11, orc.FLT_MAX)[1], axis=1) == 0).any(axis=1)
    tied[m:] = False
    return {"outlier_d2": sha(bd), "tied": np.flatnonzero(tied).tolist(), "cov": sha(want[2][~tied])}


def compute(orc, scan):
    from cilantro_b200 import synth

    g = {"nanoflann_version": int(orc.ref().ref_nanoflann_version())}
    # tests/test_oracle_kat.py
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 1, 1], [1, 0, 1], [1, 1, 0], [1, 1, 1]], np.float32)
    idx, d2 = orc.RefKnn(pts).knn_in_radius([0.1, 0.1, 0.4], 2, 1.001)
    g["kd_tree_example"] = {"idx": idx.tolist(), "d2": d2.astype(np.float64).tolist()}
    dst, src, _, T_ref = synth.icp_pair(60000, seed=4, noise=0.003, n_src=20000)
    q = orc.transform_points(T_ref.astype(np.float32), src)
    knn = orc.RefKnn(dst)
    g["knn1_60k"] = [knn1_entry(knn, q, r2) for r2 in (np.float32(0.004**2), np.float32(0.05**2), FLT_MAX)]
    g["nn1_60k_d2"] = sha(knn.nn(q)[1])
    # tests/test_oracle_normals.py
    pts = np.random.default_rng(5).random((5000, 3), dtype=np.float32)
    knn = orc.RefKnn(pts)
    g["neighbourhoods_5k"] = []
    for k, r2 in ((8, orc.FLT_MAX), (16, 0.05**2)):
        ri, rd, rc = knn.neighborhoods(pts, k, r2)
        g["neighbourhoods_5k"].append({"idx": sha(ri), "d2": sha(rd), "cnt": sha(rc)})
    rn = orc.estimate_normals(pts, knn, k=10, view_point=[0.5, 0.5, 3.0])
    g["normals_5k"] = {"cov": sha(rn[2]), "normals": sha(rn[0]), "radius_cnt": sha(knn.neighborhoods(pts, 0, 0.04**2, stride=1)[2])}
    # tests/test_oracle_engine.py
    dst, src, _, T_ref = synth.icp_pair(20000, seed=4, noise=0.003, n_src=15000)
    T0 = (0.7 * np.asarray(T_ref) + 0.3 * np.hstack([np.eye(3), np.zeros((3, 1))])).astype(np.float32)
    max_d2 = np.float32((2.0 * 20000 ** (-1.0 / 3.0)) ** 2)
    knn = orc.RefKnn(dst)
    g["engine_f2s"] = []
    for mode in ENGINE_MODES:
        a = orc.engine_correspondences(dst, src, T0, knn, max_d2, f2s_reference=True, **mode)
        g["engine_f2s"].append({"n": int(a[0].size), "first": sha(a[0]), "second": sha(a[1]), "value": sha(a[2])})
    ra = orc.icp(dst, src, knn, f2s_reference=True, max_d2=max_d2, **ENGINE_ICP)
    g["engine_icp"] = {"T": ra["T"].reshape(-1).tolist(), "num_corr": ra["num_corr"]}
    # tests/test_gpu_knn.py
    dst, src, _, T_ref = synth.icp_pair(250000, seed=1, noise=0.001)
    g["knn1_250k"] = knn1_entry(orc.RefKnn(dst), orc.transform_points(T_ref.astype(np.float32), src), np.float32(0.02**2))
    rng = np.random.default_rng(23)
    dst = rng.random((15000, 3), dtype=np.float32)
    qry = rng.random((800, 3), dtype=np.float32)
    knn = orc.RefKnn(dst)
    _, _, cnt = knn.neighborhoods(qry, 0, 0.05**2, stride=1)
    ri, rd, cnt = knn.neighborhoods(qry, 0, 0.05**2, stride=int(cnt.max()))
    used = np.arange(ri.shape[1])[None, :] < cnt[:, None]
    g["radius_15k"] = {"cnt": sha(cnt.astype(np.int64)), "idx": sha(ri[used]), "d2": sha(rd[used])}
    g["normals_outliers_300k"] = outlier_normals_entry(orc)
    # tests/test_config1_real_scan.py, tests/test_ply_io.py
    g["scan_crop"] = make_crop(orc, scan)
    # tests/test_gpu_full_size.py
    g["full_size_p2p_1m"] = full_size_entry(orc, 1_000_000, 15, dict(metric="p2p", max_d2=np.float32(0.02**2)),
                                            False, 0.001)
    g["full_size_combined_10m"] = full_size_entry(
        orc, 10_000_000, 10, dict(metric="combined", max_d2=np.float32(0.01**2), w_pt=0.1, w_pl=1.0), True, 0.001)
    return g


# tests/test_oracle_engine.py::test_first_to_second_search_pinned_on_reference_nanoflann
ENGINE_MODES = (dict(search_dir="first_to_second"), dict(search_dir="first_to_second", one_to_one=True),
                dict(search_dir="both"), dict(search_dir="both", require_reciprocal=True, inlier_fraction=0.7))
ENGINE_ICP = dict(metric="p2p", max_iter=6, tol=0.0, search_dir="both", require_reciprocal=True)


if __name__ == "__main__":
    import oracle

    oracle.build()
    assert oracle.have_ref(), "oracle/_ref (the reference's nanoflann) is not built"
    g = compute(oracle, os.path.join(sys.argv[1], "examples", "test_clouds", "test.ply"))
    with open(JSON, "w") as f:
        json.dump(g, f, indent=1)
    print(f"wrote {JSON} and {CROP} ({g['scan_crop']['n_vertices']} vertices)")
