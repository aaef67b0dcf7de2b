#!/usr/bin/env python
"""Small-size pass over every kernel family of libcilantro_b200.so: the target of scripts/sanitize.sh
(compute-sanitizer memcheck / racecheck / synccheck). Each call is checked against the oracle or a property, so a
sanitizer-clean run is also a correct run. Sizes are tiny: the sanitizers slow kernels down 10-1000x."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from cilantro_b200 import capi, synth  # noqa: E402

N = int(os.environ.get("SANITIZE_N", "6000"))


def main():
    ctx = capi.Context(0)
    dst, src, nrm, T_ref = synth.icp_pair(N, seed=3, noise=0.002, with_normals=True)
    knn = oracle.BruteKnn(dst)
    d_dst, d_src = capi.Cloud(ctx, dst, nrm), capi.Cloud(ctx, src)
    max_d2 = np.float32(0.06 ** 2)
    # grid index + 1-NN kernel
    T = T_ref.astype(np.float32)
    idx, d2 = capi.knn1_radius(ctx, d_dst, d_src, T, max_d2)
    oi, od = knn.query(oracle.transform_points(T, src), max_d2)
    assert np.array_equal(idx, oi), "1-NN"
    icp = capi.Icp(ctx, d_dst, d_src)
    # device-resident loop (cold search kernel, cached pass, warm search kernel, device solve) and host loop
    for kw in (dict(metric="p2p"), dict(metric="combined", w_pt=0.1, w_pl=1.0),
               dict(metric="combined", w_pt=0.1, w_pl=1.0, pt_rbf_sigma=0.01, pl_rbf_sigma=0.01)):
        want = oracle.icp(dst, src, knn, dst_n=nrm if kw["metric"] == "combined" else None, max_iter=5, tol=0.0, max_d2=max_d2, **kw)
        for host in (False, True):
            got = icp.estimate(max_iter=5, tol=0.0, max_d2=max_d2, host_loop=host, **kw)
            assert got["num_corr"] == want["num_corr"] and np.linalg.norm(got["T"].astype(np.float64) - want["T"]) < 1e-5, (kw, host)
    icp.estimate(metric="p2p", max_iter=4, tol=0.0, max_d2=max_d2)
    icp.loop_cache()
    icp.correspondences()
    icp.residuals(T, metric="combined", w_pt=0.1, w_pl=1.0)
    # inner Gauss-Newton iterations (stored correspondences) and the engine modes (pair lists, radix sorts)
    icp.estimate(metric="combined", w_pt=0.1, w_pl=1.0, max_iter=3, max_opt_iter=3, opt_tol=0.0, tol=0.0, max_d2=max_d2)
    for extra in (dict(search_dir="both", require_reciprocal=True), dict(inlier_fraction=0.7), dict(one_to_one=True),
                  dict(search_dir="first_to_second")):
        icp.estimate(metric="p2p", max_iter=2, tol=0.0, max_d2=max_d2, **extra)
        icp.correspondences()
    # general-k kNN, radius lists, normals, downsample
    capi.knn_radius(ctx, d_dst, d_src, 8, T, np.float32(3e38))
    capi.radius_search(ctx, d_dst, d_src, np.float32(0.05 ** 2), T)
    sheet, _ = synth.surface_cloud(N, seed=5, noise=0.0005)
    c = capi.Cloud(ctx, sheet)
    ds = c.grid_downsample(0.03)
    ds.estimate_normals(k=8, view_point=[0.5, 0.5, 5.0])
    ds.estimate_normals(k=0, radius2=0.06 ** 2)
    # connected components: union passes (radius / kNN), seeded traversals, finalise
    col = np.random.default_rng(0).uniform(0, 1, (ds.n, 3)).astype(np.float32)
    for kw in (dict(radius2=0.06 ** 2, evaluator="normals", max_angle=0.2), dict(k=8, evaluator="points_colors",
               max_distance=0.05 ** 2, color_thresh=0.5, colors=col)):
        capi.segment(ctx, ds, min_size=2, **kw)
        capi.segment(ctx, ds, seeds=np.arange(0, ds.n, 37), **kw)
    # k-means, RANSAC, PCA
    pts, cent = synth.kmeans_data(N, 16, seed=1)
    capi.kmeans_cluster(ctx, capi.Cloud(ctx, pts), cent, max_iter=3, tol=0.0)
    rd, rs, _, _ = synth.ransac_pairs(N, 0.4, seed=2)
    c_rd, c_rs = capi.Cloud(ctx, rd), capi.Cloud(ctx, rs)
    capi.ransac_rigid(ctx, c_rd, c_rs, seed=5, max_iter=64, thresh=0.01)
    capi.pca(ctx, capi.Cloud(ctx, pts))
    ctx.close()
    print("sanitize target: all checks passed")


if __name__ == "__main__":
    main()
