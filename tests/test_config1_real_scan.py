"""BASELINE config 1 — the reference's own CPU-runnable case (examples/rigid_icp.cpp on the bundled scan
examples/test_clouds/test.ply) — on the committed fixture tests/golden/config1_cloud.npz (the scan, voxel-downsampled
at 12 mm by the oracle; tests/golden/make_config1_fixture.py).

CPU part: the oracle runs the example's recipe (rigid_icp.cpp:25-65, settings :119-123) and recovers tf_ref^-1 — the
self-checking property the example prints; a crop of the scan itself (tests/golden/scan_crop.ply) must downsample to
exactly the fixture's rows of the voxels it covers.
GPU part: the same recipe through the C ABI against the oracle: transforms within 1e-5, neighbour indices and residuals
bit-exact, plus downsampling and normal estimation on real scan data.
"""
import os

import numpy as np
import pytest

from cilantro_b200 import synth
from conftest import frob
from golden import make_ref_golden as ref_golden

FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "config1_cloud.npz")
# icp.setMaxNumberOfOptimizationStepIterations(1).setPointToPointMetricWeight(0).setPointToPlaneMetricWeight(1);
# setMaxDistance(0.1 * 0.1); setConvergenceTolerance(1e-4).setMaxNumberOfIterations(30)   (rigid_icp.cpp:119-123)
SETTINGS = dict(metric="combined", w_pt=0.0, w_pl=1.0, max_opt_iter=1, max_d2=np.float32(0.1 * 0.1))


def _scan():
    z = np.load(FIXTURE)
    return z["points"], z["normals"], int(z["n_source"]), int(z["n_bins_5mm"])


def test_fixture_matches_the_reference_scan(orc):
    pts, nrm, n_source, n5 = _scan()
    assert pts.shape == nrm.shape and pts.shape[0] > 40000 and n_source == 573663
    assert np.all(np.abs(np.linalg.norm(nrm, axis=1) - 1) < 1e-4)
    from golden.make_config1_fixture import read_test_ply

    crop = ref_golden.load()["scan_crop"]  # the scan's vertices inside a box of whole 12 mm voxels, in file order
    p, n, c = read_test_ply(ref_golden.CROP)
    assert p.shape[0] == crop["n_vertices"] and 0 < p.shape[0] < n_source
    assert orc.grid_downsample(p, 0.005, normals=n, colors=c)[0].shape[0] == crop["n_bins_5mm"]
    p12, n12, _ = orc.grid_downsample(p, 0.012, normals=n)
    rows = crop["fixture_rows"]
    assert len(rows) > 100 and p12.shape[0] == len(rows)
    assert np.array_equal(p12.view(np.uint32), pts[rows].view(np.uint32))
    assert np.array_equal(n12.view(np.uint32), nrm[rows].view(np.uint32))


def test_oracle_runs_the_example_recipe(orc):
    pts, nrm, _, _ = _scan()
    dst_p, dst_n, src_p, src_n, tf_ref = synth.rigid_icp_example_pair(pts, nrm, seed=1)
    assert dst_p.shape[0] < pts.shape[0] and src_p.shape[0] == pts.shape[0]  # dst lost its x <= -0.4 part
    res = orc.icp(dst_p, src_p, orc.make_knn(dst_p), dst_n=dst_n, max_iter=30, tol=1e-4, **SETTINGS)
    assert res["converged"] and res["iterations"] < 30
    # "TRUE transformation" vs "ESTIMATED transformation" of the example: tf_ref^-1, up to the 1 cm point noise
    assert frob(res["T"], synth.invert(tf_ref)) < 2e-2


@pytest.mark.gpu
def test_gpu_matches_oracle_on_the_real_scan(cb, ctx, orc):
    pts, nrm, _, _ = _scan()
    dst_p, dst_n, src_p, src_n, tf_ref = synth.rigid_icp_example_pair(pts, nrm, seed=1)
    knn = orc.make_knn(dst_p)
    d, s = cb.cloud_pair(ctx, dst_p, dst_n, src_p, None)
    icp = cb.Icp(ctx, d, s)
    # the example's own settings: converges, like the oracle, to tf_ref^-1
    res = icp.estimate(max_iter=30, tol=1e-4, **SETTINGS)
    ref = orc.icp(dst_p, src_p, knn, dst_n=dst_n, max_iter=30, tol=1e-4, **SETTINGS)
    assert res["converged"] and abs(res["iterations"] - ref["iterations"]) <= 1
    assert frob(res["T"], synth.invert(tf_ref)) < 2e-2
    # fixed iteration count: transform parity at the 1e-5 bar
    res = icp.estimate(max_iter=12, tol=0.0, **SETTINGS)
    ref = orc.icp(dst_p, src_p, knn, dst_n=dst_n, max_iter=12, tol=0.0, accum_double=True, **SETTINGS)
    assert abs(res["num_corr"] - ref["num_corr"]) <= 3
    assert frob(res["T"], ref["T"]) < (1e-5 if res["num_corr"] == ref["num_corr"] else 1e-4)
    # symmetric metric (source normals too), two Gauss-Newton steps per iteration
    kw = dict(SETTINGS, w_pt=0.1, max_opt_iter=2, opt_tol=0.0)
    d2, s2 = cb.cloud_pair(ctx, dst_p, dst_n, src_p, src_n)
    res2 = cb.Icp(ctx, d2, s2).estimate(max_iter=8, tol=0.0, **kw)
    ref2 = orc.icp(dst_p, src_p, knn, dst_n=dst_n, src_n=src_n, max_iter=8, tol=0.0, accum_double=True, **kw)
    assert frob(res2["T"], ref2["T"]) < (1e-5 if res2["num_corr"] == ref2["num_corr"] else 1e-4)
    # neighbour search and residuals at the estimate: bit-exact on scan data (surfaces, varying density)
    T = ref["T"]
    idx, dd = cb.knn1_radius(ctx, d, s, T, SETTINGS["max_d2"])
    oi, od = orc.BruteKnn(dst_p).query(orc.transform_points(T, src_p), SETTINGS["max_d2"])
    assert np.array_equal(idx, oi) and np.array_equal(dd.view(np.uint32), od.view(np.uint32))
    r = icp.residuals(T, **{k: SETTINGS[k] for k in ("metric", "w_pt", "w_pl")})
    o = orc.icp_residuals(dst_p, src_p, T, knn, metric="combined", dst_n=dst_n, w_pt=0.0, w_pl=1.0)
    assert np.array_equal(r.view(np.uint32), o.view(np.uint32))


@pytest.mark.gpu
def test_gpu_downsample_and_normals_on_the_real_scan(cb, ctx, orc):
    pts, nrm, _, _ = _scan()
    got = cb.grid_downsample(ctx, pts, 0.03, normals=nrm)
    want = orc.grid_downsample(pts, 0.03, normals=nrm)
    assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32))
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    # estimateNormalsKNN(7) as in examples/normal_estimation.cpp, oriented towards the origin (PointCloud default)
    est = cb.Cloud(ctx, pts).estimate_normals(k=7, view_point=[0.0, 0.0, 0.0], want_cov=True)
    knn = orc.make_knn(pts)
    ref = orc.estimate_normals(pts, knn, k=7, view_point=[0.0, 0.0, 0.0])
    d8 = knn.neighborhoods(pts, 8, orc.FLT_MAX)[1]
    tied = (np.diff(d8, axis=1) == 0).any(axis=1)  # the grid-averaged scan has a few exactly tied distances
    assert tied.mean() < 0.01
    assert np.array_equal(est["cov6"][~tied].view(np.uint32), ref[2][~tied].view(np.uint32))
    # and they are the scan's normals (up to the side the scanner chose)
    agree = np.abs(np.sum(est["normals"][~tied] * nrm[~tied], axis=1))
    assert np.median(agree) > 0.95
