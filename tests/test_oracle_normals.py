"""CPU: the normal-estimation oracle (oracle/cilantro_oracle.cpp: orc_normals_from_neighbors) against known
answers and against the neighbourhoods of the reference's own nanoflann (tests/golden/ref_nanoflann.json).

Reference behaviour under test: core/normal_estimation.hpp:279-332 (normals, view-point flip), :357-421
(curvature), core/covariance.hpp:83-138 (subset mean / covariance, min sample size 3).
"""
import numpy as np

from golden import make_ref_golden as ref_golden


def _plane_cloud(n, normal, seed=0, noise=0.0):
    rng = np.random.default_rng(seed)
    normal = np.asarray(normal, np.float64)
    normal /= np.linalg.norm(normal)
    a = np.cross(normal, [1.0, 0.3, 0.2])
    a /= np.linalg.norm(a)
    b = np.cross(normal, a)
    uv = rng.random((n, 2))
    p = uv[:, :1] * a + uv[:, 1:] * b + noise * rng.standard_normal((n, 1)) * normal + np.array([0.2, -0.1, 0.4])
    return p.astype(np.float32), normal


def test_plane_normals_and_viewpoint(orc):
    pts, nrm = _plane_cloud(4000, [0.3, -0.5, 0.8], seed=1)
    knn = orc.BruteKnn(pts)
    vp = np.array([0.2, -0.1, 0.4], np.float64) + 5.0 * nrm
    n_out, curv, cov6, cnt = orc.estimate_normals(pts, knn, k=12, view_point=vp)
    assert np.all(cnt == 12)
    assert np.all(n_out @ nrm > 0.9999)  # oriented towards the view point
    assert np.all(np.abs(np.linalg.norm(n_out, axis=1) - 1) < 1e-5)
    assert np.all(np.abs(curv) < 1e-4)  # planar: smallest eigenvalue ~ 0
    n_flip, _, _, _ = orc.estimate_normals(pts, knn, k=12, view_point=vp - 10.0 * nrm)
    assert np.all(n_flip @ nrm < -0.9999)
    # no view point: direction correct up to sign
    n_free, _, _, _ = orc.estimate_normals(pts, knn, k=12)
    assert np.all(np.abs(n_free @ nrm) > 0.9999)


def test_covariance_matches_numpy_and_min_sample(orc):
    rng = np.random.default_rng(3)
    pts = rng.random((600, 3), dtype=np.float32)
    knn = orc.BruteKnn(pts)
    k = 9
    idx, d2, cnt = knn.neighborhoods(pts, k, orc.FLT_MAX)
    assert np.all(idx[:, 0] == np.arange(600)) and np.all(d2[:, 0] == 0)  # the point itself comes first
    n_out, curv, cov6, _ = orc.estimate_normals(pts, knn, k=k)
    for i in (0, 17, 599):
        c = np.cov(pts[idx[i]].astype(np.float64).T)
        got = cov6[i]
        full = np.array([[got[0], got[1], got[2]], [got[1], got[3], got[4]], [got[2], got[4], got[5]]])
        assert np.allclose(full, c, rtol=2e-4, atol=1e-7)
        w, v = np.linalg.eigh(c)
        assert abs(abs(v[:, 0] @ n_out[i]) - 1) < 1e-4
        assert abs(curv[i] - w[0] / w.sum()) < 1e-4
    # radius so small that most points have < 3 neighbours -> NaN (covariance.hpp:93-97)
    n_r, curv_r, _, cnt_r = orc.estimate_normals(pts, knn, k=0, radius2=0.03**2)
    few = cnt_r < 3
    assert few.any() and (~few).any()
    assert np.all(np.isnan(n_r[few])) and np.all(np.isnan(curv_r[few]))
    assert not np.isnan(n_r[~few]).any()


def test_reference_nanoflann_neighbourhoods_agree_with_brute(orc):
    g = ref_golden.load()
    rng = np.random.default_rng(5)
    pts = rng.random((5000, 3), dtype=np.float32)
    brute = orc.BruteKnn(pts)
    for (k, r2), want in zip(((8, orc.FLT_MAX), (16, 0.05**2)), g["neighbourhoods_5k"]):
        bi, bd, bc = brute.neighborhoods(pts, k, r2)
        assert ref_golden.sha(bc) == want["cnt"]
        assert ref_golden.sha(bd) == want["d2"]  # bit-equal
        assert ref_golden.sha(bi) == want["idx"]  # random data: no exact distance ties
    bn = orc.estimate_normals(pts, brute, k=10, view_point=[0.5, 0.5, 3.0])
    assert ref_golden.sha(bn[2]) == g["normals_5k"]["cov"]  # covariance bit-equal
    assert ref_golden.sha(bn[0]) == g["normals_5k"]["normals"]
    # radius neighbourhoods: same sets (order of exact ties aside)
    _, _, c0 = brute.neighborhoods(pts, 0, 0.04**2, stride=1)
    assert ref_golden.sha(c0) == g["normals_5k"]["radius_cnt"]
