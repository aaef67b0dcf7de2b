"""Pin the oracle (CPU, no GPU): known answers derivable from the reference's examples, agreement of
the brute-force restatement with the reference's own nanoflann (its answers stored in tests/golden/ref_nanoflann.json
by tests/golden/make_ref_golden.py), and self-checks of the restated estimators. The reference ships no tests or
golden vectors (SURVEY.md F2); these plus the committed fixtures in tests/golden/ are what anchors parity.
"""
import json
import os

import numpy as np

from cilantro_b200 import synth
from conftest import frob
from golden import make_ref_golden as ref_golden

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_kd_tree_example(orc):
    """examples/kd_tree.cpp:6-19 -> neighbours 0, 3 with d2 0.18, 0.38."""
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 1, 1], [1, 0, 1], [1, 1, 0], [1, 1, 1]], np.float32)
    i, d = orc.BruteKnn(pts).query(np.array([[0.1, 0.1, 0.4]], np.float32), 1.001)
    assert i[0] == 0 and abs(d[0] - 0.18) < 1e-6
    g = ref_golden.load()
    assert g["nanoflann_version"] == 0x171
    want = g["kd_tree_example"]  # the reference's nanoflann, kNNInRadius k = 2
    assert want["idx"] == [0, 3] and np.allclose(want["d2"], [0.18, 0.38], rtol=1e-6)
    idx, d2, cnt = orc.BruteKnn(pts).neighborhoods(np.array([[0.1, 0.1, 0.4]], np.float32), 2, 1.001)
    assert cnt[0] == 2 and list(idx[0]) == want["idx"] and np.array_equal(d2[0], np.float32(want["d2"]))


def test_pca_example(orc):
    """examples/principal_component_analysis.cpp:6-16."""
    box = np.array([[x, y, z] for x in (0, 1) for y in (0, 100) for z in (0, 1000)], np.float32)
    r = orc.pca(box)
    assert np.allclose(r["mean"], [0.5, 50, 500])
    assert np.allclose(r["eigenvalues"], [8 * 250000 / 7, 8 * 2500 / 7, 8 * 0.25 / 7], rtol=1e-6)
    assert np.allclose(np.abs(r["eigenvectors"]), [[0, 0, 1], [0, 1, 0], [1, 0, 0]], atol=1e-6)
    assert np.linalg.det(r["eigenvectors"].astype(np.float64)) > 0


def test_brute_restatement_agrees_with_reference_nanoflann(orc):
    g = ref_golden.load()
    dst, src, _, T_ref = synth.icp_pair(60000, seed=4, noise=0.003, n_src=20000)
    q = orc.transform_points(T_ref.astype(np.float32), src)
    for r2, want in zip((np.float32(0.004**2), np.float32(0.05**2), np.float32(np.finfo(np.float32).max)), g["knn1_60k"]):
        bi, bd = orc.BruteKnn(dst).query(q, r2)
        assert ref_golden.sha(bd) == want["d2"]  # bit-equal squared distances
        # equal indices once the reference's exact ties are resolved to the lowest index, and only a few such ties
        assert ref_golden.sha(bi) == want["idx"] and want["ties"] <= 2
    # unbounded nearestNeighborSearch path
    bi, bd = orc.BruteKnn(dst).query(q, np.float32(np.finfo(np.float32).max))
    assert ref_golden.sha(bd) == g["nn1_60k_d2"]


def test_kabsch_recovers_known_transform(orc):
    rng = np.random.default_rng(0)
    src = rng.random((5000, 3), dtype=np.float32)
    T = synth.rigid_from_axis_angle([0.2, -0.5, 0.8], 0.4, [0.3, -0.1, 0.7])
    dst = synth.apply(T, src)
    for dbl in (False, True):
        Te, ok = orc.kabsch(dst, src, accum_double=dbl)
        assert ok and frob(Te, T) < 5e-6
    # reflection handling: a mirrored cloud must still give det = +1
    Te, _ = orc.kabsch(dst * np.float32([1, 1, -1]), src)
    assert np.linalg.det(Te[:, :3].astype(np.float64)) > 0.999
    # degenerate sizes (transform_estimation.hpp:20-23,47)
    Te, ok = orc.kabsch(dst[:0], src[:0])
    assert not ok and frob(Te, orc.identity()) == 0
    Te, ok = orc.kabsch(dst[:2], src[:2])
    assert not ok


def test_rotation_projection(orc):
    R = synth.rigid_from_axis_angle([1, 2, 3], 0.3, [0, 0, 0])[:, :3]
    noisy = (R + 1e-3 * np.random.default_rng(1).normal(size=(3, 3))).astype(np.float32)
    P = orc.rotation(noisy).astype(np.float64)
    assert np.allclose(P @ P.T, np.eye(3), atol=1e-6) and np.linalg.det(P) > 0
    assert np.abs(P - R).max() < 3e-3


def test_rigid_icp_example_recipe_self_check(orc):
    """examples/rigid_icp.cpp:25-65,116-133: src = noisy copy of dst moved by tf_ref (Z*Y*X angle-axis
    -0.1/0.1/-0.1 rad, t = (-0.20,-0.05,0.10)); point-to-plane ICP, max_distance 0.1^2, tol 1e-4,
    30 iterations max; the estimate must come out close to tf_ref^-1."""
    rng = np.random.default_rng(5)
    # a smooth surface with analytic normals stands in for the downsampled PLY scan
    u = rng.random((6000, 2)) * 2 - 1
    z = 0.3 * np.sin(2 * u[:, 0]) * np.cos(1.5 * u[:, 1])
    dst = np.column_stack([u, z]).astype(np.float32)
    gx = 0.6 * np.cos(2 * u[:, 0]) * np.cos(1.5 * u[:, 1])
    gy = -0.45 * np.sin(2 * u[:, 0]) * np.sin(1.5 * u[:, 1])
    nrm = np.column_stack([-gx, -gy, np.ones_like(gx)])
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    Rz = synth.rigid_from_axis_angle([0, 0, 1], -0.1, [0, 0, 0])[:, :3]
    Ry = synth.rigid_from_axis_angle([0, 1, 0], 0.1, [0, 0, 0])[:, :3]
    Rx = synth.rigid_from_axis_angle([1, 0, 0], -0.1, [0, 0, 0])[:, :3]
    tf_ref = np.zeros((3, 4))
    tf_ref[:, :3] = Rz @ Ry @ Rx
    tf_ref[:, 3] = [-0.20, -0.05, 0.10]
    src = synth.apply(tf_ref, dst + 0.01 * (rng.random(dst.shape) * 2 - 1).astype(np.float32))
    res = orc.icp(dst, src, orc.make_knn(dst), metric="combined", dst_n=nrm, max_iter=30, tol=1e-4,
                  max_d2=np.float32(0.1 * 0.1), w_pt=0.0, w_pl=1.0)
    assert res["converged"] and res["iterations"] < 30
    assert frob(res["T"], synth.invert(tf_ref)) < 2e-2


def test_kmeans_oracle_basics(orc):
    rng = np.random.default_rng(3)
    blobs = np.vstack([rng.normal(c, 0.01, (500, 3)) for c in ((0, 0, 0), (1, 0, 0), (0, 1, 0))]).astype(np.float32)
    cent, labels, it = orc.kmeans(blobs, blobs[[0, 500, 1000]], max_iter=50)
    assert it < 10
    assert np.array_equal(labels, np.repeat([0, 1, 2], 500))
    assert np.abs(cent - [[0, 0, 0], [1, 0, 0], [0, 1, 0]]).max() < 5e-3
    idx = orc.kmeans_seed_indices(1000, 50, 7)
    assert len(set(idx.tolist())) == 50 and idx.max() < 1000


def test_ransac_oracle_basics(orc):
    dst, src, T_ref, inl = synth.ransac_pairs(4000, 0.3, seed=1)
    r = orc.ransac_rigid(dst, src, seed=3, max_iter=300, thresh=0.01, inlier_count_thresh=1000)
    assert r["iterations"] < 300 and frob(r["T"], T_ref) < 2e-3
    assert abs(r["num_inliers"] - inl.sum()) < 0.05 * inl.sum()
    T_h = orc.ransac_fit_samples(dst, src, orc.ransac_samples(4000, 3, 20, 11))
    c = orc.ransac_score(dst, src, T_h, 0.01)
    # count restated in numpy
    for h in range(3):
        q = orc.transform_points(T_h[h], src)
        e = q - dst
        res = np.sqrt(e[:, 0] * e[:, 0] + (e[:, 1] * e[:, 1] + e[:, 2] * e[:, 2]))
        assert c[h] == int((res <= np.float32(0.01)).sum())


def test_golden_fixtures(orc):
    """tests/golden/oracle_golden.json was produced by tests/golden/make_golden.py in the build
    container, where oracle/_ref (the reference's nanoflann) exists: it pins the oracle's outputs so
    that a later edit of the restatement cannot silently move the parity target."""
    path = os.path.join(GOLDEN, "oracle_golden.json")
    with open(path) as f:
        g = json.load(f)
    from golden.make_golden import compute

    now = compute(orc)
    assert now["knn_idx_sha"] == g["knn_idx_sha"]
    assert now["knn_d2_sha"] == g["knn_d2_sha"]
    assert now["kmeans_labels_sha"] == g["kmeans_labels_sha"]
    assert now["ransac_counts"] == g["ransac_counts"]
    for key in ("icp_p2p_T", "icp_combined_T", "pca_eigenvalues"):
        assert np.allclose(now[key], g[key], rtol=0, atol=2e-6), key
    # §8(f) rows: neighbourhood lists / covariances / downsampled clouds / engine lists are integer or
    # bit-exact fp32 work — the brute-force restatement must reproduce the hashes made with the reference nanoflann
    for key in ("nbr_idx_sha", "nbr_d2_sha", "nbr_cnt_sha", "normals_cov_sha", "radius_cnt_sha", "radius_d2_sha",
                "downsample_order0_sha", "downsample_order1_sha", "engine_both_recip_frac_sha", "engine_f2s_1to1_sha"):
        assert now[key] == g[key], key
    for key in ("normals_first", "curvature_first"):
        assert np.allclose(now[key], g[key], rtol=0, atol=2e-6), key
