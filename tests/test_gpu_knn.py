"""GPU parity: grid nearest-neighbour search vs the oracle (bit-exact indices and squared distances).

Calls go through the C ABI (cb_knn1_radius / cb_find_correspondences / cb_knn_radius). Oracle:
orc.BruteKnn (restatement; lowest index wins exact ties — the same rule as the CUDA path) and
the answers of the reference's own nanoflann stored in tests/golden/ref_nanoflann.json (ties may
pick another index with a bit-equal d2).
"""
import numpy as np
import pytest

from cilantro_b200 import synth
from golden import make_ref_golden as ref_golden

pytestmark = pytest.mark.gpu
FMAX = float(np.finfo(np.float32).max)


def _check_exact(cb, ctx, orc, dst, qry, T, max_d2):
    ref = cb.Cloud(ctx, dst)
    q = cb.Cloud(ctx, qry)
    idx, d2 = cb.knn1_radius(ctx, ref, q, T, max_d2)
    qt = orc.transform_points(T if T is not None else orc.identity(), qry)
    oi, od = orc.BruteKnn(dst).query(qt, max_d2)
    assert np.array_equal(idx, oi), f"{(idx != oi).sum()} index mismatches"
    assert np.array_equal(d2.view(np.uint32), od.view(np.uint32)), "squared distances differ bitwise"
    return idx, d2


@pytest.mark.parametrize("n,m,max_d2", [(20000, 20000, 0.02**2), (50000, 7777, 0.05**2), (3000, 9000, FMAX)])
def test_knn1_matches_oracle_bitexact(cb, ctx, orc, n, m, max_d2):
    dst, src, _, T_ref = synth.icp_pair(n, seed=3, noise=0.002, n_src=min(m, n))
    if m > n:
        src = np.random.default_rng(5).random((m, 3), dtype=np.float32)
    T = (T_ref * 0.9 + 0.1 * np.hstack([np.eye(3), np.zeros((3, 1))])).astype(np.float32)
    _check_exact(cb, ctx, orc, dst, src, T, max_d2)


def test_knn1_identity_transform_none(cb, ctx, orc):
    rng = np.random.default_rng(11)
    dst = rng.random((10000, 3), dtype=np.float32)
    qry = rng.random((5000, 3), dtype=np.float32)
    _check_exact(cb, ctx, orc, dst, qry, None, 0.03**2)


def test_knn1_edge_cases(cb, ctx, orc):
    rng = np.random.default_rng(7)
    dst = rng.random((5000, 3), dtype=np.float32)
    # queries far outside the bounding box, on its faces, and NaN-free extremes
    qry = np.vstack([
        rng.random((200, 3), dtype=np.float32) * 4 - 2,
        np.array([[0, 0, 0], [1, 1, 1], [0.5, 0.5, 0.5], [-10, 0.5, 0.5], [0.5, 20, 0.5], [5, 5, -5]], np.float32),
    ]).astype(np.float32)
    for max_d2 in (0.05**2, 1.0, FMAX):
        _check_exact(cb, ctx, orc, dst, qry, None, max_d2)
    # tiny radius: almost nothing qualifies
    idx, d2 = _check_exact(cb, ctx, orc, dst, qry, None, 1e-12)
    assert (idx >= 0).sum() == 0 and np.all(d2 == np.float32(1e-12))


def test_knn1_ties_pick_lowest_index(cb, ctx, orc):
    # duplicated reference points: exact ties everywhere
    rng = np.random.default_rng(2)
    base = rng.random((500, 3), dtype=np.float32)
    dst = np.vstack([base, base, base])[rng.permutation(1500)]
    qry = base + np.float32(1e-3)
    idx, _ = _check_exact(cb, ctx, orc, dst, qry, None, 0.1)
    # the winner is the lowest index among the coincident copies
    for i in range(0, 500, 50):
        same = np.where((dst == dst[idx[i]]).all(axis=1))[0]
        assert idx[i] == same.min()


def test_knn1_degenerate_clouds(cb, ctx, orc):
    rng = np.random.default_rng(4)
    plane = rng.random((4000, 3), dtype=np.float32)
    plane[:, 2] = 0.25  # planar reference set
    line = np.zeros((300, 3), np.float32)
    line[:, 0] = np.linspace(0, 1, 300)
    single = np.array([[0.3, 0.3, 0.3]], np.float32)
    coincident = np.repeat(single, 100, axis=0)
    qry = rng.random((1000, 3), dtype=np.float32)
    for dst in (plane, line, single, coincident):
        _check_exact(cb, ctx, orc, dst, qry, None, FMAX)
        _check_exact(cb, ctx, orc, dst, qry, None, 0.1**2)


def test_knn1_empty_inputs(cb, ctx):
    empty = cb.Cloud(ctx, np.zeros((0, 3), np.float32))
    pts = cb.Cloud(ctx, np.random.default_rng(0).random((100, 3), dtype=np.float32))
    idx, d2 = cb.knn1_radius(ctx, empty, pts, None, 1.0)
    assert np.all(idx == -1) and np.all(d2 == 1.0)
    idx, d2 = cb.knn1_radius(ctx, pts, empty, None, 1.0)
    assert idx.shape == (0,)
    i1, i2, v = cb.find_correspondences(ctx, empty, pts, None, 1.0)
    assert i1.size == 0


def test_find_correspondences_matches_oracle(cb, ctx, orc):
    dst, src, _, T_ref = synth.icp_pair(30000, seed=9, noise=0.004)
    T = T_ref.astype(np.float32)
    max_d2 = np.float32(0.004**2)  # many queries have no neighbour inside the radius
    ref, q = cb.Cloud(ctx, dst), cb.Cloud(ctx, src)
    i1, i2, v = cb.find_correspondences(ctx, ref, q, T, max_d2)
    o1, o2, ov = orc.find_correspondences(T, src, orc.BruteKnn(dst), max_d2)
    assert 0 < i1.size < src.shape[0]
    assert np.array_equal(i1, o1) and np.array_equal(i2, o2)
    assert np.array_equal(v.view(np.uint32), ov.view(np.uint32))
    assert np.all(np.diff(i2) > 0), "correspondences must be compacted in query order"


def test_knn1_vs_reference_nanoflann_250k(cb, ctx):
    """Against the reference's own kd-tree: equal index, or an exact tie (bit-equal d2)."""
    want = ref_golden.load()["knn1_250k"]
    dst, src, _, T_ref = synth.icp_pair(250000, seed=1, noise=0.001)
    T = T_ref.astype(np.float32)
    max_d2 = np.float32(0.02**2)
    idx, d2 = cb.knn1_radius(ctx, cb.Cloud(ctx, dst), cb.Cloud(ctx, src), T, max_d2)
    assert ref_golden.sha(d2) == want["d2"]
    # the reference's list with its exact ties resolved to the lowest index (the CUDA path's rule), and few such ties
    assert ref_golden.sha(idx) == want["idx"]
    assert want["ties"] <= 5, f"{want['ties']} index differences (only exact ties may differ)"


def test_knn_k_matches_numpy(cb, ctx):
    rng = np.random.default_rng(13)
    dst = rng.random((4000, 3), dtype=np.float32)
    qry = rng.random((300, 3), dtype=np.float32)
    ref, q = cb.Cloud(ctx, dst), cb.Cloud(ctx, qry)
    for k, r2 in ((2, FMAX), (8, 0.08**2), (20, FMAX), (50, FMAX), (100, 0.3**2), (200, FMAX), (256, FMAX)):
        idx, d2, cnt = cb.knn_radius(ctx, ref, q, k, None, r2)
        # numpy restatement with the same fp32 arithmetic order
        dx = qry[:, None, 0] - dst[None, :, 0]
        dy = qry[:, None, 1] - dst[None, :, 1]
        dz = qry[:, None, 2] - dst[None, :, 2]
        D = (dx * dx + dy * dy) + dz * dz
        order = np.lexsort((np.broadcast_to(np.arange(dst.shape[0]), D.shape), D), axis=1)[:, :k]
        for i in range(qry.shape[0]):
            ok = D[i, order[i]] < r2
            want = order[i][ok]
            assert cnt[i] == want.size
            assert np.array_equal(idx[i, : want.size], want)
            assert np.array_equal(d2[i, : want.size], D[i, want])
            assert np.all(idx[i, want.size:] == -1)


def test_kd_tree_example_known_answer(cb, ctx):
    """examples/kd_tree.cpp:6-19: unit-cube corners, query (0.1,0.1,0.4), k=2, r2=1.001 -> 0,3 / 0.18,0.38."""
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 1, 1], [1, 0, 1], [1, 1, 0], [1, 1, 1]], np.float32)
    ref = cb.Cloud(ctx, pts)
    q = cb.Cloud(ctx, np.array([[0.1, 0.1, 0.4]], np.float32))
    idx, d2, cnt = cb.knn_radius(ctx, ref, q, 2, None, 1.001)
    assert cnt[0] == 2 and list(idx[0]) == [0, 3]
    assert np.allclose(d2[0], [0.18, 0.38], rtol=1e-6)


def _check_radius(cb, ctx, orc, dst, qry, r2, T=None):
    off, idx, d2 = cb.radius_search(ctx, cb.Cloud(ctx, dst), cb.Cloud(ctx, qry), r2, T=T)
    qt = orc.transform_points(T, qry) if T is not None else qry
    _, _, cnt = orc.BruteKnn(dst).neighborhoods(qt, 0, r2, stride=1)
    oi, od, cnt = orc.BruteKnn(dst).neighborhoods(qt, 0, r2, stride=max(1, int(cnt.max())))
    assert np.array_equal(np.diff(off), cnt.astype(np.int64))
    for i in range(qry.shape[0]):  # ragged rows: compare the used prefix of the padded oracle rows
        m = cnt[i]
        assert np.array_equal(idx[off[i]:off[i + 1]], oi[i, :m])
        assert np.array_equal(d2[off[i]:off[i + 1]].view(np.uint32), od[i, :m].view(np.uint32))
    return off, idx, d2


def test_radius_search_matches_oracle_bitexact(cb, ctx, orc):
    rng = np.random.default_rng(17)
    dst = rng.random((20000, 3), dtype=np.float32)
    qry = np.vstack([rng.random((1500, 3), dtype=np.float32), rng.random((50, 3), dtype=np.float32) * 3 - 1]).astype(np.float32)
    off, idx, d2 = _check_radius(cb, ctx, orc, dst, qry, 0.06**2)
    assert off[-1] > 10 * qry.shape[0] and (np.diff(off) == 0).any()  # long lists and empty ones
    T = synth.rigid_from_axis_angle([0.2, 1, -0.4], 0.3, [0.05, -0.02, 0.01]).astype(np.float32)
    _check_radius(cb, ctx, orc, dst, qry[:400], 0.04**2, T=T)
    # duplicated reference points: equal distances come out in ascending index
    dup = np.vstack([dst[:3000], dst[:3000]]).astype(np.float32)
    _check_radius(cb, ctx, orc, dup, qry[:300], 0.08**2)
    # radius 0 / empty clouds
    off, idx, d2 = cb.radius_search(ctx, cb.Cloud(ctx, dst), cb.Cloud(ctx, qry[:10]), 0.0)
    assert off[-1] == 0 and idx.size == 0
    off, idx, d2 = cb.radius_search(ctx, cb.Cloud(ctx, dst[:0]), cb.Cloud(ctx, qry[:10]), 1.0)
    assert off[-1] == 0


def test_radius_search_agrees_with_reference_nanoflann(cb, ctx):
    want = ref_golden.load()["radius_15k"]
    rng = np.random.default_rng(23)
    dst = rng.random((15000, 3), dtype=np.float32)
    qry = rng.random((800, 3), dtype=np.float32)
    r2 = 0.05**2
    off, idx, d2 = cb.radius_search(ctx, cb.Cloud(ctx, dst), cb.Cloud(ctx, qry), r2)
    assert ref_golden.sha(np.diff(off).astype(np.int64)) == want["cnt"]
    # the rows one after the other; random data: no equal distances, so the order is unique
    assert ref_golden.sha(idx.astype(np.int64)) == want["idx"]
    assert ref_golden.sha(d2.astype(np.float32)) == want["d2"]


def _hollow_sphere(n, seed=0, radius=0.45, noise=0.002):
    rng = np.random.default_rng(seed)
    g = rng.standard_normal((n, 3))
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    r = radius + noise * rng.standard_normal((n, 1))
    return (0.5 + g * r).astype(np.float32)


def test_far_queries_cross_empty_space_exactly_and_fast(cb, ctx, orc):
    # The far-query path (far_sweep.cuh): queries at the centre of a hollow scan and far outside it would cost
    # O(shells^3) row tests with the shell sweep alone; they must stay exact and finish quickly.
    import time

    dst = _hollow_sphere(1_000_000, seed=3)
    rng = np.random.default_rng(4)
    qry = np.vstack([
        0.5 + 0.05 * rng.standard_normal((3000, 3)),          # deep inside the hollow
        0.5 + 40.0 * rng.standard_normal((1000, 3)),          # far outside the bounding box
        rng.random((1000, 3)),                                # anywhere in the box
        dst[:500] + np.float32(1e-4),                         # on the surface
    ]).astype(np.float32)
    ref, q = cb.Cloud(ctx, dst), cb.Cloud(ctx, qry)
    cb.knn1_radius(ctx, ref, q, None, FMAX)  # builds the indices
    t0 = time.perf_counter()
    idx, d2 = cb.knn1_radius(ctx, ref, q, None, FMAX)
    dt = time.perf_counter() - t0
    oi, od = orc.BruteKnn(dst).query(qry, FMAX)
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2.view(np.uint32), od.view(np.uint32))
    assert dt < 5.0, f"unbounded 1-NN of {qry.shape[0]} far queries took {dt:.1f} s"
    # k nearest of far queries (k-best sweep restarts on the block list too)
    sub = qry[::10]
    t0 = time.perf_counter()
    kidx, kd2, cnt = cb.knn_radius(ctx, ref, cb.Cloud(ctx, sub), 10, None, FMAX)
    dt = time.perf_counter() - t0
    bi, bd, bc = orc.BruteKnn(dst).neighborhoods(sub, 10, FMAX)
    assert np.array_equal(cnt, bc) and np.array_equal(kidx, bi)
    assert np.array_equal(kd2.view(np.uint32), bd.view(np.uint32))
    assert dt < 5.0, f"unbounded 10-NN of {sub.shape[0]} far queries took {dt:.1f} s"
    # bounded searches of the same queries still report "nothing within the radius"
    idx_b, d2_b = cb.knn1_radius(ctx, ref, q, None, 0.01**2)
    oi_b, od_b = orc.BruteKnn(dst).query(qry, np.float32(0.01**2))
    assert np.array_equal(idx_b, oi_b) and np.array_equal(d2_b.view(np.uint32), od_b.view(np.uint32))


def test_normals_with_isolated_outliers(cb, ctx, orc):
    # scanner outliers far from the surface ask for k neighbours across empty space
    want = ref_golden.load()["normals_outliers_300k"]
    pts, _ = synth.surface_cloud(300_000, seed=8, noise=0.0005)
    rng = np.random.default_rng(9)
    outliers = (np.array([0.5, 0.5, 0.5]) + 3.0 * rng.standard_normal((25, 3))).astype(np.float32)
    cloud = np.vstack([pts, outliers]).astype(np.float32)
    got = cb.Cloud(ctx, cloud).estimate_normals(k=10, view_point=[0.5, 0.5, 10.0], want_cov=True)
    # Neighbourhoods: the reference's nanoflann for the surface points; brute force (ascending (d2, index), the
    # CUDA path's rule) for the outliers, whose ~10 nearest surface points are several units away and so tie in
    # fp32 d2 — the one case where the reference's order is its kd-tree traversal order (DESIGN.md §4.7). The oracle's
    # covariances of those neighbourhoods are stored (tests/golden/make_ref_golden.py: outlier_normals_entry).
    _, bd, _ = orc.BruteKnn(cloud).neighborhoods(outliers, 10, orc.FLT_MAX)
    assert ref_golden.sha(bd) == want["outlier_d2"]  # the reference's distances, sorted, are the same
    # at 300 k points a couple of surface rows hold two neighbours with bit-equal d2 as well (probability
    # ~ ulp / spacing per pair): bit-exact wherever the distances are distinct, fp32 rounding elsewhere
    # (k + 1 distances: a tie between the 10th and the excluded 11th neighbour changes the SET, not just the order)
    tied = np.zeros(cloud.shape[0], bool)
    tied[want["tied"]] = True
    assert tied.sum() < 20
    assert ref_golden.sha(got["cov6"][~tied]) == want["cov"]
    assert np.isfinite(got["cov6"][tied]).all()  # a legitimate alternative neighbourhood: nothing more to compare


def test_nan_and_inf_points_are_inert(cb, ctx, orc):
    # NaN / Inf coordinates (organised depth clouds carry them): such a query finds nothing, such a reference
    # point is never found, and nothing hangs — in every search flavour and in normal estimation.
    rng = np.random.default_rng(31)
    dst = rng.random((20000, 3), dtype=np.float32)
    dst[[5, 77, 1234]] = np.nan
    dst[[9, 500]] = np.inf
    qry = rng.random((3000, 3), dtype=np.float32)
    qry[[0, 10]] = np.nan
    qry[[1, 11], 1] = np.inf
    qry[2, 2] = -np.inf
    ref, q = cb.Cloud(ctx, dst), cb.Cloud(ctx, qry)
    brute = orc.BruteKnn(dst)
    for max_d2 in (np.float32(0.05**2), FMAX):
        idx, d2 = cb.knn1_radius(ctx, ref, q, None, max_d2)
        oi, od = brute.query(qry, max_d2)
        assert np.array_equal(idx, oi) and np.array_equal(d2.view(np.uint32), od.view(np.uint32))
        assert np.all(idx[[0, 1, 2, 10, 11]] == -1)
        kidx, kd2, cnt = cb.knn_radius(ctx, ref, q, 6, None, max_d2)
        bi, bd, bc = brute.neighborhoods(qry, 6, max_d2)
        assert np.array_equal(cnt, bc) and np.array_equal(kidx, bi) and np.array_equal(kd2.view(np.uint32), bd.view(np.uint32))
    off, ridx, rd2 = cb.radius_search(ctx, ref, q, 0.04**2)
    _, _, bc = brute.neighborhoods(qry, 0, np.float32(0.04**2), stride=1)
    assert np.array_equal(np.diff(off), bc.astype(np.int64)) and bc[[0, 1, 2, 10, 11]].sum() == 0
    bad = np.array([5, 9, 77, 500, 1234])
    assert not np.isin(idx, bad).any() and not np.isin(ridx, bad).any()
    # normals of the cloud with its own bad points as queries: NaN rows there, exact elsewhere
    got = ref.estimate_normals(k=8, view_point=[0.5, 0.5, 5.0], want_cov=True)
    want = orc.estimate_normals(dst, brute, k=8, view_point=[0.5, 0.5, 5.0])
    assert np.isnan(got["normals"][bad]).all() and np.isnan(got["curvature"][bad]).all()
    good = np.setdiff1d(np.arange(dst.shape[0]), bad)
    assert np.array_equal(got["cov6"][good].view(np.uint32), want[2][good].view(np.uint32))
