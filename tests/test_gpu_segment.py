"""Connected-component segmentation on the device (cb_cloud_segment, segment.cu) against the serial restatement of
extractConnectedComponents (tests/cpp/segment_oracle.cpp) on brute-force neighbourhoods: labels, segment offsets,
segment points and the segment count exactly equal. At full size, against scipy's components over the edges built from
cb_radius_search's lists; on chains, the bounds that guard against one host round trip per graph level."""
import math
import os
import time

import numpy as np
import pytest

import segment_oracle as so
from cilantro_b200 import synth
from golden import make_ref_golden as ref_golden
from golden.make_config1_fixture import read_test_ply

pytestmark = pytest.mark.gpu

DEG2 = float(np.float32(2.0 * math.pi / 180.0))  # (float)(2.0 * M_PI / 180.0), the example's angle


def _same(got, want, what=""):
    assert got[3] == want[3], (what, got[3], want[3])
    assert np.array_equal(got[1], want[1]), what
    assert np.array_equal(got[2], want[2]), what
    assert np.array_equal(got[0], want[0]), what


def _pair(cb, orc, ctx, pts, k=0, radius2=0.0, normals=None, colors=None, cloud_normals=None, **kw):
    """GPU and oracle on the same cloud; normals are passed explicitly, or taken from the cloud (cloud_normals)."""
    cloud = cb.Cloud(ctx, pts, cloud_normals)
    got = cb.segment(ctx, cloud, k=k, radius2=radius2, normals=normals, colors=colors, **kw)
    cloud.close()
    nrm = normals if normals is not None else cloud_normals
    want = so.segment(pts, orc.BruteKnn(pts), k=k, radius2=radius2, normals=nrm, colors=colors, **kw)
    return got, want


# ---- 1. the real scan ------------------------------------------------------------------------------------------------
def _scan():
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config1_cloud.npz"))
    return z["points"], z["normals"]


@pytest.mark.parametrize("variant", ["example", "always_true", "unoriented"])
def test_real_scan_example_recipe(cb, orc, ctx, variant):
    """examples/connected_component_extraction.cpp: radius 0.02^2, NormalsProximityEvaluator(2 deg), min 100, max n."""
    pts, nrm = _scan()
    n = pts.shape[0]
    kw = dict(k=0, radius2=float(np.float32(0.02) * np.float32(0.02)), min_size=100, max_size=n)
    if variant == "example":
        kw.update(evaluator="normals", max_angle=DEG2)
    elif variant == "unoriented":
        kw.update(evaluator="normals", max_angle=-DEG2)
    got, want = _pair(cb, orc, ctx, pts, cloud_normals=nrm, **kw)
    _same(got, want, variant)
    assert got[3] >= 1
    print(f"config1 {variant}: {got[3]} segments, {got[1][-1]} of {n} points labelled")


@pytest.mark.parametrize("evaluator", ["colors", "points_colors", "normals_colors", "points_normals_colors",
                                       "points_normals"])
def test_scan_crop_colour_evaluators(cb, orc, ctx, evaluator):
    p, nrm, col = read_test_ply(ref_golden.CROP)
    kw = dict(k=0, radius2=0.01**2, evaluator=evaluator, max_distance=0.006**2, max_angle=0.2, color_thresh=0.08)
    got, want = _pair(cb, orc, ctx, p, normals=nrm, colors=col, **kw)
    _same(got, want, evaluator)
    assert 1 < got[3] < p.shape[0]


# ---- 2. synthetic clouds ---------------------------------------------------------------------------------------------
def _synthetic(seed, n=6000):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(0, 1, (12, 3))
    lab = rng.integers(0, 12, n)
    pts = (centres[lab] + rng.normal(0, 0.03, (n, 3))).astype(np.float32)
    nrm = rng.normal(0, 1, (12, 3))[lab] + rng.normal(0, 0.05, (n, 3))
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    col = np.clip(rng.uniform(0, 1, (12, 3))[lab] + rng.normal(0, 0.05, (n, 3)), 0, 1).astype(np.float32)
    pts[10:13] = pts[2000]  # duplicates on both sides of the original
    pts[4000] = pts[11]
    pts[[7, 3000]] = np.nan
    pts[3001] = [np.inf, 0, 0]
    return pts, nrm, col


EVALUATORS = list(so.EVALUATORS)
SPECS = {"radius": (0, 0.03**2), "knn": (8, 0.0), "knn_in_radius": (8, 0.03**2)}
THRESH = dict(max_distance=0.02**2, max_angle=0.3, color_thresh=0.15)


@pytest.mark.parametrize("spec", sorted(SPECS))
@pytest.mark.parametrize("evaluator", EVALUATORS)
def test_every_evaluator_and_neighbourhood(cb, orc, ctx, spec, evaluator):
    pts, nrm, col = _synthetic(1)
    k, r2 = SPECS[spec]
    got, want = _pair(cb, orc, ctx, pts, k=k, radius2=r2, normals=nrm, colors=col, evaluator=evaluator, **THRESH)
    _same(got, want, (spec, evaluator))


@pytest.mark.parametrize("spec", sorted(SPECS))
@pytest.mark.parametrize("seeding", ["one_percent", "repeated", "empty", "duplicate_later", "nan"])
def test_seed_lists(cb, orc, ctx, spec, seeding):
    pts, nrm, col = _synthetic(2)
    n = pts.shape[0]
    rng = np.random.default_rng(3)
    seeds = {"one_percent": rng.choice(n, n // 100, replace=False), "repeated": np.r_[rng.choice(n, 30), [11] * 5],
             "empty": np.zeros(0, np.int64), "duplicate_later": [2000, 4000], "nan": [7, 3001, 5]}[seeding]
    k, r2 = SPECS[spec]
    for ev in ("always_true", "points_normals"):
        got, want = _pair(cb, orc, ctx, pts, k=k, radius2=r2, normals=nrm, seeds=seeds, evaluator=ev, **THRESH)
        _same(got, want, (spec, seeding, ev))


def test_seed_of_the_later_duplicate(cb, orc, ctx):
    pts = np.array([[0, 0, 0], [0, 0, 0], [0.5, 0, 0]], np.float32)
    d = cb.Cloud(ctx, pts)
    assert cb.segment(ctx, d, radius2=0.01, seeds=[1])[2].tolist() == [1]
    assert cb.segment(ctx, d, radius2=0.01, seeds=[0])[2].tolist() == [0, 1]
    assert cb.segment(ctx, d, radius2=0.01)[2].tolist() == [0, 1, 2]
    d.close()


@pytest.mark.parametrize("spec", sorted(SPECS))
def test_filters_and_equal_size_ties(cb, orc, ctx, spec):
    rng = np.random.default_rng(5)
    isl = [rng.uniform(0, 100, 3) + rng.normal(0, 0.002, (s, 3)) for s in [3, 1, 5, 2, 6, 4, 9] * 4]
    pts = np.concatenate(isl).astype(np.float32)[rng.permutation(sum(len(i) for i in isl))]
    k, r2 = SPECS[spec]
    for lo, hi in [(1, 2**64 - 1), (2, 5), (4, 4), (10, 20), (0, 0)]:
        got, want = _pair(cb, orc, ctx, pts, k=k, radius2=r2, min_size=lo, max_size=hi)
        _same(got, want, (lo, hi))


def test_parallel_normals_whose_dot_rounds_above_one(cb, orc, ctx):
    """acos(dot > 1) is NaN and the reference calls such a pair not similar; no clamping on either side."""
    rng = np.random.default_rng(9)
    v = None
    while v is None:
        c = rng.normal(0, 1, 3)
        c = (c / np.linalg.norm(c)).astype(np.float32)
        if c[0] * c[0] + (c[1] * c[1] + c[2] * c[2]) > np.float32(1):
            v = c
    pts = (np.arange(40)[:, None] * np.array([[0.001, 0, 0]])).astype(np.float32)
    nrm = np.tile(v, (40, 1))
    got, want = _pair(cb, orc, ctx, pts, k=0, radius2=0.0015**2, normals=nrm, evaluator="normals", max_angle=DEG2)
    _same(got, want)
    assert got[3] == 40  # every pair rejected: 40 singletons


@pytest.mark.parametrize("evaluator,angle", [("normals", DEG2), ("points_normals", DEG2), ("normals", -DEG2),
                                             ("normals", 0.0)])
def test_dots_at_the_interval_ends(cb, orc, ctx, evaluator, angle):
    """Isolated pairs whose float dot products run over consecutive floats around cos(angle) and -cos(angle)."""
    t = abs(angle)
    th = np.concatenate([t * (1 + np.arange(-300, 300) * 2e-7), math.pi - t * (1 + np.arange(-300, 300) * 2e-7)])
    m = th.size
    pts = np.zeros((2 * m, 3), np.float32)
    pts[0::2, 0] = np.arange(m) * 1.0
    pts[1::2, 0] = np.arange(m) * 1.0 + 0.001
    nrm = np.zeros((2 * m, 3), np.float32)
    nrm[0::2, 2] = 1.0
    nrm[1::2, 0] = np.sin(th)
    nrm[1::2, 2] = np.cos(th)
    got, want = _pair(cb, orc, ctx, pts, k=0, radius2=0.01**2, normals=nrm, evaluator=evaluator, max_distance=1.0,
                      max_angle=angle)
    _same(got, want)
    assert m < got[3] < 2 * m  # some pairs joined, some not


def test_tiny_clouds(cb, orc, ctx):
    for n in (0, 1):
        pts = np.zeros((n, 3), np.float32)
        d = cb.Cloud(ctx, pts)
        labels, off, points, m = cb.segment(ctx, d, radius2=1.0)
        assert m == n and points.tolist() == list(range(n)) and labels.tolist() == [0] * n
        d.close()


def test_error_codes(cb, ctx):
    pts, nrm, col = _synthetic(4, n=5000)
    d = cb.Cloud(ctx, pts)
    with pytest.raises(cb.CbError, match="error -1"):
        cb.segment(ctx, d, radius2=0.01, seeds=[0, 5000])
    with pytest.raises(cb.CbError, match="error -5"):
        cb.segment(ctx, d, k=257)
    with pytest.raises(cb.CbError, match="error -1"):
        cb.segment(ctx, d, radius2=0.01, evaluator="normals", max_angle=0.1)  # the cloud has no normals
    with pytest.raises(cb.CbError, match="error -1"):
        cb.segment(ctx, d, radius2=0.01, evaluator="colors", color_thresh=0.1)
    assert cb.segment(ctx, d, radius2=0.01, evaluator="normals", max_angle=0.1, normals=nrm)[3] > 0
    d.close()


# ---- 3. full size ----------------------------------------------------------------------------------------------------
def test_full_size_scene_against_scipy(cb, ctx):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    pts, nrm, r2, objects, faces = synth.segment_scene(2_000_000, seed=2)
    n = pts.shape[0]
    d = cb.Cloud(ctx, pts, nrm)
    off, idx, d2 = cb.radius_search(ctx, d, d, r2)
    u = np.repeat(np.arange(n), np.diff(off))
    cos_t = np.float32(math.cos(DEG2))
    dot = nrm[u, 0] * nrm[idx, 0] + (nrm[u, 1] * nrm[idx, 1] + nrm[u, 2] * nrm[idx, 2])
    for evaluator, mask, count in (("always_true", np.ones(u.size, bool), objects),
                                   ("normals", (dot >= cos_t) & (dot <= 1), faces)):
        labels, soff, spts, m = cb.segment(ctx, d, radius2=r2, evaluator=evaluator, max_angle=DEG2, min_size=100,
                                           max_size=n)
        assert m == count, (evaluator, m, count)
        nc, comp = connected_components(coo_matrix((np.ones(int(mask.sum())), (u[mask], idx[mask])), shape=(n, n)),
                                        directed=False)
        # same partition: the map label -> component is one to one on the labelled points and covers everything
        sizes = np.bincount(comp)
        big = sizes[comp] >= 100
        assert np.array_equal(labels < m, big)
        pairs = np.unique(np.stack([labels[big], comp[big]], 1), axis=0)
        assert pairs.shape[0] == m and np.unique(pairs[:, 0]).size == m and np.unique(pairs[:, 1]).size == m
        assert np.all(np.diff(np.diff(soff)) <= 0)
    d.close()


# ---- 4 / 5. depth ----------------------------------------------------------------------------------------------------
def _chain(n):
    pts = np.zeros((n, 3), np.float32)
    pts[:, 0] = (np.arange(n) * 0.01).astype(np.float32)  # 10 m per 1000 points, spacing 1 cm
    return pts


def test_chain_all_seeds_is_one_segment(cb, ctx):
    d = cb.Cloud(ctx, _chain(1_000_000))
    cb.segment(ctx, d, radius2=0.015**2)  # warm-up (index build, module load)
    t0 = time.perf_counter()
    labels, off, points, m = cb.segment(ctx, d, radius2=0.015**2)
    dt = time.perf_counter() - t0
    assert m == 1 and off[1] == 1_000_000 and not labels.any()
    assert dt < 5.0, dt
    print(f"1M chain, all seeds: {dt * 1e3:.1f} ms")
    d.close()


@pytest.mark.parametrize("spec", ["radius", "knn"])
def test_chain_from_one_end(cb, ctx, spec):
    d = cb.Cloud(ctx, _chain(100_000))
    kw = dict(radius2=0.015**2) if spec == "radius" else dict(k=3)
    cb.segment(ctx, d, seeds=[0], **kw)
    t0 = time.perf_counter()
    labels, off, points, m = cb.segment(ctx, d, seeds=[0], **kw)
    dt = time.perf_counter() - t0
    assert m == 1 and off[1] == 100_000
    assert dt < 10.0, dt
    print(f"100k chain from one end ({spec}): {dt * 1e3:.1f} ms")
    d.close()


# ---- 6. repeat runs --------------------------------------------------------------------------------------------------
def test_repeat_runs_are_bit_identical(cb, ctx):
    pts, nrm, r2, _, _ = synth.segment_scene(300_000, seed=4)
    d = cb.Cloud(ctx, pts, nrm)
    rng = np.random.default_rng(1)
    seeds = rng.choice(pts.shape[0], 3000, replace=False)
    for kw in (dict(radius2=r2, evaluator="normals", max_angle=DEG2), dict(k=8, evaluator="normals", max_angle=DEG2),
               dict(radius2=r2, seeds=seeds, evaluator="normals", max_angle=DEG2)):
        a = cb.segment(ctx, d, **kw)
        b = cb.segment(ctx, d, **kw)
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(x, y)
        assert a[3] == b[3]
    d.close()
