"""The segmentation oracle (tests/cpp/segment_oracle.cpp, the serial reference loop) against an independent
formulation, without a GPU: R = the points reachable from the seeds along the directed edges u -> L(u)[j], j >= 1, that
the evaluator accepts (scipy breadth_first_order from a virtual source joined to every seed); segments = the connected
components (scipy connected_components) of the undirected graph on R with those edges. This is the statement the
device implementation (segment.cu) is built on."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import breadth_first_order, connected_components

import segment_oracle as so

SPECS = [(0, 0.05**2), (8, 0.0), (8, 0.05**2)]  # radius, kNN, kNN in radius


def _cloud(seed, n=900):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(0, 1, (6, 3))
    pts = (centres[rng.integers(0, 6, n)] + rng.normal(0, 0.04, (n, 3))).astype(np.float32)
    pts[10:13] = pts[200]  # triple duplicates (one after the original index, two before)
    pts[500] = pts[11]
    pts[[7, 300]] = np.nan
    pts[301] = [np.inf, 0, 0]
    colors = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    return pts, colors


def _closure(n, lists, accept, seeds, min_size, max_size):
    off, idx, d2 = lists
    src = np.repeat(np.arange(n), np.diff(off).astype(np.int64))
    first = np.zeros(idx.shape[0], bool)
    first[off[:-1][np.diff(off) > 0].astype(np.int64)] = True
    keep = ~first & accept(src, idx, d2)
    u, v = src[keep], idx[keep]
    seeds = np.arange(n) if seeds is None else np.asarray(seeds, np.int64)
    # reachability from a virtual source n joined to every seed
    g = coo_matrix((np.ones(u.size + seeds.size), (np.r_[u, np.full(seeds.size, n)], np.r_[v, seeds])),
                   shape=(n + 1, n + 1)).tocsr()
    reach = breadth_first_order(g, n, directed=True, return_predecessors=False)
    in_r = np.zeros(n + 1, bool)
    in_r[reach] = True
    in_r = in_r[:n]
    e = in_r[u]
    ncomp, comp = connected_components(coo_matrix((np.ones(int(e.sum())), (u[e], v[e])), shape=(n, n)), directed=False)
    segs = {}
    for i in np.flatnonzero(in_r):
        segs.setdefault(comp[i], []).append(i)
    segs = [s for s in segs.values() if min_size <= len(s) <= max_size]
    segs.sort(key=lambda s: (-len(s), s[0]))
    labels = np.full(n, len(segs), np.int64)
    for r, s in enumerate(segs):
        labels[s] = r
    offsets = np.r_[0, np.cumsum([len(s) for s in segs])].astype(np.int64)
    points = np.array([i for s in segs for i in s], np.int64)
    return labels, offsets, points, len(segs)


def _check(got, want):
    assert got[3] == want[3]
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2])


EVALS = {
    "always_true": (dict(), lambda c: lambda u, v, d2: np.ones(u.size, bool)),
    "points": (dict(max_distance=0.03**2), lambda c: lambda u, v, d2: d2 < np.float32(0.03**2)),
    "colors": (dict(color_thresh=0.6),
               lambda c: lambda u, v, d2: _color_d2(c, u, v) < np.float32(np.float32(0.6) * np.float32(0.6))),
}


def _color_d2(c, u, v):
    d = c[u] - c[v]
    return d[:, 0] * d[:, 0] + (d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])


@pytest.mark.parametrize("spec", SPECS, ids=["radius", "knn", "knn_in_radius"])
@pytest.mark.parametrize("ev", sorted(EVALS))
@pytest.mark.parametrize("seeding", ["all", "one_percent", "repeated", "empty"])
def test_oracle_equals_reachable_closure(orc, spec, ev, seeding):
    pts, colors = _cloud(3)
    n = pts.shape[0]
    knn = orc.BruteKnn(pts)
    lists = so.neighbour_lists(pts, spec[0], spec[1], knn)
    rng = np.random.default_rng(11)
    seeds = {"all": None, "one_percent": rng.choice(n, n // 100, replace=False),
             "repeated": np.r_[rng.choice(n, 20), [11, 11, 200, 7]], "empty": np.zeros(0, np.int64)}[seeding]
    kw, accept = EVALS[ev]
    got = so.connected_components(n, lists, evaluator=ev, seeds=seeds, colors=colors, **kw)
    _check(got, _closure(n, lists, accept(colors), seeds, 1, 2**64 - 1))


@pytest.mark.parametrize("spec", SPECS, ids=["radius", "knn", "knn_in_radius"])
def test_oracle_filters_and_equal_size_ties(orc, spec):
    # islands of 1..6 points, three of each size, far apart: equal sizes are ordered by their smallest index
    rng = np.random.default_rng(5)
    isl = []
    for size in [3, 1, 5, 2, 6, 4] * 3:
        c = rng.uniform(0, 100, 3)
        isl.append(c + rng.normal(0, 0.005, (size, 3)))
    pts = np.concatenate(isl).astype(np.float32)
    perm = rng.permutation(pts.shape[0])
    pts = pts[perm]
    knn = orc.BruteKnn(pts)
    lists = so.neighbour_lists(pts, spec[0], spec[1], knn)
    for lo, hi in [(1, 2**64 - 1), (2, 5), (4, 4), (7, 10)]:
        got = so.connected_components(pts.shape[0], lists, min_size=lo, max_size=hi)
        want = _closure(pts.shape[0], lists, EVALS["always_true"][1](None), None, lo, hi)
        _check(got, want)


def test_oracle_seed_of_the_later_duplicate_reaches_nothing(orc):
    """Exact duplicates w < u: L(u) = [w, u, ...] and the reference skips entry 0, so seeding u alone gives {u} and
    seeding w gives {w, u}."""
    pts = np.array([[0, 0, 0], [0, 0, 0]], np.float32)
    lists = so.neighbour_lists(pts, 0, 1.0, orc.BruteKnn(pts))
    assert so.connected_components(2, lists, seeds=[1])[2].tolist() == [1]
    assert so.connected_components(2, lists, seeds=[0])[2].tolist() == [0, 1]
    assert so.connected_components(2, lists)[2].tolist() == [0, 1]


def test_oracle_empty_neighbourhoods_and_nan_seeds(orc):
    pts, _ = _cloud(4, n=600)
    lists = so.neighbour_lists(pts, 0, 0.0, orc.BruteKnn(pts))
    labels, off, points, m = so.connected_components(600, lists, seeds=[7, 3, 3, 599])
    assert m == 3 and points.tolist() == [3, 7, 599] and off.tolist() == [0, 1, 2, 3]
    lists = so.neighbour_lists(pts, 0, 0.05**2, orc.BruteKnn(pts))
    labels, off, points, m = so.connected_components(600, lists, seeds=[7])
    assert m == 1 and points.tolist() == [7]  # a NaN point has an empty list
