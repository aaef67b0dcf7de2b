"""CPU: the correspondence-engine oracle (engine_correspondences in oracle/cilantro_oracle.cpp) on a case small
enough to derive by hand.

Reference behaviour: correspondence_search/correspondence_search_kd_tree.hpp:195-229 (directions, filters),
correspondence_search_kd_tree_utilities.hpp:64-99 (set_union / set_intersection on (first, second)),
core/correspondence.hpp:57-100 (fraction: sort by value, keep llround(f * size); one-to-one: per index the pair of
smallest value).
"""
import numpy as np

DST = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0]], np.float32)
SRC = np.array([[0.1, 0, 0], [0.2, 0, 0], [1.1, 0, 0], [5, 0, 0]], np.float32)
# by hand (squared distances, max 1.0):
#   second -> first: src0 -> dst0 (.01), src1 -> dst0 (.04), src2 -> dst1 (.01), src3 -> nothing (9 >= 1)
#   first -> second: dst0 -> src0 (.01), dst1 -> src2 (.01), dst2 -> src2 (.81)
S2F = [(0, 0), (0, 1), (1, 2)]
F2S = [(0, 0), (1, 2), (2, 2)]


def _pairs(orc, **mode):
    f, s, v = orc.engine_correspondences(DST, SRC, orc.identity(), orc.BruteKnn(DST), np.float32(1.0), **mode)
    return list(zip(f.tolist(), s.tolist())), v


def test_directions_union_and_intersection(orc):
    p, v = _pairs(orc)
    assert p == S2F and np.allclose(v, [0.01, 0.04, 0.01], atol=1e-6)
    p, v = _pairs(orc, search_dir="first_to_second")
    assert p == F2S and np.allclose(v, [0.01, 0.01, 0.81], atol=1e-6)
    p, _ = _pairs(orc, search_dir="both")
    assert p == [(0, 0), (0, 1), (1, 2), (2, 2)]  # set_union, lexicographic
    p, _ = _pairs(orc, search_dir="both", require_reciprocal=True)
    assert p == [(0, 0), (1, 2)]  # set_intersection


def test_fraction_and_one_to_one(orc):
    # 3 pairs, f = 0.5 -> llround(1.5) = 2 closest: src0 and src2 (fp32: 0.1^2 < (1.1 - 1)^2), ascending value
    p, v = _pairs(orc, inlier_fraction=0.5)
    assert p == [(0, 0), (1, 2)] and v[0] < v[1]
    p, _ = _pairs(orc, inlier_fraction=0.34)  # llround(1.02) = 1
    assert p == [(0, 0)]
    for f in (0.0, 1.0, 2.0):  # outside (0, 1): the filter is off
        assert _pairs(orc, inlier_fraction=f)[0] == S2F
    # one-to-one keeps, per dst point, the closest src: dst0 <- src0 (not src1)
    assert _pairs(orc, one_to_one=True)[0] == [(0, 0), (1, 2)]
    # first -> second: per src point the closest dst: src2 <- dst1 (.01), not dst2 (.81)
    assert _pairs(orc, search_dir="first_to_second", one_to_one=True)[0] == [(0, 0), (1, 2)]
    # the one-to-one filter does nothing for BOTH (core/correspondence.hpp:97-99)
    assert _pairs(orc, search_dir="both", one_to_one=True)[0] == [(0, 0), (0, 1), (1, 2), (2, 2)]
    # fraction first, then one-to-one (correspondence_search_kd_tree.hpp:224-225)
    assert _pairs(orc, search_dir="both", inlier_fraction=0.75)[0] == [(0, 0), (1, 2), (0, 1)]


def test_first_to_second_search_pinned_on_reference_nanoflann(orc):
    """FIRST_TO_SECOND / BOTH rebuild a kd-tree over the transformed source on every call
    (correspondence_search_kd_tree.hpp:195-204, :214-226). With the reference's own nanoflann doing that search (tree
    built and queried per call; its lists and ICP transform stored in tests/golden/ref_nanoflann.json), the brute-force
    restatement the GPU tests compare against must give the same lists on data without exact ties, and the same ICP
    transforms."""
    from cilantro_b200 import synth
    from golden import make_ref_golden as ref_golden

    g = ref_golden.load()
    dst, src, _, T_ref = synth.icp_pair(20000, seed=4, noise=0.003, n_src=15000)
    T0 = (0.7 * np.asarray(T_ref) + 0.3 * np.hstack([np.eye(3), np.zeros((3, 1))])).astype(np.float32)
    max_d2 = np.float32((2.0 * 20000 ** (-1.0 / 3.0)) ** 2)
    for mode, want in zip(ref_golden.ENGINE_MODES, g["engine_f2s"]):
        b = orc.engine_correspondences(dst, src, T0, orc.BruteKnn(dst), max_d2, f2s_reference=False, **mode)
        assert want["n"] > 1000 and len(b[0]) == want["n"]
        assert ref_golden.sha(b[0]) == want["first"] and ref_golden.sha(b[1]) == want["second"]
        assert ref_golden.sha(b[2]) == want["value"]
    rb = orc.icp(dst, src, orc.BruteKnn(dst), f2s_reference=False, max_d2=max_d2, **ref_golden.ENGINE_ICP)
    assert rb["num_corr"] == g["engine_icp"]["num_corr"]
    assert np.array_equal(rb["T"], np.float32(g["engine_icp"]["T"]).reshape(3, 4))


def test_engine_icp_recovers_a_shift(orc):
    rng = np.random.default_rng(0)
    dst = rng.random((1500, 3), dtype=np.float32)
    shift = np.array([0.004, -0.003, 0.002], np.float32)
    src = (dst[:1000] - shift).astype(np.float32)
    for mode in (dict(search_dir="both", require_reciprocal=True), dict(search_dir="first_to_second", one_to_one=True),
                 dict(inlier_fraction=0.9)):
        r = orc.icp(dst, src, orc.BruteKnn(dst), metric="p2p", max_iter=10, tol=1e-7, max_d2=np.float32(0.02**2), **mode)
        assert np.allclose(r["T"][:, 3], shift, atol=2e-5), (mode, r["T"][:, 3])
        assert np.allclose(r["T"][:, :3], np.eye(3), atol=2e-5)
