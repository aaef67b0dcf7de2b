"""Every device reduction against an exact float64 sum, at sizes that cross its block and group boundaries.

For each reduced value the per-element terms t_i are rebuilt in numpy and the reference is math.fsum(t), which is
correctly rounded. A double sum of N terms in any order is within (N - 1) * 2^-53 * sum|t_i| of the exact sum, so
|gpu - ref| <= (N + 4) * 2^-53 * sum|t_i| holds for every summation order (the +4 covers the few roundings inside a
term: nvcc contracts `acc += w * (a*a + b*b)` into FMAs, so per-term values are not bit-reproducible in numpy). A block
row dropped or counted twice, or a wrong term, lands orders of magnitude above the bound; correct code never exceeds it.

The fp32 stages before the double accumulation are reproduced bit for bit: the kernels use __fsub_rn / __fmul_rn and
numpy float32 does not fuse, so the restatements below follow the kernels' operation order exactly.

The two-level reductions (reduce.cuh) fold rows in groups of kReduceGroup = 64 blocks of 256 threads. The ICP pass runs
one thread per source point, so its edges are at n_src = 256 * 64 * g (+-1), and above 64 groups the grid-level fold
loops. Each test prints the largest |gpu - ref| / bound it saw.
"""
import math

import numpy as np
import pytest

from cilantro_b200 import synth
from conftest import frob

gpu = pytest.mark.gpu

U = 2.0 ** -53
# CUDA's expf is within 2 ulp (<= 2^-22 relative); the float product with the metric weight adds 2^-24
RBF_REL = 6.0 * 2.0 ** -24
REDUCE_BLOCK, REDUCE_GROUP = 256, 64


def _ut(r, c):
    return r * 6 - (r * (r - 1)) // 2 + (c - r)


def _exact(cols):
    """cols: list of float64 arrays (the terms of each reduced value). Returns (fsum per value, rigorous bound)."""
    ref = np.array([math.fsum(c) for c in cols])
    bound = np.array([(len(c) + 4) * U * float(np.abs(c).sum()) for c in cols])
    return ref, bound


def _check(got, ref, bound, what):
    """Asserts |got - ref| <= bound value by value; returns the largest |got - ref| / bound."""
    got = np.asarray(got, np.float64).reshape(-1)
    diff = np.abs(got - ref)
    bad = ~(diff <= bound)
    assert not bad.any(), (f"{what}: values {np.flatnonzero(bad).tolist()} differ by {diff[bad]} > bound {bound[bad]} "
                           f"(gpu {got[bad]}, exact {ref[bad]})")
    return float(np.max(np.where(bound > 0, diff / np.where(bound > 0, bound, 1.0), 0.0), initial=0.0))


def _f32_mean(x):
    """float32 of the float64 mean, as the device computes it (double sum / n, then a float conversion). Asserts that
    the double sum's error cannot move the result across a float32 rounding boundary. When every partial sum is a
    multiple of the smallest input ulp below 2^53 of them, the device's double sum is exact in any order and the mean
    is the same correctly rounded quotient on both sides: no margin is needed."""
    n = x.shape[0]
    out = np.empty(3, np.float32)
    for r in range(3):
        c = x[:, r].astype(np.float64)
        m = math.fsum(c) / n
        nz = np.abs(x[:, r][x[:, r] != 0])
        exact = len(nz) == 0 or float(np.abs(c).sum()) < 2.0 ** 53 * float(np.spacing(nz).min())
        eps = 0.0 if exact else (n + 4) * U * float(np.abs(c).sum()) / n + abs(m) * 2.0 ** -51
        assert np.float32(m - eps) == np.float32(m + eps), f"mean {m!r} sits on a float32 rounding tie: pick another seed"
        out[r] = np.float32(m)
    return out


def _rotate(T, v):
    """R v in the contract order of rotate_rigid / sum3: r0 x + (r1 y + r2 z), float32 round-to-nearest."""
    T = np.asarray(T, np.float32)
    v = np.asarray(v, np.float32)
    return np.stack([T[r, 0] * v[:, 0] + (T[r, 1] * v[:, 1] + T[r, 2] * v[:, 2]) for r in range(3)], axis=1)


# ---- restatements of the ICP accumulation (icp_accumulate.cuh) -------------------------------------------------------
def p2p_terms(dst, q, i1, i2):
    """kModeP2P: {1, d, q, d q^T} per pair. A product of two floats is exact in double."""
    d = dst[i1].astype(np.float64)
    s = q[i2].astype(np.float64)
    cols = [np.ones(len(i1))] + [d[:, r] for r in range(3)] + [s[:, r] for r in range(3)]
    cols += [d[:, r] * s[:, c] for r in range(3) for c in range(3)]
    return cols


def combined_terms(dst, dst_n, q, i1, i2, dm, sm, w_pt, w_pl, src_n_rot=None, d2=None, wc_pt=None, wc_pl=None):
    """kModeCombined with an identity inner transform: 28 term columns (count, 21 upper-triangle entries of A, 6 of b),
    and per column the sum of |t| over the terms that carry an RBF weight."""
    m = len(i1)
    d = dst[i1] - dm
    s = q[i2] - sm
    v, e = d + s, d - s
    V, E = v.astype(np.float64), e.astype(np.float64)
    zero = np.zeros(m)
    pt = [zero] * 28
    pl = [zero] * 28
    rbf = np.zeros(28)

    def weight(w, wc):
        if wc is None:
            return np.full(m, float(np.float32(w)))
        return float(np.float32(w)) * np.exp((np.float32(wc) * d2).astype(np.float64))

    if w_pt > 0:
        w = weight(w_pt, wc_pt)
        A = {(0, 0): w * (V[:, 1] * V[:, 1] + V[:, 2] * V[:, 2]), (0, 1): -(w * (V[:, 0] * V[:, 1])),
             (0, 2): -(w * (V[:, 0] * V[:, 2])), (1, 1): w * (V[:, 0] * V[:, 0] + V[:, 2] * V[:, 2]),
             (1, 2): -(w * (V[:, 1] * V[:, 2])), (2, 2): w * (V[:, 0] * V[:, 0] + V[:, 1] * V[:, 1]),
             (0, 4): -(w * V[:, 2]), (0, 5): w * V[:, 1], (1, 3): w * V[:, 2], (1, 5): -(w * V[:, 0]),
             (2, 3): -(w * V[:, 1]), (2, 4): w * V[:, 0], (3, 3): w, (4, 4): w, (5, 5): w}
        for (r, c), t in A.items():
            pt[1 + _ut(r, c)] = t
        b = [w * (V[:, 1] * E[:, 2] - V[:, 2] * E[:, 1]), w * (V[:, 2] * E[:, 0] - V[:, 0] * E[:, 2]),
             w * (V[:, 0] * E[:, 1] - V[:, 1] * E[:, 0]), w * E[:, 0], w * E[:, 1], w * E[:, 2]]
        for r in range(6):
            pt[22 + r] = b[r]
        if wc_pt is not None:
            rbf += np.array([np.abs(t).sum() for t in pt])
    if w_pl > 0:
        n = dst_n[i1]
        if src_n_rot is not None:  # symmetric metric: n = n_dst + R_T n_src
            n = n + src_n_rot[i2]
        c0 = v[:, 1] * n[:, 2] - v[:, 2] * n[:, 1]
        c1 = v[:, 2] * n[:, 0] - v[:, 0] * n[:, 2]
        c2 = v[:, 0] * n[:, 1] - v[:, 1] * n[:, 0]
        N = n.astype(np.float64)
        av = [c0.astype(np.float64), c1.astype(np.float64), c2.astype(np.float64), N[:, 0], N[:, 1], N[:, 2]]
        rd = N[:, 0] * E[:, 0] + (N[:, 1] * E[:, 1] + N[:, 2] * E[:, 2])
        w = weight(w_pl, wc_pl)
        for r in range(6):
            wr = w * av[r]
            for c in range(r, 6):
                pl[1 + _ut(r, c)] = wr * av[c]
            pl[22 + r] = wr * rd
        if wc_pl is not None:
            rbf += np.array([np.abs(t).sum() for t in pl])
    pt[0] = np.ones(m)
    cols = [np.concatenate([a, b]) if (w_pt > 0 and w_pl > 0) else (a if w_pt > 0 or j == 0 else b)
            for j, (a, b) in enumerate(zip(pt, pl))]
    return cols, rbf


def kabsch64(d, s):
    """Float64 Kabsch (SVD with the reflection fix): T with d ~ R s + t."""
    d = np.asarray(d, np.float64)
    s = np.asarray(s, np.float64)
    mu_d, mu_s = d.mean(0), s.mean(0)
    H = (d - mu_d).T @ (s - mu_s)
    Uh, _, Vt = np.linalg.svd(H)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Uh @ Vt))])
    R = Uh @ D @ Vt
    return np.hstack([R, (mu_d - R @ mu_s)[:, None]]), mu_s


# ---- ICP inputs -------------------------------------------------------------------------------------------------------
T_ICP = synth.rigid_from_axis_angle([1, 2, 3], 0.05, [0.01, -0.02, 0.03]).astype(np.float32)
M_DST = 2048          # small destination cloud: the brute-force oracle stays cheap at 1 M queries
MAX_D2 = np.float32(0.01 ** 2)
RBF_SIGMA = 0.003     # exp(coeff * d2) spans ~(0.3, 1) for the 0.002 noise below


def _unit(rng, n):
    g = rng.standard_normal((n, 3))
    return (g / np.linalg.norm(g, axis=1, keepdims=True)).astype(np.float32)


def icp_inputs(n_src, seed, offset=None, far_half=False, all_far=False):
    """dst: M_DST points in the unit cube (+ normals); src: n_src noisy copies of dst points mapped by T_ICP^-1, so
    T_ICP src lands within 0.002 of a dst point. far_half moves the second half of src 5 away along x (after the
    cell sort those points fill whole blocks of their own); all_far moves every source point."""
    rng = np.random.default_rng(seed)
    dst = rng.random((M_DST, 3), dtype=np.float32)
    nrm = _unit(rng, M_DST)
    base = dst[rng.integers(0, M_DST, n_src)] + (rng.random((n_src, 3), dtype=np.float32) - 0.5) * np.float32(0.004)
    if far_half:
        base[n_src // 2:, 0] += np.float32(5.0)
    if all_far:
        base[:, 0] += np.float32(5.0)
    if offset is not None:
        off = np.asarray(offset, np.float32)
        dst = (dst + off).astype(np.float32)
        base = (base + off).astype(np.float32)
    src = synth.apply(synth.invert(T_ICP), base)
    return dst, nrm, src, _unit(rng, n_src)


# (label, metric kwargs for accumulate, use source normals)
VARIANTS = [
    ("pt", dict(w_pt=1.0, w_pl=0.0), False),
    ("pl", dict(w_pt=0.0, w_pl=1.0), False),
    ("pt+pl", dict(w_pt=0.3, w_pl=1.0), False),
    ("symmetric", dict(w_pt=0.3, w_pl=1.0), True),
    ("rbf pt", dict(w_pt=0.3, w_pl=1.0, pt_rbf_sigma=RBF_SIGMA), False),
    ("rbf pl", dict(w_pt=0.3, w_pl=1.0, pl_rbf_sigma=RBF_SIGMA), False),
]


def _combined_reference(cb, kw, dst, nrm, q, src, src_n, T, i1, i2, v):
    dm = _f32_mean(dst)
    sm = _rotate(T, _f32_mean(src)[None])[0] + T[:, 3]  # apply_point: (r0 x + (r1 y + r2 z)) + t
    cols, rbf = combined_terms(dst, nrm, q, i1, i2, dm, sm, kw["w_pt"], kw["w_pl"],
                               src_n_rot=_rotate(T, src_n) if src_n is not None else None, d2=v,
                               wc_pt=cb.rbf_coeff(kw["pt_rbf_sigma"]) if "pt_rbf_sigma" in kw else None,
                               wc_pl=cb.rbf_coeff(kw["pl_rbf_sigma"]) if "pl_rbf_sigma" in kw else None)
    ref, bound = _exact(cols)
    return ref, bound + RBF_REL * rbf


# 1 and 2 points, one block +-1, 64 blocks = one full group (+1 = a second group of one block), 129 blocks, a partial
# last group (~300 k: 1172 blocks = 18 groups + 20), and 1048577 = 4097 blocks = 65 groups (the grid fold loops)
ICP_SIZES = [1, 2, 255, 256, 257, 16384, 16385, 32769, 300_001, 1_048_577]


@gpu
@pytest.mark.parametrize("n_src", ICP_SIZES)
def test_icp_accumulate_exact(cb, ctx, orc, n_src):
    dst, nrm, src, src_n = icp_inputs(n_src, seed=100 + n_src % 97)
    T = T_ICP
    q = orc.transform_points(T, src)
    oi, od = orc.BruteKnn(dst).query(q, MAX_D2)
    keep = oi >= 0
    i2 = np.flatnonzero(keep)
    i1, v = oi[keep], od[keep]
    assert len(i1) == n_src  # every source point matches: the sums cover every block of the grid
    worst = {}
    d_dst = cb.Cloud(ctx, dst, nrm)
    icp = cb.Icp(ctx, d_dst, cb.Cloud(ctx, src))
    sums = icp.accumulate(T, metric="p2p", max_d2=MAX_D2)
    g1, g2, gv = icp.correspondences()
    assert np.array_equal(g1, i1) and np.array_equal(g2, i2) and np.array_equal(gv.view(np.uint32), v.view(np.uint32))
    assert sums[0] == len(i1)
    ref, bound = _exact(p2p_terms(dst, q, i1, i2))
    worst["p2p"] = _check(sums, ref, bound, f"p2p moments, n_src={n_src}")
    icp_sym = None
    for label, kw, with_src_n in VARIANTS:
        if with_src_n and icp_sym is None:
            icp_sym = cb.Icp(ctx, d_dst, cb.Cloud(ctx, src, src_n))
        sums = (icp_sym if with_src_n else icp).accumulate(T, metric="combined", max_d2=MAX_D2, **kw)
        assert sums[0] == len(i1)
        ref, bound = _combined_reference(cb, kw, dst, nrm, q, src, src_n if with_src_n else None, T, i1, i2, v)
        worst[label] = _check(sums, ref, bound, f"combined {label}, n_src={n_src}")
    print(f"icp accumulate n_src={n_src}: max |gpu - exact| / bound " + ", ".join(f"{k} {w:.3g}" for k, w in worst.items()))


@gpu
def test_icp_accumulate_offset_cloud(cb, ctx, orc):
    """Far from the origin: the combined sums are centred on dm / sm, the point-to-point sums are raw."""
    n_src = 16385
    dst, nrm, src, src_n = icp_inputs(n_src, seed=7, offset=(2000.0, -1500.0, 800.0))
    q = orc.transform_points(T_ICP, src)
    oi, od = orc.BruteKnn(dst).query(q, MAX_D2)
    keep = oi >= 0
    i1, i2, v = oi[keep], np.flatnonzero(keep), od[keep]
    assert len(i1) > 0.99 * n_src
    icp = cb.Icp(ctx, cb.Cloud(ctx, dst, nrm), cb.Cloud(ctx, src))
    sums = icp.accumulate(T_ICP, metric="p2p", max_d2=MAX_D2)
    g1, g2, _ = icp.correspondences()
    assert np.array_equal(g1, i1) and np.array_equal(g2, i2)
    worst = {"p2p": _check(sums, *_exact(p2p_terms(dst, q, i1, i2)), "offset p2p")}
    for label, kw, with_src_n in VARIANTS:
        if with_src_n:
            continue
        sums = icp.accumulate(T_ICP, metric="combined", max_d2=MAX_D2, **kw)
        ref, bound = _combined_reference(cb, kw, dst, nrm, q, src, None, T_ICP, i1, i2, v)
        worst[label] = _check(sums, ref, bound, f"offset combined {label}")
    print("icp accumulate offset (2000, -1500, 800): max |gpu - exact| / bound " +
          ", ".join(f"{k} {w:.3g}" for k, w in worst.items()))


@gpu
def test_icp_accumulate_half_out_of_range_and_no_match(cb, ctx, orc):
    n_src = 32769
    # half the source beyond max_d2: after the cell sort whole blocks contribute zero rows
    dst, nrm, src, _ = icp_inputs(n_src, seed=11, far_half=True)
    q = orc.transform_points(T_ICP, src)
    oi, od = orc.BruteKnn(dst).query(q, MAX_D2)
    keep = oi >= 0
    i1, i2, v = oi[keep], np.flatnonzero(keep), od[keep]
    assert len(i1) == n_src // 2
    icp =cb.Icp(ctx, cb.Cloud(ctx, dst, nrm), cb.Cloud(ctx, src))
    sums = icp.accumulate(T_ICP, metric="p2p", max_d2=MAX_D2)
    assert sums[0] == len(i1)
    worst = {"p2p": _check(sums, *_exact(p2p_terms(dst, q, i1, i2)), "half-matched p2p")}
    kw = dict(w_pt=0.3, w_pl=1.0)
    sums = icp.accumulate(T_ICP, metric="combined", max_d2=MAX_D2, **kw)
    worst["pt+pl"] = _check(sums, *_combined_reference(cb, kw, dst, nrm, q, src, None, T_ICP, i1, i2, v),
                            "half-matched combined")
    print("icp accumulate, half the source out of range: max |gpu - exact| / bound " +
          ", ".join(f"{k} {w:.3g}" for k, w in worst.items()))
    # nothing matches: every sum is exactly zero
    dst, nrm, src, src_n = icp_inputs(n_src, seed=12, all_far=True)
    assert (orc.BruteKnn(dst).query(orc.transform_points(T_ICP, src), MAX_D2)[0] < 0).all()
    icp = cb.Icp(ctx, cb.Cloud(ctx, dst, nrm), cb.Cloud(ctx, src, src_n))
    assert np.array_equal(icp.accumulate(T_ICP, metric="p2p", max_d2=MAX_D2), np.zeros(16))
    for _, kw, _ in VARIANTS:
        assert np.array_equal(icp.accumulate(T_ICP, metric="combined", max_d2=MAX_D2, **kw), np.zeros(28)), kw


# ---- covariance / PCA (stats_kernels.cu moments_kernel, capi_stats.cu) ------------------------------------------------
def _mean_cov_reference(p):
    """Exact float64 mean and two-pass centred covariance, and the tolerances of the float32 outputs."""
    n = p.shape[0]
    P = p.astype(np.float64)
    mean = np.array([math.fsum(P[:, r]) / n for r in range(3)])
    X = P - mean
    cov = np.array([[math.fsum(X[:, r] * X[:, c]) / (n - 1) for c in range(3)] for r in range(3)])
    # the device sums about a float32 pivot c (the mean of the first <= 4096 points) in double
    head = p[: min(n, 4096)].astype(np.float64)
    c = np.float32(head.mean(0)).astype(np.float64)
    Y = P - c
    eps_mean = 2 * (n + 4) * U * np.abs(Y).sum(0) / n
    tol_mean = np.spacing(np.abs(np.float32(mean))).astype(np.float64) + eps_mean
    q = np.sqrt((Y * Y).sum(0))
    eps_cov = 4 * (n + 4) * U * np.outer(q, q) / (n - 1)
    d = np.sqrt(np.diag(cov))
    tol_cov = 2.0 ** -23 * np.outer(d, d) + 2 * eps_cov
    return mean, cov, tol_mean, tol_cov


def _check_mean_cov(cb, ctx, p, what):
    cloud = cb.Cloud(ctx, p)
    mean, cov, ok = cb.mean_cov(ctx, cloud)
    assert ok
    rm, rc, tm, tc = _mean_cov_reference(p)
    worst = max(_check(mean, rm, tm, f"mean, {what}"), _check(cov, rc.reshape(-1), tc.reshape(-1), f"cov, {what}"))
    got = cb.pca(ctx, cloud)
    assert got["ok"] and np.array_equal(got["mean"], mean) and np.array_equal(got["cov"], cov)
    ev, V = got["eigenvalues"].astype(np.float64), got["eigenvectors"].astype(np.float64)
    recon = V @ np.diag(ev) @ V.T
    assert np.abs(recon - cov).max() <= 1e-5 * np.abs(ev).max(), what
    return worst


def _odd_trip_n(sm_count):
    """An n with n % 4 == 3 whose float4 group count ng, for every occupancy of 1..8 blocks per SM (grid capped at
    sm_count * per_sm blocks, stride S = 256 * blocks), runs moments_kernel's paired loop at least twice and then leaves
    a single trip for some threads: ng >= 4 S and ng % 2S != 0."""
    strides = [sm_count * p * REDUCE_BLOCK for p in range(1, 9)]
    ng = 4 * strides[-1] + 1
    while any(ng % (2 * s) == 0 for s in strides):
        ng += 1
    return 4 * ng + 3


MEAN_COV_SIZES = [2, 3, 4, 5, 7, 8, 9, 4095, 4096, 4097, 3 * 2 ** 20 + 3]


@gpu
@pytest.mark.parametrize("n", MEAN_COV_SIZES)
def test_mean_cov_exact(cb, ctx, n):
    rng = np.random.default_rng(n)
    p = (rng.random((n, 3), dtype=np.float32) * np.float32([2.0, 1.0, 0.5]) + np.float32([0.3, -0.7, 1.1]))
    w = _check_mean_cov(cb, ctx, p.astype(np.float32), f"n={n}")
    print(f"mean_cov n={n}: max |gpu - exact| / tol {w:.3g}")


@gpu
def test_mean_cov_grid_stride_odd_trip(cb, ctx):
    n = _odd_trip_n(ctx.device_info()["sm_count"])
    p = np.random.default_rng(5).random((n, 3), dtype=np.float32)
    w = _check_mean_cov(cb, ctx, p, f"n={n}")
    print(f"mean_cov n={n} (odd grid-stride trip): max |gpu - exact| / tol {w:.3g}")


@gpu
def test_mean_cov_far_from_origin_and_skewed_pivot(cb, ctx):
    rng = np.random.default_rng(9)
    n = 100_003
    far = (rng.random((n, 3), dtype=np.float32) * np.float32(1e-2) + np.float32(1e4)).astype(np.float32)
    w1 = _check_mean_cov(cb, ctx, far, "offset 1e4, spread 1e-2")
    # the first 4096 points, which set the pivot, all sit at one end of the cloud
    n = 200_001
    p = rng.random((n, 3), dtype=np.float32)
    p[:4096] = (p[:4096] * np.float32(0.01) + np.float32([5.0, -3.0, 4.0])).astype(np.float32)
    w2 = _check_mean_cov(cb, ctx, p, "pivot at one end")
    print(f"mean_cov: max |gpu - exact| / tol offset cloud {w1:.3g}, skewed pivot {w2:.3g}")


# ---- k-means sums (kmeans.cu kmeans_assign_kernel) --------------------------------------------------------------------
def _global_atomic_path(K):
    # kmeans_step: the per-block shared-memory sums are used while K * 4 doubles + the 1024-centroid float4 chunk fit
    # in 200 KiB (K <= 5888); above that kmeans_assign_kernel<false> adds straight into global memory
    return K * 4 * 8 + 1024 * 16 > 200 * 1024


def _cluster_sums(pts, labels, K):
    """Exact per-cluster sums and bounds (K x 3)."""
    order = np.argsort(labels, kind="stable")
    cuts = np.searchsorted(labels[order], np.arange(K + 1))
    P = pts[order].astype(np.float64)
    ref = np.zeros((K, 3))
    bound = np.zeros((K, 3))
    for j in range(K):
        blk = P[cuts[j]:cuts[j + 1]]
        if len(blk):
            ref[j] = [math.fsum(blk[:, r]) for r in range(3)]
            bound[j] = (len(blk) + 4) * U * np.abs(blk).sum(0)
    return ref, bound


# n not a multiple of the 1024-point tile, or smaller than one tile; K on both sides of the smem / global switch
@gpu
@pytest.mark.parametrize("K,n", [(1, 700), (1024, 700), (1024, 5001), (1025, 5001), (5888, 20003), (5889, 20003),
                                 (8192, 30001)])
def test_kmeans_assign_exact(cb, ctx, orc, K, n):
    assert _global_atomic_path(K) == (K >= 5889)
    rng = np.random.default_rng(K + n)
    pts = rng.random((n, 3), dtype=np.float32)
    cent = rng.random((K, 3), dtype=np.float32)
    labels, sums, counts = cb.kmeans_assign(ctx, cb.Cloud(ctx, pts), cent)
    want, _ = orc.kmeans_assign(pts, cent)
    assert np.array_equal(labels, want.astype(np.int64))
    assert np.array_equal(counts, np.bincount(labels, minlength=K))
    ref, bound = _cluster_sums(pts, labels, K)
    w = _check(sums, ref.reshape(-1), bound.reshape(-1), f"k-means sums K={K} n={n}")
    print(f"kmeans_assign K={K} n={n} ({'global' if _global_atomic_path(K) else 'shared'} sums): "
          f"max |gpu - exact| / bound {w:.3g}")


@gpu
@pytest.mark.parametrize("K", [64, 5889])
def test_kmeans_one_iteration_centroids(cb, ctx, K):
    """centroid = float(sum) * (1.0f / float(count)) (kmeans.cu, kmeans.hpp:179-181) of the exact sums, within 1 ulp
    (the device's double sum may round to the neighbouring float)."""
    n = 4 * K + 333
    rng = np.random.default_rng(K)
    pts = rng.random((n, 3), dtype=np.float32)
    cent0 = pts[rng.permutation(n)[:K]].copy()  # distinct data points: no cluster is empty, no repair step runs
    res = cb.kmeans_cluster(ctx, cb.Cloud(ctx, pts), cent0, max_iter=1, tol=0.0)
    assert res["iterations"] == 1
    labels, _, counts = cb.kmeans_assign(ctx, cb.Cloud(ctx, pts), cent0)
    assert counts.min() > 0
    ref, _ = _cluster_sums(pts, labels, K)
    inv = np.float32(1.0) / counts.astype(np.float32)
    want = ref.astype(np.float32) * inv[:, None]
    ulps = np.abs(res["centroids"].view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, (K, ulps.max())


# ---- RANSAC re-estimation (ransac.cu inlier_moments_kernel) -----------------------------------------------------------
def _ransac_inputs(n, seed, offset=0.0):
    rng = np.random.default_rng(seed)
    src = (rng.random((n, 3), dtype=np.float32) + np.float32(offset)).astype(np.float32)
    T = synth.t_ref_default()
    dst = synth.apply(T, src) + (rng.standard_normal((n, 3)) * 0.002).astype(np.float32)
    out = rng.random(n) >= 0.6
    dst[out] = (rng.random((int(out.sum()), 3), dtype=np.float32) + np.float32(offset)).astype(np.float32)
    return dst.astype(np.float32), src


def _ransac_sizes(sm_count):
    cap = sm_count * 4 * REDUCE_BLOCK  # the grid is capped at sm_count * 4 blocks
    return [200, REDUCE_BLOCK * REDUCE_GROUP + 1, cap, 2 * cap + 1001]


def _ransac_check(cb, ctx, dst, src, seed):
    d_dst, d_src = cb.Cloud(ctx, dst), cb.Cloud(ctx, src)
    plain = cb.ransac_rigid(ctx, d_dst, d_src, seed=seed, max_iter=200, re_estimate=False)
    res = cb.ransac_rigid(ctx, d_dst, d_src, seed=seed, max_iter=200, re_estimate=True)
    inl = plain["inliers"]
    assert len(inl) >= 3
    T64, mu_s = kabsch64(dst[inl], src[inl])
    T = res["T"].astype(np.float64)
    err_R = np.abs(T[:, :3] - T64[:, :3]).max() / 2.0 ** -22
    err_t = np.abs(T[:, 3] - T64[:, 3]).max() / (2.0 ** -22 * (np.linalg.norm(T64[:, 3]) + 3 * np.linalg.norm(mu_s)))
    assert err_R <= 1 and err_t <= 1, (len(dst), err_R, err_t)
    return max(err_R, err_t), len(inl)


@gpu
def test_ransac_reestimate_matches_float64_kabsch(cb, ctx):
    for n in _ransac_sizes(ctx.device_info()["sm_count"]):
        dst, src = _ransac_inputs(n, seed=n)
        w, k = _ransac_check(cb, ctx, dst, src, seed=3)
        print(f"ransac re-estimate n={n} ({k} inliers): max |gpu - float64 Kabsch| / tol {w:.3g}")


@gpu
def test_ransac_reestimate_offset_cloud(cb, ctx):
    n = ctx.device_info()["sm_count"] * 4 * REDUCE_BLOCK
    dst, src = _ransac_inputs(n, seed=21, offset=1e3)
    w, k = _ransac_check(cb, ctx, dst, src, seed=4)
    print(f"ransac re-estimate n={n} offset 1e3 ({k} inliers): max |gpu - float64 Kabsch| / tol {w:.3g}")


# ---- run-to-run determinism (reduce.cuh: fixed summation order) -------------------------------------------------------
@gpu
def test_reductions_are_deterministic(cb, ctx):
    dst, nrm, src, src_n = icp_inputs(300_001, seed=2)
    icp = cb.Icp(ctx, cb.Cloud(ctx, dst, nrm), cb.Cloud(ctx, src, src_n))
    for kw in (dict(metric="p2p"), dict(metric="combined", w_pt=0.3, w_pl=1.0, pl_rbf_sigma=RBF_SIGMA)):
        runs = [icp.accumulate(T_ICP, max_d2=MAX_D2, **kw) for _ in range(3)]
        assert all(np.array_equal(r.view(np.uint64), runs[0].view(np.uint64)) for r in runs), kw
    pts = cb.Cloud(ctx, np.random.default_rng(3).random((3 * 2 ** 20 + 3, 3), dtype=np.float32))
    runs = [cb.mean_cov(ctx, pts) for _ in range(3)]
    assert all(np.array_equal(r[0], runs[0][0]) and np.array_equal(r[1], runs[0][1]) for r in runs)
    n = 2 * ctx.device_info()["sm_count"] * 4 * REDUCE_BLOCK + 1001
    dst, src = _ransac_inputs(n, seed=8)
    d_dst, d_src = cb.Cloud(ctx, dst), cb.Cloud(ctx, src)
    runs = [cb.ransac_rigid(ctx, d_dst, d_src, seed=5, max_iter=200)["T"] for _ in range(3)]
    assert all(np.array_equal(r.view(np.uint32), runs[0].view(np.uint32)) for r in runs)


# ---- the restatement itself, checked on the CPU ------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["p2p"] + [v[0] for v in VARIANTS[:4]])
def test_restated_sums_solve_like_the_oracle(cb, orc, variant):
    """The restated 16 / 28 sums, fed to the product's host solvers, give the oracle's double-accumulated Kabsch /
    Gauss-Newton estimate: validates the restatement without a GPU."""
    dst, nrm, src, src_n = icp_inputs(3000, seed=31)
    T = T_ICP
    q = orc.transform_points(T, src)
    i1, i2, v = orc.find_correspondences(T, src, orc.BruteKnn(dst), MAX_D2)
    assert len(i1) == 3000
    if variant == "p2p":
        sums, _ = _exact(p2p_terms(dst, q, i1, i2))
        got, ok = cb.solve_kabsch_moments(sums)
        want, ok_o = orc.kabsch(dst[i1], q[i2], accum_double=True)
        assert ok and ok_o
        assert frob(got, want) < 1e-6, frob(got, want)
        return
    kw, with_src_n = {label: (kw, s) for label, kw, s in VARIANTS}[variant]
    sums, _ = _combined_reference(cb, kw, dst, nrm, q, src, src_n if with_src_n else None, T, i1, i2, v)
    got, _ = cb.solve_gauss_newton(sums)
    dm = _f32_mean(dst)
    sm = _rotate(T, _f32_mean(src)[None])[0] + T[:, 3]
    got = got.astype(np.float64)
    got[:, 3] = got[:, 3] - got[:, :3] @ sm.astype(np.float64) + dm.astype(np.float64)  # transform_estimation.hpp:365
    want, _ = orc.estimate_combined(dst, nrm, q, i1, i2, kw["w_pt"], kw["w_pl"], 1, 1e-5, dm, sm,
                                    src_n=_rotate(T, src_n) if with_src_n else None, accum_double=True)
    assert frob(got, want) < 1e-6, (variant, frob(got, want))
