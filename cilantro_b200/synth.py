"""Seeded synthetic workloads (SURVEY.md §8(d)); shared by tests/ and bench.py. numpy only."""
import numpy as np


def rigid_from_axis_angle(axis, angle, t):
    axis = np.asarray(axis, np.float64)
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    R = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)
    T = np.zeros((3, 4), np.float64)
    T[:, :3] = R
    T[:, 3] = np.asarray(t, np.float64)
    return T


def invert(T):
    T = np.asarray(T, np.float64)
    R, t = T[:, :3], T[:, 3]
    out = np.zeros((3, 4), np.float64)
    out[:, :3] = R.T
    out[:, 3] = -R.T @ t
    return out


def apply(T, pts):
    T = np.asarray(T, np.float64)
    return (np.asarray(pts, np.float64) @ T[:, :3].T + T[:, 3]).astype(np.float32)


def t_ref_default():
    """AngleAxis(0.02 rad about (1,1,1)/sqrt(3)), t = (0.01, -0.005, 0.008)."""
    return rigid_from_axis_angle([1, 1, 1], 0.02, [0.01, -0.005, 0.008])


def t_ref_for(n):
    """Generating pose for an n-point uniform cloud in the unit cube.

    SURVEY.md §8(d) proposes AngleAxis(0.02 rad, (1,1,1)/sqrt 3), t = (0.01,-0.005,0.008) for every
    size. Measured here with the oracle: at 1 M points (mean spacing 0.01) that offset (up to 0.03 at
    the cube corners) is outside ICP's basin of convergence on a dense uniform cloud — nearest
    neighbours are almost all wrong matches and BOTH the reference path and ours stall at
    |T - T_ref|_F = 3e-2. The work per iteration is unchanged, but the run is useless as a
    correctness check, so the pose is scaled with the point spacing s = n^(-1/3): angle =
    min(0.02, s/4), translation scaled by the same factor. For n <= 2000 this is SURVEY's pose."""
    s = float(n) ** (-1.0 / 3.0)
    f = min(1.0, (s / 4.0) / 0.02)
    return rigid_from_axis_angle([1, 1, 1], 0.02 * f, [0.01 * f, -0.005 * f, 0.008 * f])


def icp_pair(n, seed=1, noise=0.001, with_normals=False, n_src=None, T_ref=None):
    """dst uniform in [0,1)^3; src = T_ref^-1 dst + uniform noise in +-noise (SURVEY §8(d) configs 2/3).

    Returns dst (n,3), src (n_src,3), dst_normals or None, T_ref (3,4 float64): the transform ICP
    should recover (src -> dst)."""
    rng = np.random.default_rng(seed)
    dst = rng.random((n, 3), dtype=np.float32)
    if T_ref is None:
        T_ref = t_ref_for(n)
    m = n if n_src is None else n_src
    base = dst[:m] if m <= n else rng.random((m, 3), dtype=np.float32)
    src = apply(invert(T_ref), base)
    src = (src + (rng.random((m, 3), dtype=np.float32) - 0.5) * np.float32(2 * noise)).astype(np.float32)
    nrm = None
    if with_normals:
        g = rng.standard_normal((n, 3)).astype(np.float32)
        nrm = (g / np.linalg.norm(g, axis=1, keepdims=True)).astype(np.float32)
    return dst, src, nrm, T_ref


def surface_cloud(n, seed=1, noise=0.0005):
    """A scanned-surface stand-in: the sheet z = 0.5 + 0.1 sin(6x) cos(5y) over [0,1)^2, sampled uniformly in
    (x, y) with Gaussian noise along z. Returns points (n,3) float32 and the analytic unit normals (n,3), +z side."""
    rng = np.random.default_rng(seed)
    xy = rng.random((n, 2))
    x, y = xy[:, 0], xy[:, 1]
    z = 0.5 + 0.1 * np.sin(6 * x) * np.cos(5 * y) + noise * rng.standard_normal(n)
    g = np.stack([-0.6 * np.cos(6 * x) * np.cos(5 * y), 0.5 * np.sin(6 * x) * np.sin(5 * y), np.ones(n)], axis=1)
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    return np.stack([x, y, z], axis=1).astype(np.float32), g.astype(np.float32)


def rigid_icp_example_pair(points, normals, seed=1):
    """The input recipe of the reference's examples/rigid_icp.cpp:25-65 on a loaded scan (BASELINE config 1):
    src = dst + 0.01 * U(-1,1)^3 (normals + 0.02 * U, re-normalised), dst keeps only x > -0.4, then
    src <- tf_ref * src with tf_ref = Rz(-0.1) Ry(0.1) Rx(-0.1), t = (-0.20, -0.05, 0.10).
    Returns dst_p, dst_n, src_p, src_n, tf_ref (3x4 float64); ICP should recover tf_ref^-1."""
    rng = np.random.default_rng(seed)
    p = np.asarray(points, np.float32)
    n = np.asarray(normals, np.float32)
    src_p = (p + np.float32(0.01) * (rng.random(p.shape, dtype=np.float32) * 2 - 1)).astype(np.float32)
    src_n = n + np.float32(0.02) * (rng.random(n.shape, dtype=np.float32) * 2 - 1)
    src_n = (src_n / np.linalg.norm(src_n, axis=1, keepdims=True)).astype(np.float32)
    keep = p[:, 0] > np.float32(-0.4)
    dst_p, dst_n = np.ascontiguousarray(p[keep]), np.ascontiguousarray(n[keep])

    def rot(axis, a):
        return np.asarray(rigid_from_axis_angle(axis, a, [0, 0, 0]))[:, :3]

    R = rot([0, 0, 1], -0.1) @ rot([0, 1, 0], 0.1) @ rot([1, 0, 0], -0.1)
    tf_ref = np.hstack([R, np.array([[-0.20], [-0.05], [0.10]])])
    src_p = apply(tf_ref, src_p).astype(np.float32)
    src_n = (src_n.astype(np.float64) @ R.T).astype(np.float32)
    return dst_p, dst_n, src_p, src_n, tf_ref


def kmeans_data(n, k, seed=1):
    """uniform [0,1)^3 points; initial centroids = first k points of a seeded shuffle (config 4)."""
    rng = np.random.default_rng(seed)
    pts = rng.random((n, 3), dtype=np.float32)
    idx = rng.permutation(n)[:k]
    return pts, pts[idx].copy()


def ransac_pairs(n, inlier_frac=0.3, seed=1, sigma=0.002):
    """src uniform [0,1)^3; dst = T_ref src + N(0, sigma^2) for inliers, uniform otherwise (config 5)."""
    rng = np.random.default_rng(seed)
    src = rng.random((n, 3), dtype=np.float32)
    T_ref = t_ref_default()
    dst = apply(T_ref, src) + (rng.standard_normal((n, 3)) * sigma).astype(np.float32)
    out = rng.random(n) >= inlier_frac
    dst[out] = rng.random((int(out.sum()), 3), dtype=np.float32)
    return dst.astype(np.float32), src, T_ref, ~out


def frobenius(Ta, Tb):
    return float(np.linalg.norm(np.asarray(Ta, np.float64) - np.asarray(Tb, np.float64)))


def segment_scene(n, seed=1, r_over_spacing=2.5):
    """The segmentation benchmark scene: a ground plane, floating boxes and spheres with analytic normals, every object
    more than r away from every other one. Returns (points, normals, radius2, objects, faces): radius2 = (2.5 x the
    point spacing)^2; `objects` = segments of the all-true evaluator, `faces` = segments of the normals evaluator at 2
    degrees (each box face is its own segment, a sphere stays whole: neighbouring normals differ by r / R < 2 degrees).
    Points are shuffled."""
    rng = np.random.default_rng(seed)
    n_box, n_sph = 8, 4
    # areas: ground 16 x 16 (scaled below), boxes 6 faces of edge 1.5, spheres of radius 1
    area = 16.0 * 16.0 + n_box * 6 * 1.5**2 + n_sph * 4 * np.pi
    h = float(np.sqrt(area / n))  # point spacing
    parts_p, parts_n = [], []

    def grid(u0, u1, v0, v1):
        us = np.arange(u0, u1 + 1e-9, h)
        vs = np.arange(v0, v1 + 1e-9, h)
        U, V = np.meshgrid(us, vs, indexing="ij")
        return U.ravel(), V.ravel()

    U, V = grid(0, 16, 0, 16)
    parts_p.append(np.stack([U, V, np.zeros_like(U)], 1))
    parts_n.append(np.tile([0.0, 0.0, 1.0], (U.size, 1)))
    # boxes on a 4 x 2 layout over the ground, floating 0.5 above it; spheres in a row beside them
    for b in range(n_box):
        o = np.array([1.0 + 3.5 * (b % 4), 1.0 + 3.5 * (b // 4), 0.5])
        e = 1.5
        for axis in range(3):
            for side in (0.0, e):
                U, V = grid(0, e, 0, e)
                p = np.zeros((U.size, 3))
                a1, a2 = [a for a in range(3) if a != axis]
                p[:, axis] = side
                p[:, a1], p[:, a2] = U, V
                nn = np.zeros((U.size, 3))
                nn[:, axis] = 1.0 if side > 0 else -1.0
                parts_p.append(p + o)
                parts_n.append(nn)
    for s in range(n_sph):
        c = np.array([2.0 + 3.8 * s, 11.0, 1.6])
        m = int(4 * np.pi / h**2)
        i = np.arange(m) + 0.5
        phi = np.arccos(1 - 2 * i / m)
        th = np.pi * (1 + 5**0.5) * i
        d = np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
        parts_p.append(c + d)
        parts_n.append(d)
    pts = np.concatenate(parts_p).astype(np.float32)
    nrm = np.concatenate(parts_n)
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    perm = rng.permutation(pts.shape[0])
    radius2 = float(np.float32((r_over_spacing * h) ** 2))
    return pts[perm], nrm[perm], radius2, 1 + n_box + n_sph, 1 + 6 * n_box + n_sph
