"""Seeded synthetic graphs of the shapes named in BASELINE.json (SURVEY.md section 8(d)).

No dataset ships with the reference (/root/reference/data/Readme.txt lists download URLs only), so every
configuration is generated here, deterministically from a seed, directly in the reference's *internal*
representation (inverse camera model ``x_cam = R(w) X + t``, intrinsics ``fx fy cx cy d`` with the
distortion already focal-scaled; include/slam/BASolverBase.h:260-327).
"""
from __future__ import annotations

import numpy as np

from .sppio import BAGraph, PoseGraph, GRAPH_SE2, GRAPH_SE3


def _rotmat_to_axis_angle(R: np.ndarray) -> np.ndarray:
    """Batched log map SO(3) -> axis-angle (magnitude in [0, pi])."""
    # via quaternion for stability near pi
    n = R.shape[0]
    q = np.empty((n, 4))  # w x y z
    tr = R[:, 0, 0] + R[:, 1, 1] + R[:, 2, 2]
    for i in range(n):
        m = R[i]
        if tr[i] > 0:
            s = np.sqrt(tr[i] + 1.0) * 2
            q[i] = [0.25 * s, (m[2, 1] - m[1, 2]) / s, (m[0, 2] - m[2, 0]) / s, (m[1, 0] - m[0, 1]) / s]
        elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
            s = np.sqrt(1.0 + m[0, 0] - m[1, 1] - m[2, 2]) * 2
            q[i] = [(m[2, 1] - m[1, 2]) / s, 0.25 * s, (m[0, 1] + m[1, 0]) / s, (m[0, 2] + m[2, 0]) / s]
        elif m[1, 1] > m[2, 2]:
            s = np.sqrt(1.0 + m[1, 1] - m[0, 0] - m[2, 2]) * 2
            q[i] = [(m[0, 2] - m[2, 0]) / s, (m[0, 1] + m[1, 0]) / s, 0.25 * s, (m[1, 2] + m[2, 1]) / s]
        else:
            s = np.sqrt(1.0 + m[2, 2] - m[0, 0] - m[1, 1]) * 2
            q[i] = [(m[1, 0] - m[0, 1]) / s, (m[0, 2] + m[2, 0]) / s, (m[1, 2] + m[2, 1]) / s, 0.25 * s]
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[q[:, 0] < 0] *= -1
    vn = np.linalg.norm(q[:, 1:], axis=1)
    ang = 2 * np.arctan2(vn, q[:, 0])
    scale = np.where(vn > 1e-12, ang / np.maximum(vn, 1e-300), 2.0)
    return q[:, 1:] * scale[:, None]


def _axis_angle_to_rotmat(w: np.ndarray) -> np.ndarray:
    th = np.linalg.norm(w, axis=1)
    k = w / np.maximum(th, 1e-300)[:, None]
    K = np.zeros((w.shape[0], 3, 3))
    K[:, 0, 1], K[:, 0, 2] = -k[:, 2], k[:, 1]
    K[:, 1, 0], K[:, 1, 2] = k[:, 2], -k[:, 0]
    K[:, 2, 0], K[:, 2, 1] = -k[:, 1], k[:, 0]
    I = np.eye(3)[None]
    return I + np.sin(th)[:, None, None] * K + (1 - np.cos(th))[:, None, None] * (K @ K)


def make_ba(n_cams: int, n_pts: int, seed: int, mean_extra_track: float = 3.35, max_track: int = 60,
            max_stride: int = 11, pixel_sigma: float = 0.5, cam_noise: float = 1e-2, rot_noise: float = 1e-3,
            pt_noise: float = 1e-2, distortion: float = 0.0, ring_radius: float = 8.0,
            interleave_ids: bool = False, shuffle_edges: bool = False, loops: int = 1) -> BAGraph:
    """Ring-of-cameras BA problem.

    Cameras sit on ``loops`` turns of a ring looking at the origin, points are uniform in the unit cube,
    track length is ``2 + Geometric(mean mean_extra_track)`` capped at ``max_track``; the cameras of a track
    are strided neighbours ``c0 + stride * j`` (so the reduced camera system is banded/structured as in real
    sequences). Observations carry N(0, pixel_sigma^2) noise and identity information.
    """
    rng = np.random.default_rng(seed)
    fx = fy = 800.0
    cx = cy = 400.0
    ang = 2 * np.pi * loops * np.arange(n_cams) / n_cams
    rad = ring_radius * (1.0 + 0.15 * np.arange(n_cams) / max(n_cams, 1) * (loops > 1))
    pos = np.stack([rad * np.sin(ang), 0.3 * np.sin(3 * ang), -rad * np.cos(ang)], 1)
    zc = -pos / np.linalg.norm(pos, axis=1, keepdims=True)
    up = np.array([0.0, 1.0, 0.0])
    xc = np.cross(np.broadcast_to(up, zc.shape), zc)
    xc /= np.linalg.norm(xc, axis=1, keepdims=True)
    yc = np.cross(zc, xc)
    R = np.stack([xc, yc, zc], 1)  # world -> camera
    t = -np.einsum("nij,nj->ni", R, pos)
    pts = rng.uniform(-1, 1, (n_pts, 3))

    k = 2 + rng.geometric(1.0 / (mean_extra_track + 1.0), n_pts) - 1
    k = np.minimum(k, min(max_track, n_cams))
    stride = rng.integers(1, max_stride + 1, n_pts)
    # keep stride * k below n_cams so that a track never visits a camera twice
    stride = np.minimum(stride, np.maximum((n_cams - 1) // np.maximum(k, 1), 1))
    k = np.minimum(k, (n_cams - 1) // stride + 1)
    c0 = rng.integers(0, n_cams, n_pts)
    total = int(k.sum())
    obs_pt_l = np.repeat(np.arange(n_pts), k)
    start = np.cumsum(k) - k
    j = np.arange(total) - np.repeat(start, k)
    obs_cam_l = (c0[obs_pt_l] + stride[obs_pt_l] * j) % n_cams

    x = np.einsum("nij,nj->ni", R[obs_cam_l], pts[obs_pt_l]) + t[obs_cam_l]
    kk = distortion / (0.5 * (fx + fy))
    u = fx * x[:, 0] / x[:, 2] + cx
    v = fy * x[:, 1] / x[:, 2] + cy
    r2 = (u - cx) ** 2 + (v - cy) ** 2
    u = cx + (1 + r2 * kk) * (u - cx)
    v = cy + (1 + r2 * kk) * (v - cy)
    z = np.stack([u, v], 1) + rng.normal(0, pixel_sigma, (total, 2))
    info = np.broadcast_to(np.eye(2), (total, 2, 2)).copy()

    # perturbed initial estimate
    pos_n = pos + rng.normal(0, cam_noise, pos.shape)
    dR = _axis_angle_to_rotmat(rng.normal(0, rot_noise, (n_cams, 3)))
    R_n = np.einsum("nij,njk->nik", dR, R)
    t_n = -np.einsum("nij,nj->ni", R_n, pos_n)
    aa = _rotmat_to_axis_angle(R_n)
    cams = np.concatenate([t_n, aa, np.tile([fx, fy, cx, cy, distortion], (n_cams, 1))], 1)
    pts_n = pts + rng.normal(0, pt_noise, pts.shape)

    nv = n_cams + n_pts
    if interleave_ids:
        # mix camera and point ids (cameras still appear in increasing order among themselves)
        slots = np.sort(rng.choice(nv, n_cams, replace=False))
        vtype = np.ones(nv, np.int64)
        vtype[slots] = 0
        cam_ids = slots
        pt_ids = np.flatnonzero(vtype == 1)
    else:
        vtype = np.concatenate([np.zeros(n_cams, np.int64), np.ones(n_pts, np.int64)])
        cam_ids = np.arange(n_cams)
        pt_ids = n_cams + np.arange(n_pts)
    obs_pt = pt_ids[obs_pt_l]
    obs_cam = cam_ids[obs_cam_l]
    if shuffle_edges:
        perm = rng.permutation(total)
        obs_pt, obs_cam, z, info = obs_pt[perm], obs_cam[perm], z[perm], info[perm]
    return BAGraph(vtype, cams, pts_n, obs_pt.astype(np.int64), obs_cam.astype(np.int64), z, info)


def add_outliers(g: BAGraph, fraction: float, seed: int):
    """A copy of `g` in which a seeded `fraction` of the measurements is replaced by pixels drawn uniformly from
    [0, 800)^2 (gross mismatches, as automatic feature matching leaves them), and the sorted edge indices replaced."""
    rng = np.random.default_rng(seed)
    n = len(g.obs_pt)
    idx = np.sort(rng.choice(n, int(round(fraction * n)), replace=False))
    z = np.array(g.z, np.float64, copy=True)
    z[idx] = rng.uniform(0.0, 800.0, (len(idx), 2))
    return BAGraph(g.vtype, g.cams, g.pts, g.obs_pt, g.obs_cam, z, g.info), idx


BA_SHAPES = {
    # name: (n_cams, n_pts, seed, kwargs)
    "venice871": (871, 530304, 871, dict(mean_extra_track=3.35, max_track=60, max_stride=11)),
    # max_stride 12: the reduced camera system has 2.4 % non-zero blocks (SURVEY 8(d): "locality window so that S fill is 1-3 %")
    "bal13682": (13682, 4456117, 13682, dict(mean_extra_track=4.5, max_track=120, max_stride=12, loops=3)),
    "mid": (100, 20000, 100, dict(mean_extra_track=3.0, max_track=30, max_stride=3)),
    # a long sequence with short tracks: the elimination tree of its reduced camera system branches (multi-GPU tests of
    # the block-sparse factorisation shared out by subtrees)
    "seq300": (300, 20000, 7, dict(mean_extra_track=2.0, max_track=8, max_stride=2, loops=1)),
    "small": (24, 1500, 24, dict(mean_extra_track=3.0, max_track=12, max_stride=2)),
    "tiny": (6, 40, 6, dict(mean_extra_track=2.0, max_track=5, max_stride=1)),
}


def ba_shape(name: str, **over) -> BAGraph:
    c, p, seed, kw = BA_SHAPES[name]
    kw = dict(kw)
    kw.update(over)
    return make_ba(c, p, seed, **kw)


def make_manhattan(n_poses: int = 3500, n_loops: int = 1954, seed: int = 3500,
                   sigma_t: float = 0.05, sigma_r: float = 0.02, fill_loops: bool = False) -> PoseGraph:
    """SE(2) Manhattan-world random walk: n_poses-1 odometry edges + (up to) n_loops loop closures between poses that
    revisit a grid cell. fill_loops: when the walk revisits too few cells, poses in ADJACENT cells (8-neighbourhood) close
    loops as well until n_loops is reached -- make_manhattan(fill_loops=True) is the BASELINE.json configs[0] shape,
    3500 poses and 3499 + 1954 = 5453 edges. (Off by default: the committed golden vectors were made from the graphs
    without it.)"""
    rng = np.random.default_rng(seed)
    gt = np.zeros((n_poses, 3))
    heading = 0
    for i in range(1, n_poses):
        if rng.random() < 0.25:
            heading += rng.choice([-1, 1])
        th = heading * np.pi / 2
        gt[i] = [gt[i - 1, 0] + np.cos(th), gt[i - 1, 1] + np.sin(th), np.arctan2(np.sin(th), np.cos(th))]

    def rel(a, b):
        c, s = np.cos(a[2]), np.sin(a[2])
        d = b[:2] - a[:2]
        dth = b[2] - a[2]
        return np.array([c * d[0] + s * d[1], -s * d[0] + c * d[1], np.arctan2(np.sin(dth), np.cos(dth))])

    e_from = list(range(n_poses - 1))
    e_to = list(range(1, n_poses))
    # loop closures between spatially close, temporally distant poses
    cand = []
    cells = {}
    for i in range(n_poses):
        key = (int(round(gt[i, 0])), int(round(gt[i, 1])))
        for j in cells.get(key, []):
            if i - j > 10:
                cand.append((j, i))
        cells.setdefault(key, []).append(i)
    if fill_loops and len(cand) < n_loops:
        near = []
        have = set(cand)
        seen = {}
        for i in range(n_poses):
            cx, cy = int(round(gt[i, 0])), int(round(gt[i, 1]))
            for dx in (-1, 0, 1):
                for dy in (-1, 0, 1):
                    for j in seen.get((cx + dx, cy + dy), []):
                        if i - j > 10 and (j, i) not in have:
                            near.append((j, i))
            seen.setdefault((cx, cy), []).append(i)
        if len(near) > n_loops - len(cand):
            near = [near[k] for k in np.sort(rng.choice(len(near), n_loops - len(cand), replace=False))]
        cand = sorted(cand + near, key=lambda ab: (ab[1], ab[0]))
    cand = np.array(cand) if cand else np.zeros((0, 2), np.int64)
    if len(cand) > n_loops:
        cand = cand[np.sort(rng.choice(len(cand), n_loops, replace=False))]
    # loop closures are appended in the order of their later pose, like an online run would see them
    for a, b in cand:
        e_from.append(int(b))
        e_to.append(int(a))
    e_from = np.array(e_from, np.int64)
    e_to = np.array(e_to, np.int64)
    z = np.stack([rel(gt[a], gt[b]) for a, b in zip(e_from, e_to)])
    z += rng.normal(0, 1, z.shape) * np.array([sigma_t, sigma_t, sigma_r])
    info = np.broadcast_to(np.diag([1 / sigma_t ** 2, 1 / sigma_t ** 2, 1 / sigma_r ** 2]), (len(z), 3, 3)).copy()
    # initial estimate = dead reckoning over the noisy odometry
    est = np.zeros_like(gt)
    for i in range(1, n_poses):
        a = est[i - 1]
        c, s = np.cos(a[2]), np.sin(a[2])
        d = z[i - 1]
        est[i] = [a[0] + c * d[0] - s * d[1], a[1] + s * d[0] + c * d[1], a[2] + d[2]]
        est[i, 2] = np.arctan2(np.sin(est[i, 2]), np.cos(est[i, 2]))
    return PoseGraph(GRAPH_SE2, est, e_from, e_to, z, info)


def make_sphere(n_rings: int = 50, n_per_ring: int = 50, seed: int = 2500, radius: float = 50.0,
                sigma_t: float = 0.05, sigma_r: float = 0.01) -> PoseGraph:
    """SE(3) sphere: rings of poses; odometry along the spiral + an edge to the pose one ring below."""
    rng = np.random.default_rng(seed)
    n = n_rings * n_per_ring
    Rs = np.empty((n, 3, 3))
    ts = np.empty((n, 3))
    for i in range(n):
        ring, k = divmod(i, n_per_ring)
        phi = np.pi * (ring + 1 + k / n_per_ring) / (n_rings + 2)
        lam = 2 * np.pi * k / n_per_ring
        p = radius * np.array([np.sin(phi) * np.cos(lam), np.sin(phi) * np.sin(lam), np.cos(phi)])
        zax = p / np.linalg.norm(p)
        xax = np.array([-np.sin(lam), np.cos(lam), 0.0])
        yax = np.cross(zax, xax)
        Rs[i] = np.stack([xax, yax, zax], 1)
        ts[i] = p
    e_from = list(range(n - 1))
    e_to = list(range(1, n))
    for i in range(n_per_ring, n):
        e_from.append(i - n_per_ring)
        e_to.append(i)
    e_from = np.array(e_from, np.int64)
    e_to = np.array(e_to, np.int64)
    Rrel = np.einsum("nji,njk->nik", Rs[e_from], Rs[e_to])
    trel = np.einsum("nji,nj->ni", Rs[e_from], ts[e_to] - ts[e_from])
    nR = _axis_angle_to_rotmat(rng.normal(0, sigma_r, (len(e_from), 3)))
    Rrel = np.einsum("nij,njk->nik", Rrel, nR)
    trel = trel + rng.normal(0, sigma_t, trel.shape)
    z = np.concatenate([trel, _rotmat_to_axis_angle(Rrel)], 1)
    info = np.broadcast_to(np.diag([1 / sigma_t ** 2] * 3 + [1 / sigma_r ** 2] * 3), (len(z), 6, 6)).copy()
    # dead-reckoning initial estimate over the spiral odometry
    Re = np.empty_like(Rs)
    te = np.empty_like(ts)
    Re[0], te[0] = Rs[0], ts[0]
    for i in range(1, n):
        te[i] = te[i - 1] + Re[i - 1] @ trel[i - 1]
        Re[i] = Re[i - 1] @ Rrel[i - 1]
    poses = np.concatenate([te, _rotmat_to_axis_angle(Re)], 1)
    return PoseGraph(GRAPH_SE3, poses, e_from, e_to, z, info)


def rcs_block_pattern(g: BAGraph):
    """Upper block structure (block CSC: col_ptr, row_idx, rows ascending, diagonal last) of the reduced camera system of
    a BA graph: cameras i <= j share a block when some landmark is seen by both (LinearSolver_Schur.h:1757-1767)."""
    vtype = np.asarray(g.vtype)
    cam_local = np.cumsum(vtype == 0) - 1
    n_cams = int((vtype == 0).sum())
    oc = cam_local[np.asarray(g.obs_cam, np.int64)]
    op = np.asarray(g.obs_pt, np.int64)
    order = np.argsort(op, kind="stable")
    oc, op = oc[order], op[order]
    _, start, k = np.unique(op, return_index=True, return_counts=True)
    j = np.arange(len(oc)) - np.repeat(start, k)
    kk = np.repeat(k, k)
    keys = [np.arange(n_cams, dtype=np.int64) * n_cams + np.arange(n_cams)]
    for dj in range(1, int(k.max()) if len(k) else 1):
        m = np.flatnonzero(j + dj < kk)
        a, b = oc[m], oc[m + dj]
        keys.append(np.unique(np.maximum(a, b) * n_cams + np.minimum(a, b)))  # key = col * C + row
    keys = np.unique(np.concatenate(keys))
    col, row = keys // n_cams, keys % n_cams
    col_ptr = np.zeros(n_cams + 1, np.uint64)
    np.add.at(col_ptr, col + 1, 1)
    return np.cumsum(col_ptr).astype(np.uint64), row.astype(np.uint64)


def pose_block_pattern(g: PoseGraph):
    """Upper block structure of lambda of a pose graph (one block per edge + the diagonal)."""
    n = len(g.poses)
    a, b = np.asarray(g.e_from, np.int64), np.asarray(g.e_to, np.int64)
    keys = np.unique(np.concatenate([np.arange(n, dtype=np.int64) * n + np.arange(n), np.maximum(a, b) * n + np.minimum(a, b)]))
    col, row = keys // n, keys % n
    col_ptr = np.zeros(n + 1, np.uint64)
    np.add.at(col_ptr, col + 1, 1)
    return np.cumsum(col_ptr).astype(np.uint64), row.astype(np.uint64)
