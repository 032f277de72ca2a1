"""numpy + scipy restatement of the point-cloud front end (catgrasp_b200/cloud.py, csrc/cg_cloud.cu).

Pinned parts: nearest / within-radius / hybrid neighbour queries are scipy's cKDTree itself (what the reference calls);
``depth2xyzmap``, ``cloudA_minus_cloudB`` and ``correct_pcd_normal_direction`` are checked against the reference's own
functions executed on tests/golden/cloud_frontend.npz.  Unpinned: voxel down-sampling and normal estimation restate
open3d's documented algorithms (open3d is not installed and the reference does not pin its version).
"""
import numpy as np
from scipy.spatial import cKDTree

INT_MAX = 2 ** 31 - 1


def depth2xyzmap(depth, K):
    """Utils.py:239-251."""
    invalid = depth < 0.1
    H, W = depth.shape[:2]
    vs, us = np.meshgrid(np.arange(0, H), np.arange(0, W), sparse=False, indexing="ij")
    zs = depth.reshape(-1)
    xs = (us.reshape(-1) - K[0, 2]) * zs / K[0, 0]
    ys = (vs.reshape(-1) - K[1, 2]) * zs / K[1, 1]
    xyz = np.stack((xs, ys, zs), 1).reshape(H, W, 3).astype(np.float32)
    xyz[invalid] = 0
    return xyz


def voxel_down_sample(pts, voxel, normals=None):
    """open3d VoxelDownSample: index floor((p - (min - voxel/2)) / voxel), per-voxel sums in input order (np.add.at)
    divided by the count; voxels in ascending index order (x, then y, then z).  Returns (points, normals or None)."""
    pts = np.asarray(pts, dtype=np.float64)
    if not voxel > 0:
        raise ValueError("voxel_size <= 0")
    if len(pts) == 0:
        return np.zeros((0, 3)), (None if normals is None else np.zeros((0, 3)))
    if not np.isfinite(pts).all():
        raise ValueError("non-finite points")
    vmin = pts.min(0) - voxel * 0.5
    vmax = pts.max(0) + voxel * 0.5
    if voxel * INT_MAX < (vmax - vmin).max():
        raise ValueError("voxel_size is too small")
    idx = np.floor((pts - vmin) / voxel).astype(np.int64)
    _, inv = np.unique(idx, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    M = inv.max() + 1
    cnt = np.bincount(inv, minlength=M).astype(np.float64)
    sp = np.zeros((M, 3))
    np.add.at(sp, inv, pts)
    out_n = None
    if normals is not None:
        sn = np.zeros((M, 3))
        np.add.at(sn, inv, np.asarray(normals, dtype=np.float64))
        out_n = sn / cnt[:, None]
    return sp / cnt[:, None], out_n


def voxel_members(pts, voxel):
    """(voxel id of every input point, number of voxels) in the oracle's output order."""
    pts = np.asarray(pts, dtype=np.float64)
    vmin = pts.min(0) - voxel * 0.5
    idx = np.floor((pts - vmin) / voxel).astype(np.int64)
    u, inv = np.unique(idx, axis=0, return_inverse=True)
    return inv.reshape(-1), len(u)


def nearest(pts, q):
    return cKDTree(pts).query(q)


def any_within(pts, q, r):
    """run_grasp_simulation.py:130-133: dists <= r of the nearest point."""
    if len(pts) == 0:
        return np.zeros(len(q), bool)
    d, _ = cKDTree(pts).query(q)
    return d <= r


def cloudA_minus_cloudB(ptsA, ptsB, thres):
    """Utils.py:482-488 (``n_jobs`` is ``workers`` in current scipy); keep ascending."""
    tree = cKDTree(ptsA)
    hits = tree.query_ball_point(ptsB, r=thres, workers=-1)
    remove = np.unique(np.concatenate([np.asarray(h, dtype=np.int64) for h in hits] + [np.zeros(0, np.int64)]))
    keep = np.setdiff1d(np.arange(len(ptsA)), remove)
    return ptsA[keep], keep


def correct_pcd_normal_direction(pts, normals, view_port=(0.0, 0.0, 0.0)):
    """Utils.py:205-213 on arrays."""
    view_dir = np.asarray(view_port, dtype=float).reshape(-1, 3) - pts
    view_dir = view_dir / np.linalg.norm(view_dir, axis=1).reshape(-1, 1)
    normals = normals / (np.linalg.norm(normals, axis=1) + 1e-10).reshape(-1, 1)
    dots = (view_dir * normals).sum(axis=1)
    normals = normals.copy()
    normals[dots < 0] = -normals[dots < 0]
    return normals


def hybrid_neighbors(tree, q, radius, max_nn):
    """cKDTree.query(k=max_nn, distance_upper_bound=radius): (dist, idx) padded with (inf, n)."""
    d, i = tree.query(q, k=max_nn, distance_upper_bound=radius)
    return d.reshape(len(q), max_nn), i.reshape(len(q), max_nn)


def normals_from_neighbors(pts, nbr, view_port=(0.0, 0.0, 0.0), centers=None):
    """open3d ComputeNormal (cumulant covariance, smallest-eigenvalue eigenvector, (0,0,1) below 3 neighbours) +
    correct_pcd_normal_direction.  nbr (Q, k) indices padded with len(pts).  Returns (normals, eigenvalues (Q,3))."""
    n_pts = len(pts)
    valid = nbr < n_pts
    cnt = valid.sum(1)
    P = np.where(valid[..., None], pts[np.minimum(nbr, n_pts - 1)], 0.0)
    c = np.stack([P[..., 0], P[..., 1], P[..., 2], P[..., 0] * P[..., 0], P[..., 0] * P[..., 1], P[..., 0] * P[..., 2],
                  P[..., 1] * P[..., 1], P[..., 1] * P[..., 2], P[..., 2] * P[..., 2]], -1).sum(1) / np.maximum(cnt, 1)[:, None]
    cov = np.empty((len(nbr), 3, 3))
    cov[:, 0, 0] = c[:, 3] - c[:, 0] * c[:, 0]
    cov[:, 1, 1] = c[:, 6] - c[:, 1] * c[:, 1]
    cov[:, 2, 2] = c[:, 8] - c[:, 2] * c[:, 2]
    cov[:, 0, 1] = cov[:, 1, 0] = c[:, 4] - c[:, 0] * c[:, 1]
    cov[:, 0, 2] = cov[:, 2, 0] = c[:, 5] - c[:, 0] * c[:, 2]
    cov[:, 1, 2] = cov[:, 2, 1] = c[:, 7] - c[:, 1] * c[:, 2]
    w, v = np.linalg.eigh(cov)
    n = v[:, :, 0].copy()
    n[cnt < 3] = [0.0, 0.0, 1.0]
    centers = pts[: len(nbr)] if centers is None else centers
    return correct_pcd_normal_direction(centers, n, view_port), w
