"""Point-cloud front end of the grasp stage on the GPU: the open3d / cKDTree calls that turn a depth scan into the
clouds the later stages take (run_grasp_simulation.py:113-139,171-175,198-211,245-251; Utils.py:205-213,239-251,482-488).

Inputs are numpy arrays or CUDA tensors; outputs are CUDA tensors (float64 geometry, like ``toOpen3dCloud``,
Utils.py:195).  There is no CPU fallback.

One difference from open3d: ``voxel_down_sample`` returns its voxels in ascending voxel-index order (x, then y,
then z).  open3d returns them in the iteration order of its hash map, which no other implementation reproduces.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib


def _ctx(device=None):
    ctx = _lib.Context.get(device)
    ctx.use_torch_stream()
    return ctx


def _points(x, dev, name="pts"):
    t = torch.as_tensor(x).to(device=dev, dtype=torch.float64)
    if t.ndim != 2 or t.shape[1] != 3:
        raise ValueError(f"{name} must be (N,3), got {tuple(t.shape)}")
    if t.shape[0] >= 2 ** 30:
        raise ValueError(f"{name}: at most 2^30 points")
    return t.contiguous()


def _device(x, device):
    if isinstance(device, torch.device):
        return device
    if device is not None:
        return torch.device("cuda", int(device))
    if isinstance(x, torch.Tensor) and x.is_cuda:
        return x.device
    return torch.device("cuda", torch.cuda.current_device())


def depth2xyzmap(depth, K):
    """Utils.py:239-251: (H,W) depth + 3x3 K -> (H,W,3) float32 map, zero where depth < 0.1.  The arithmetic is
    float64 like numpy's (int pixel grid minus float64 K entries, times the depth), rounded to float32 at the end:
    bit-identical to the reference."""
    dev = _device(depth, None)
    d = torch.as_tensor(depth).to(device=dev)
    if d.ndim != 2:
        raise ValueError(f"depth must be (H,W), got {tuple(d.shape)}")
    if not d.is_floating_point():
        d = d.to(torch.float64)
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    H, W = d.shape
    vs = torch.arange(H, device=dev, dtype=torch.float64)[:, None].expand(H, W)
    us = torch.arange(W, device=dev, dtype=torch.float64)[None, :].expand(H, W)
    zs = d.to(torch.float64)
    xs = (us - float(K[0, 2])) * zs / float(K[0, 0])
    ys = (vs - float(K[1, 2])) * zs / float(K[1, 1])
    xyz = torch.stack((xs, ys, zs), -1).to(torch.float32)
    xyz[d < 0.1] = 0
    return xyz


def voxel_down_sample(pts, voxel_size, normals=None, device=None):
    """open3d ``voxel_down_sample`` (run_grasp_simulation.py:114,137,173,246): the mean of every occupied voxel,
    summed in input order.  Returns (points (M,3), normals (M,3) or None) in ascending voxel-index order."""
    dev = _device(pts, device)
    p = _points(pts, dev)
    n = None if normals is None else _points(normals, dev, "normals")
    if n is not None and n.shape[0] != p.shape[0]:
        raise ValueError("normals must have one row per point")
    voxel = float(voxel_size)
    if not voxel > 0:
        raise ValueError("voxel_size must be positive")
    N = p.shape[0]
    out_p = torch.empty((N, 3), dtype=torch.float64, device=dev)
    out_n = None if n is None else torch.empty((N, 3), dtype=torch.float64, device=dev)
    count = torch.zeros((1,), dtype=torch.int32, device=dev)
    ctx = _ctx(dev.index)
    ctx.check(ctx.lib.cg_voxel_down_sample_dev(ctx.h, _lib.ptr(p), _lib.ptr(n), N, C.c_double(voxel), _lib.ptr(out_p),
                                               _lib.ptr(out_n), _lib.ptr(count)))
    M = int(count.item())
    return out_p[:M], (None if out_n is None else out_n[:M])


class CloudIndex:
    """(N,3) points resident on the GPU with an occupied-cell grid of edge ``cell`` (the query cost is lowest when the
    cell is near the query radius / the point spacing).  Replaces the cKDTree builds of the front end."""

    def __init__(self, pts, cell, device=None):
        dev = _device(pts, device)
        self.device = dev
        self.pts = _points(pts, dev)
        self.cell = float(cell)
        if not self.cell > 0:
            raise ValueError("cell must be positive")
        self.ctx = _ctx(dev.index)
        h = C.c_void_p()
        self.ctx.check(self.ctx.lib.cg_cloud_create_dev(self.ctx.h, _lib.ptr(self.pts), self.pts.shape[0],
                                                        C.c_double(self.cell), C.byref(h)))
        self.h = h

    def __len__(self):
        return self.pts.shape[0]

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.ctx.lib.cg_cloud_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def query(self, q):
        """cKDTree.query(q) with k=1: (dist (Q,) float64, idx (Q,) int64).  Ties go to the lower index; an empty
        index gives (inf, N)."""
        qt = _points(q, self.device, "q")
        Q = qt.shape[0]
        d = torch.empty((Q,), dtype=torch.float64, device=self.device)
        i = torch.empty((Q,), dtype=torch.int32, device=self.device)
        self.ctx.use_torch_stream()
        self.ctx.check(self.ctx.lib.cg_cloud_nearest_dev(self.h, _lib.ptr(qt), Q, _lib.ptr(d), _lib.ptr(i)))
        return d, i.to(torch.int64)

    def any_within(self, q, r):
        """(Q,) bool: some indexed point lies within distance <= r of q[i]."""
        qt = _points(q, self.device, "q")
        r = float(r)
        if not r >= 0:
            raise ValueError("r must be >= 0")
        Q = qt.shape[0]
        out = torch.empty((Q,), dtype=torch.uint8, device=self.device)
        self.ctx.use_torch_stream()
        self.ctx.check(self.ctx.lib.cg_cloud_any_within_dev(self.h, _lib.ptr(qt), Q, C.c_double(r), _lib.ptr(out)))
        return out.bool()

    def normals(self, radius, max_nn=30, view_port=(0.0, 0.0, 0.0), return_neighbors=False):
        """open3d estimate_normals(KDTreeSearchParamHybrid(radius, max_nn)) + correct_pcd_normal_direction(view_port)
        for the indexed points: (N,3) float64.  max_nn <= 32.  With ``return_neighbors`` also the (N, max_nn) int64
        neighbour indices in ascending distance, padded with N like cKDTree.query(k=max_nn, distance_upper_bound=radius)."""
        vp = (C.c_double * 3)(*[float(v) for v in np.asarray(view_port, dtype=np.float64).reshape(3)])
        out = torch.empty((len(self), 3), dtype=torch.float64, device=self.device)
        nbr = None
        if return_neighbors and 1 <= int(max_nn) <= 32:
            nbr = torch.empty((len(self), int(max_nn)), dtype=torch.int32, device=self.device)
        self.ctx.use_torch_stream()
        self.ctx.check(self.ctx.lib.cg_cloud_normals_dev(self.h, C.c_double(float(radius)), int(max_nn), vp, _lib.ptr(out),
                                                         _lib.ptr(nbr)))
        return (out, nbr.to(torch.int64)) if return_neighbors else out


def estimate_normals(pts, radius, max_nn=30, view_port=(0.0, 0.0, 0.0), device=None):
    """Normals of ``pts`` with the hybrid search (radius, max_nn), oriented toward ``view_port``
    (run_grasp_simulation.py:208-210, :247-249)."""
    return CloudIndex(pts, radius, device=device).normals(radius, max_nn, view_port)


def cloudA_minus_cloudB(ptsA, ptsB, thres, device=None):
    """Utils.py:482-488: the points of A farther than ``thres`` from every point of B -> (ptsA[keep], keep), keep
    ascending int64."""
    dev = _device(ptsA, device)
    a = _points(ptsA, dev, "ptsA")
    near = CloudIndex(ptsB, thres, device=dev).any_within(a, thres)
    keep = torch.nonzero(~near).reshape(-1)
    return a[keep], keep
