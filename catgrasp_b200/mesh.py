"""Device handles of the mesh-vs-voxel collision predicate (csrc/cg_mesh_collide.cu, the reference's registerMesh /
registerPointCloud, my_cpp/collision_manager.cpp:15-77)."""
import ctypes as C

import numpy as np
import torch

from . import _lib


def _check(ctx, rc):
    if rc == _lib.CG_EINVAL:
        msg = ctx.lib.cg_last_error(ctx.h)
        raise ValueError(msg.decode() if msg else "invalid argument")
    ctx.check(rc)


class GripperMesh:
    """A triangle mesh in the gripper frame with its triangle grid, resident on the device."""

    def __init__(self, vertices, faces, device=None, ctx=None):
        self.ctx = ctx or _lib.Context.get(device)
        V = np.ascontiguousarray(np.asarray(vertices, dtype=np.float64).astype(np.float32))
        F = np.ascontiguousarray(np.asarray(faces), dtype=np.int32)
        if V.ndim != 2 or V.shape[1] != 3 or F.ndim != 2 or F.shape[1] != 3:
            raise ValueError("GripperMesh: vertices and faces must be (N,3)")
        self.h = C.c_void_p()
        _check(self.ctx, self.ctx.lib.cg_mesh_create(self.ctx.h, _lib.ptr(V), V.shape[0], _lib.ptr(F), F.shape[0],
                                                     C.byref(self.h)))

    def info(self):
        """(dims (3,), cell edge in metres, number of (cell, triangle) entries)."""
        d, c, n = (C.c_int * 3)(), C.c_float(), C.c_int64()
        self.ctx.check(self.ctx.lib.cg_mesh_info(self.h, d, C.byref(c), C.byref(n)))
        return tuple(d), c.value, n.value

    def __del__(self):
        if getattr(self, "h", None) and self.h.value:
            self.ctx.lib.cg_mesh_destroy(self.h)
            self.h = None


class VoxelSet:
    """The occupied octree voxels of a point set at one resolution (float32 points, host array or CUDA tensor)."""

    def __init__(self, points, resolution, device=None, ctx=None):
        if isinstance(points, torch.Tensor) and points.is_cuda:
            device = points.device.index if device is None else device
        self.ctx = ctx or _lib.Context.get(device)
        dev = torch.device("cuda", self.ctx.device)
        p = torch.as_tensor(points).to(device=dev, dtype=torch.float32).contiguous()
        if p.numel() and (p.ndim != 2 or p.shape[1] != 3):
            raise ValueError(f"VoxelSet: points must be (N,3), got {tuple(p.shape)}")
        p = p.reshape(-1, 3)
        self.resolution = float(np.float32(resolution))
        self.h = C.c_void_p()
        self.ctx.use_torch_stream()
        _check(self.ctx, self.ctx.lib.cg_voxels_create_dev(self.ctx.h, _lib.ptr(p) if p.shape[0] else None, p.shape[0],
                                                           C.c_float(self.resolution), C.byref(self.h)))

    def __len__(self):
        k = C.c_int()
        self.ctx.check(self.ctx.lib.cg_voxels_count(self.h, C.byref(k)))
        return k.value

    def keys(self):
        """(K,3) int32 octomap keys, ascending in (x, y, z)."""
        out = np.zeros((len(self), 3), np.int32)
        self.ctx.check(self.ctx.lib.cg_voxels_keys_host(self.h, _lib.ptr(out)))
        return out

    def __del__(self):
        if getattr(self, "h", None) and self.h.value:
            self.ctx.lib.cg_voxels_destroy(self.h)
            self.h = None
