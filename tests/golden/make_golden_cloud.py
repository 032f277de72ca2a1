"""Golden vectors for the point-cloud front end, produced by EXECUTING THE REFERENCE's Utils.depth2xyzmap
(:239-251), Utils.cloudA_minus_cloudB (:482-488) and Utils.correct_pcd_normal_direction (:205-213).

Run in the authoring container only (needs /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_cloud.py

Import-only stubs: trimesh and transformations (absent; nothing on these paths calls them).  One stand-in computes:
``open3d`` (absent) is a numpy point cloud whose ``points`` / ``normals`` are float64 arrays, which is all that
correct_pcd_normal_direction reads and writes.  One shim: cloudA_minus_cloudB passes ``n_jobs=-1`` to
cKDTree.query_ball_point, a keyword current scipy renamed to ``workers``; the shim forwards it under the new name
and changes nothing else.
"""
import os
import sys
import types

import numpy as np
from scipy.spatial import cKDTree

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, "/root/reference")


class _Stub(types.ModuleType):
    __all__ = []
    __path__ = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return type(name, (), {})


for _m in ["trimesh", "transformations"]:
    sys.modules[_m] = _Stub(_m)


class _PointCloud:
    def __init__(self):
        self.points = np.zeros((0, 3))
        self.normals = np.zeros((0, 3))


_o3d = types.ModuleType("open3d")
_o3d.geometry = types.SimpleNamespace(PointCloud=_PointCloud)
_o3d.utility = types.SimpleNamespace(Vector3dVector=lambda a: np.array(a, dtype=np.float64))
sys.modules["open3d"] = _o3d

import Utils as ref_utils   # noqa: E402  the reference itself


class _KDTreeNJobs(cKDTree):
    def query_ball_point(self, x, r, n_jobs=None, **kw):
        if n_jobs is not None:
            kw["workers"] = n_jobs
        return super().query_ball_point(x, r, **kw)


ref_utils.cKDTree = _KDTreeNJobs

from catgrasp_b200 import synthetic   # noqa: E402

DEPTH_HW = (96, 128)


def depth_case():
    """A small scene with the reference camera's focal lengths, plus invalid pixels (0 and < 0.1 m)."""
    H, W = DEPTH_HW
    K = synthetic.REF_CAMERA_K.copy()
    K[0, 2], K[1, 2] = W / 2 - 0.5, H / 2 + 0.25
    K[0, 0] /= 16
    K[1, 1] /= 16
    depth = synthetic.make_depth_scene(H, W, K, seed=11)
    rng = np.random.RandomState(5)
    depth[rng.rand(H, W) < 0.03] = 0.0
    depth[rng.rand(H, W) < 0.01] = np.float32(0.0999)
    return depth, K


def minus_case():
    rng = np.random.RandomState(7)
    depth, K = depth_case()
    xyz = ref_utils.depth2xyzmap(depth, K)
    A = xyz[xyz[:, :, 2] >= 0.1].reshape(-1, 3).astype(np.float64)
    c = A[rng.randint(len(A))]
    B = c + rng.normal(scale=0.01, size=(400, 3))
    return A, B, 0.005


def normal_case():
    rng = np.random.RandomState(9)
    pts = rng.normal(scale=0.1, size=(500, 3)) + np.array([0, 0, 0.7])
    nrm = rng.normal(size=(500, 3))
    nrm[:20] = 0.0                           # zero-length normals
    pts[20:25] = 0.0                         # points at the view port
    vp = np.array([0.01, -0.02, 0.0])
    return pts, nrm, vp


def main():
    depth, K = depth_case()
    xyz = ref_utils.depth2xyzmap(depth, K)
    A, B, thres = minus_case()
    _, keep = ref_utils.cloudA_minus_cloudB(A, B, thres=thres)
    pts, nrm, vp = normal_case()
    pcd = _PointCloud()
    pcd.points, pcd.normals = pts.copy(), nrm.copy()
    n0 = ref_utils.correct_pcd_normal_direction(pcd).normals
    pcd = _PointCloud()
    pcd.points, pcd.normals = pts.copy(), nrm.copy()
    n1 = ref_utils.correct_pcd_normal_direction(pcd, view_port=vp).normals
    np.savez_compressed(os.path.join(HERE, "cloud_frontend.npz"), depth=depth, K=K, xyz_map=xyz,
                        minus_keep=np.sort(np.asarray(keep, np.int64)), normals_vp0=np.asarray(n0),
                        normals_vp=np.asarray(n1))
    print("cloud golden:", xyz.shape, "keep", len(keep), "of", len(A))


if __name__ == "__main__":
    main()
