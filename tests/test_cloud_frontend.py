"""Point-cloud front end (catgrasp_b200/cloud.py, csrc/cg_cloud.cu).

CPU: the numpy/scipy restatement (tests/cloud_oracle.py) against values the reference's own Utils functions produced
(tests/golden/make_golden_cloud.py), and the voxel oracle's invariants.
GPU: every device primitive against the restatement / scipy at the sizes of the reference's pipeline."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.spatial import cKDTree

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cloud_oracle as ref   # noqa: E402

from catgrasp_b200 import synthetic   # noqa: E402


@pytest.fixture(scope="module")
def golden(golden_dir):
    return dict(np.load(os.path.join(golden_dir, "cloud_frontend.npz")))


def _minus_case(golden):
    """Inputs of the golden cloudA_minus_cloudB case (same recipe as make_golden_cloud.minus_case)."""
    rng = np.random.RandomState(7)
    xyz = golden["xyz_map"]
    A = xyz[xyz[:, :, 2] >= 0.1].reshape(-1, 3).astype(np.float64)
    c = A[rng.randint(len(A))]
    B = c + rng.normal(scale=0.01, size=(400, 3))
    return A, B, 0.005


def _normal_case():
    rng = np.random.RandomState(9)
    pts = rng.normal(scale=0.1, size=(500, 3)) + np.array([0, 0, 0.7])
    nrm = rng.normal(size=(500, 3))
    nrm[:20] = 0.0
    pts[20:25] = 0.0
    return pts, nrm, np.array([0.01, -0.02, 0.0])


# ---------------------------------------------------------------- CPU

def test_oracle_depth2xyzmap_equals_reference(golden):
    got = ref.depth2xyzmap(golden["depth"], golden["K"])
    assert got.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), golden["xyz_map"].view(np.uint32))


def test_oracle_cloudA_minus_cloudB_equals_reference(golden):
    A, B, thres = _minus_case(golden)
    kept, keep = ref.cloudA_minus_cloudB(A, B, thres)
    assert np.array_equal(keep, golden["minus_keep"])
    assert 0 < len(keep) < len(A)
    assert np.array_equal(kept, A[keep])


def test_oracle_normal_direction_equals_reference(golden):
    pts, nrm, vp = _normal_case()
    with np.errstate(invalid="ignore", divide="ignore"):
        n0 = ref.correct_pcd_normal_direction(pts, nrm)
        n1 = ref.correct_pcd_normal_direction(pts, nrm, vp)
    assert np.array_equal(n0, golden["normals_vp0"], equal_nan=True)
    assert np.array_equal(n1, golden["normals_vp"], equal_nan=True)


@pytest.mark.parametrize("voxel", [0.0005, 0.001, 0.002, 0.0071])
def test_voxel_oracle_invariants(voxel):
    rng = np.random.RandomState(3)
    pts = rng.uniform(-0.02, 0.02, size=(3000, 3)) + np.array([-0.3, 0.1, 0.7])
    pts[100:200] = pts[:100]                                          # duplicates
    nrm = rng.normal(size=pts.shape)
    out, out_n = ref.voxel_down_sample(pts, voxel, nrm)
    inv, M = ref.voxel_members(pts, voxel)
    assert len(out) == M and np.bincount(inv, minlength=M).sum() == len(pts)
    for v in rng.choice(M, size=min(M, 200), replace=False):
        m = inv == v
        assert np.allclose(out[v], pts[m].mean(0), rtol=0, atol=1e-15)
        assert np.allclose(out_n[v], nrm[m].mean(0), rtol=0, atol=1e-14)
    vmin = pts.min(0) - voxel * 0.5
    idx = np.floor((out - vmin) / voxel).astype(np.int64)             # every mean lies in its own voxel ...
    order = np.lexsort((idx[:, 2], idx[:, 1], idx[:, 0]))
    assert np.array_equal(order, np.arange(M))                        # ... and the voxels ascend (x, y, z)


def test_voxel_oracle_rejects_like_open3d():
    with pytest.raises(ValueError):
        ref.voxel_down_sample(np.zeros((2, 3)), 0.0)
    with pytest.raises(ValueError):
        ref.voxel_down_sample(np.array([[0.0, 0, 0], [1.0, 0, 0]]), 1e-12)


def test_make_depth_scene_shape_and_content():
    d = synthetic.make_depth_scene(120, 160, synthetic.REF_CAMERA_K * np.array([[1 / 13], [1 / 13], [1]]), seed=1)
    assert d.shape == (120, 160) and d.dtype == np.float32
    assert d.max() == np.float32(0.70) and d.min() < 0.69            # floor plus objects in front of it


# ---------------------------------------------------------------- GPU

def _cuda():
    import torch
    return torch


@pytest.fixture(scope="module")
def full_scene():
    """The reference camera's full 2064 x 1544 depth scene and its z >= 0.1 cloud (run_grasp_simulation.py:198-199)."""
    H, W = synthetic.REF_CAMERA_HW
    depth = synthetic.make_depth_scene(H, W, synthetic.REF_CAMERA_K, seed=0)
    xyz = ref.depth2xyzmap(depth, synthetic.REF_CAMERA_K)
    pts = xyz[xyz[:, :, 2] >= 0.1].reshape(-1, 3).astype(np.float64)
    return depth, xyz, pts


@pytest.fixture(scope="module")
def scene1mm(full_scene):
    """The 1 mm voxel scene (run_grasp_simulation.py:245-246)."""
    return ref.voxel_down_sample(full_scene[2], 0.001)[0]


def _object(pts, seed=0, radius=0.035):
    """Points above the floor within `radius` (xy) of a seeded above-floor point: one object crop."""
    rng = np.random.RandomState(seed)
    above = np.nonzero(pts[:, 2] < 0.699)[0]
    c = pts[above[rng.randint(len(above))]]
    m = (np.linalg.norm(pts[:, :2] - c[:2], axis=1) < radius) & (pts[:, 2] < 0.699)
    return pts[m]


def _nearest_lowest(pts, q, k=16):
    """cKDTree nearest with ties resolved to the lowest index (the device rule)."""
    d, i = cKDTree(pts).query(q, k=k)
    tie = d == d[:, :1]
    return d[:, 0], np.where(tie, i, np.iinfo(np.int64).max).min(1)


@pytest.mark.gpu
def test_depth2xyzmap_bit_identical(golden, full_scene):
    from catgrasp_b200 import cloud
    got = cloud.depth2xyzmap(golden["depth"], golden["K"]).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), golden["xyz_map"].view(np.uint32))
    depth, xyz, _ = full_scene
    got = cloud.depth2xyzmap(depth, synthetic.REF_CAMERA_K).cpu().numpy()
    assert got.shape == (1544, 2064, 3)
    assert np.array_equal(got.view(np.uint32), xyz.view(np.uint32))


def _voxel_cases(full_scene):
    _, _, pts = full_scene
    ob = _object(pts, 1)
    diam = np.linalg.norm(ob.max(0) - ob.min(0))
    rng = np.random.RandomState(4)
    nrm = rng.normal(size=ob.shape)
    yield "ob0.5mm", ob, nrm, 0.0005
    yield "ob1mm", ob, nrm, 0.001
    yield "ob2mm", ob, nrm, 0.002
    yield "ob_diam/10", ob, nrm, diam / 10.0
    yield "negative", ob - np.array([1.0, 1.0, 1.0]), nrm, 0.001
    yield "one_point", ob[:1], nrm[:1], 0.001
    yield "one_voxel", ob[:50] * 1e-3 + 0.3, nrm[:50], 0.01
    yield "scene1mm", pts, None, 0.001


@pytest.mark.gpu
def test_voxel_down_sample_bit_identical(full_scene):
    from catgrasp_b200 import cloud
    for name, p, n, voxel in _voxel_cases(full_scene):
        gp, gn = cloud.voxel_down_sample(p, voxel, normals=n)
        rp, rn = ref.voxel_down_sample(p, voxel, n)
        assert gp.shape == rp.shape, name
        assert np.array_equal(gp.cpu().numpy().view(np.uint64), rp.view(np.uint64)), name
        if n is not None:
            assert np.array_equal(gn.cpu().numpy().view(np.uint64), rn.view(np.uint64)), name
    gp, gn = cloud.voxel_down_sample(np.zeros((0, 3)), 0.001)
    assert gp.shape == (0, 3) and gn is None


@pytest.mark.gpu
def test_nearest_equals_scipy(full_scene):
    from catgrasp_b200 import cloud
    _, _, pts = full_scene
    ob = _object(pts, 2)
    ob = np.concatenate([ob, ob[::7]])                                # duplicated points
    rng = np.random.RandomState(5)
    q = np.concatenate([ob[rng.choice(len(ob), 3000)] + rng.normal(scale=0.0005, size=(3000, 3)),
                        ob[rng.choice(len(ob), 500)],                 # exact hits, several on duplicates
                        rng.normal(size=(200, 3)) * 5.0,              # far outside the cloud
                        ob.mean(0) + np.array([[10.0, 0, 0], [0, -30.0, 0], [0, 0, 100.0]])])
    for cell in (0.0005, 0.002):
        d, i = cloud.CloudIndex(ob, cell).query(q)
        d, i = d.cpu().numpy(), i.cpu().numpy()
        sd, si = cKDTree(ob).query(q)
        assert np.array_equal(d, sd)
        d2, _ = cKDTree(ob).query(q, k=2)
        unique = d2[:, 0] < d2[:, 1]
        assert (~unique).sum() > 0
        assert np.array_equal(i[unique], si[unique])
        ld, li = _nearest_lowest(ob, q)
        assert np.array_equal(i, li)
    d, i = cloud.CloudIndex(np.zeros((0, 3)), 0.001).query(q[:5])
    assert np.isinf(d.cpu().numpy()).all() and (i.cpu().numpy() == 0).all()


@pytest.mark.gpu
def test_any_within_crop_and_minus(full_scene, scene1mm, golden):
    from catgrasp_b200 import cloud
    _, _, pts = full_scene
    scene1 = scene1mm
    ob = _object(pts, 3)
    r = 0.085 / 2                                                     # gripper_diameter / 2
    for cell in (0.005, 0.02):
        got = cloud.CloudIndex(ob, cell).any_within(scene1, r).cpu().numpy()
        assert np.array_equal(got, ref.any_within(ob, scene1, r))
    bg = scene1[ref.any_within(ob, scene1, r)]
    kept, keep = cloud.cloudA_minus_cloudB(bg, ob, 0.005)
    rk, rkeep = ref.cloudA_minus_cloudB(bg, ob, 0.005)
    assert np.array_equal(keep.cpu().numpy(), rkeep) and 0 < len(rkeep) < len(bg)
    assert np.array_equal(kept.cpu().numpy(), rk)
    A, B, thres = _minus_case(golden)
    _, keep = cloud.cloudA_minus_cloudB(A, B, thres)
    assert np.array_equal(keep.cpu().numpy(), golden["minus_keep"])


@pytest.mark.gpu
def test_normals_full_scene(full_scene):
    from catgrasp_b200 import cloud
    _, _, pts = full_scene
    assert len(pts) == 2064 * 1544
    radius, K = 0.002, 30
    nrm, nbr = cloud.CloudIndex(pts, radius).normals(radius, K, return_neighbors=True)
    rng = np.random.RandomState(0)
    sel = rng.choice(len(pts), 20000, replace=False)
    nrm, nbr = nrm.cpu().numpy()[sel], nbr.cpu().numpy()[sel]
    tree = cKDTree(pts)
    sd, si = ref.hybrid_neighbors(tree, pts[sel], radius, K + 1)
    tie = np.isfinite(sd[:, K - 1]) & (sd[:, K - 1] == sd[:, K])      # k-th and (k+1)-th at the same distance
    same = np.array([set(a) == set(b) for a, b in zip(nbr, si[:, :K])])
    assert same[~tie].all(), int((~same & ~tie).sum())
    gd = np.sort(np.linalg.norm(pts[np.minimum(nbr, len(pts) - 1)] - pts[sel][:, None], axis=2)
                 + np.where(nbr == len(pts), np.inf, 0.0), 1)
    assert np.allclose(gd[tie], sd[tie, :K], rtol=0, atol=1e-15)      # at ties the distance multiset agrees
    # on a pixel grid most k-th neighbours tie with the (k+1)-th, so the directions are checked against the restated
    # estimate on the device's own neighbour set (verified just above: scipy's set, or an equal-distance choice at ties)
    rn, w = ref.normals_from_neighbors(pts, nbr, centers=pts[sel])
    good = w[:, 1] - w[:, 0] > 1e-3 * w[:, 2]
    assert good.mean() > 0.9
    a = nrm[good] / np.linalg.norm(nrm[good], axis=1)[:, None]          # both carry the 1/(|n| + 1e-10) scale
    b = rn[good] / np.linalg.norm(rn[good], axis=1)[:, None]
    ang = np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs((a * b).sum(1)))
    assert ang.max() < 1e-6, ang.max()
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1.0, atol=1e-9)
    view = -pts[sel] / np.linalg.norm(pts[sel], axis=1)[:, None]
    assert ((view * nrm).sum(1) >= 0).all()


@pytest.mark.gpu
def test_normals_sparse_points_fall_back_to_z():
    from catgrasp_b200 import cloud
    pts = np.array([[0.0, 0, 0.7], [0.0005, 0, 0.7], [0.1, 0, 0.7], [0.2, 0.2, -0.5], [0.2, 0.2005, -0.5]])
    n = cloud.estimate_normals(pts, 0.002, 30).cpu().numpy()
    want = ref.correct_pcd_normal_direction(pts, np.tile([0.0, 0, 1], (len(pts), 1)))
    assert np.array_equal(n, want)
    assert (n[:3, 2] < 0).all() and (n[3:, 2] > 0).all()              # flipped toward the camera


@pytest.mark.gpu
def test_object_chain_equals_oracle(full_scene, scene1mm):
    """run_grasp_simulation.py:113-139 + :171-175 on the device against the restated chain."""
    from catgrasp_b200 import cloud, my_cpp
    _, _, pts = full_scene
    scene1 = scene1mm
    ob = _object(pts, 4)
    ob_n = ref.correct_pcd_normal_direction(ob, np.random.RandomState(1).normal(size=ob.shape))
    # device
    down, _ = cloud.voxel_down_sample(ob, 0.0005)
    _, idx = cloud.CloudIndex(ob, 0.0005).query(down)
    idx = idx.cpu().numpy()
    ob_down, ob_n_down = ob[idx], ob_n[idx]
    near = cloud.CloudIndex(ob, 0.005).any_within(scene1, 0.085 / 2).cpu().numpy()
    bg, _ = cloud.cloudA_minus_cloudB(scene1[near], ob, 0.005)
    bg1, _ = cloud.voxel_down_sample(bg, 0.001)
    vs = np.linalg.norm(ob_down.max(0) - ob_down.min(0)) / 10.0
    sp, sn = cloud.voxel_down_sample(ob_down, vs, normals=ob_n_down)
    # restated chain
    rdown, _ = ref.voxel_down_sample(ob, 0.0005)
    _, ridx = _nearest_lowest(ob, rdown)
    rbg, _ = ref.cloudA_minus_cloudB(scene1[ref.any_within(ob, scene1, 0.085 / 2)], ob, 0.005)
    rbg1, _ = ref.voxel_down_sample(rbg, 0.001)
    rsp, rsn = ref.voxel_down_sample(ob[ridx], vs, ob_n[ridx])
    assert np.array_equal(idx, ridx)
    assert np.array_equal(bg1.cpu().numpy(), rbg1) and len(rbg1) > 100
    assert np.array_equal(sp.cpu().numpy(), rsp) and np.array_equal(sn.cpu().numpy(), rsn)
    occ = my_cpp.makeOccupancyGridFromCloudScan(bg1.cpu().numpy(), None, 0.001)
    rocc = my_cpp.makeOccupancyGridFromCloudScan(rbg1, None, 0.001)
    assert len(rocc) > 0 and np.array_equal(occ, rocc)


@pytest.mark.gpu
def test_error_codes_are_einval():
    torch = _cuda()
    from catgrasp_b200 import _lib, cloud
    ctx = _lib.Context.get()
    ctx.use_torch_stream()
    lib = ctx.lib
    dev = torch.device("cuda", ctx.device)
    p = torch.tensor([[0.0, 0, 0], [1.0, 0, 0]], dtype=torch.float64, device=dev)
    out = torch.empty((2, 3), dtype=torch.float64, device=dev)
    cnt = torch.empty((1,), dtype=torch.int32, device=dev)
    P = _lib.ptr

    def vox(pts, v):
        return lib.cg_voxel_down_sample_dev(ctx.h, P(pts), None, pts.shape[0], C.c_double(v), P(out), None, P(cnt))

    assert vox(p, 0.0) == _lib.CG_EINVAL
    assert vox(p, -1.0) == _lib.CG_EINVAL
    assert vox(p, 1e-12) == _lib.CG_EINVAL                          # index range beyond int32
    bad = p.clone()
    bad[1, 2] = float("nan")
    assert vox(bad, 0.001) == _lib.CG_EINVAL
    bad[1, 2] = float("inf")
    assert vox(bad, 0.001) == _lib.CG_EINVAL
    h = C.c_void_p()
    assert lib.cg_cloud_create_dev(ctx.h, P(bad), 2, C.c_double(0.001), C.byref(h)) == _lib.CG_EINVAL
    assert lib.cg_cloud_create_dev(ctx.h, P(p), 2, C.c_double(0.0), C.byref(h)) == _lib.CG_EINVAL
    assert lib.cg_cloud_create_dev(ctx.h, P(p), 2, C.c_double(1e-9), C.byref(h)) == _lib.CG_EINVAL   # > 2^21 cells
    idx = cloud.CloudIndex(p, 0.01)
    vp = (C.c_double * 3)(0.0, 0.0, 0.0)
    assert lib.cg_cloud_normals_dev(idx.h, C.c_double(0.01), 33, vp, P(out), None) == _lib.CG_EINVAL
    assert lib.cg_cloud_normals_dev(idx.h, C.c_double(0.0), 30, vp, P(out), None) == _lib.CG_EINVAL
    with pytest.raises(_lib.CgError):
        idx.normals(0.01, max_nn=33)
    with pytest.raises(_lib.CgError):
        cloud.voxel_down_sample(bad, 0.001)
    torch.cuda.synchronize()
    assert np.array_equal(cloud.voxel_down_sample(p, 0.5)[0].cpu().numpy(), ref.voxel_down_sample(p.cpu().numpy(), 0.5)[0])
