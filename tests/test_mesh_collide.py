"""The mesh-vs-voxel collision predicate (my_cpp.COLLISION_PREDICATE = "mesh", csrc/cg_mesh_collide.cu): its oracle
(oracle/mesh_voxel_ref.py) on the CPU, and the device filter bit for bit against that oracle (-m gpu)."""
import numpy as np
import pytest

from catgrasp_b200 import my_cpp
from catgrasp_b200.synthetic import _hexa_mesh, make_dense_gripper_proxy, make_filter_case, random_rotation
from oracle import fcl_semantic_ref, filter_ref
from oracle import mesh_voxel_ref as mv

EYE = np.eye(4)
RES = 0.0005


def _unshifted(p1, poses, sym, nocs_pose, c2n, g):
    none = np.zeros((0, 3))
    return filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], False, False, 0, g["open"], none,
                                 g["enclosed"], none)[2]


def _verdicts(case, f32_pose, octomap_keys):
    p1, p2, poses, sym, nocs_pose, c2n, g = case
    un = _unshifted(p1, poses, sym, nocs_pose, c2n, g)
    if octomap_keys:
        ko, ke = mv.occupied_voxel_keys(p1, RES), mv.occupied_voxel_keys(p2, RES)
        r = float(np.float32(RES))
    else:
        ko = np.unique(np.floor(p1 / RES).astype(np.int64), axis=0)
        ke = np.unique(np.floor(p2 / RES).astype(np.int64), axis=0)
        r = RES
    out = np.zeros(len(un), bool)
    for i, u in enumerate(un):
        gic = my_cpp._mm4_f32(u, g["gripper_in_grasp"]).astype(np.float64) if f32_pose else u.astype(np.float64) @ g["gripper_in_grasp"]
        out[i] = (mv.mesh_hits_voxels(g["open"]["V"], g["open"]["F"], gic, ko, r) or
                  mv.mesh_hits_voxels(g["enclosed"]["V"], g["enclosed"]["F"], gic, ke, r))
    return out


@pytest.fixture(scope="module")
def case_256_2():
    return make_filter_case(43, 256, 2)


def test_restatement_is_the_fcl_semantic(case_256_2):
    """With the old conventions (float64 pose, floor(x / res) keys) the new oracle gives fcl_semantic_ref's verdict on
    every pose: the restatement computes the same semantic."""
    p1, p2, poses, sym, nocs_pose, c2n, g = case_256_2
    un = _unshifted(p1, poses, sym, nocs_pose, c2n, g)
    ours = _verdicts(case_256_2, f32_pose=False, octomap_keys=False)
    sem = np.zeros(len(un), bool)
    for i, u in enumerate(un):
        gic = u.astype(np.float64) @ g["gripper_in_grasp"]
        sem[i] = (fcl_semantic_ref.mesh_hits_points(g["open"]["V"], g["open"]["F"], gic, p1, RES) or
                  fcl_semantic_ref.mesh_hits_points(g["enclosed"]["V"], g["enclosed"]["F"], gic, p2, RES))
    assert sem.any() and (~sem).any()
    assert np.array_equal(ours, sem)


def test_reference_conventions_change_few_verdicts(case_256_2):
    """float32 gripper_in_cam and octomap keys move the posed vertices by ~1e-7 m: count the verdicts that change."""
    old = _verdicts(case_256_2, f32_pose=False, octomap_keys=False)
    new = _verdicts(case_256_2, f32_pose=True, octomap_keys=True)
    changed = int((old != new).sum())
    print(f"reference conventions change {changed} of {len(old)} verdicts ({int(new.sum())} collisions)")
    assert changed <= len(old) // 100


@pytest.mark.parametrize("res", [0.0005, 0.001])
def test_octomap_key_form_equals_division(res):
    """floor(x * (1.0 / res)) == floor(x / res) on float32 values within 3 ulps of every voxel boundary of a wide key
    range, so choosing octomap's form documents the reference without changing results."""
    r = float(np.float32(res))
    k = np.arange(-32767, 32768, 7, dtype=np.float64)
    b = (k * r).astype(np.float32)
    xs = [b]
    up, dn = b.copy(), b.copy()
    for _ in range(3):
        up = np.nextafter(up, np.float32(np.inf))
        dn = np.nextafter(dn, np.float32(-np.inf))
        xs += [up, dn]
    x = np.concatenate(xs).astype(np.float64)
    assert np.array_equal(np.floor(x * (1.0 / r)), np.floor(x / r))
    pts = np.stack([x, x[::-1], np.roll(x, 5)], 1).astype(np.float32)
    keys = mv.occupied_voxel_keys(pts, res)
    ref = np.unique(np.floor(pts.astype(np.float64) / r).astype(np.int64), axis=0)
    ref = ref[((ref >= -32768) & (ref < 32768)).all(1)]
    assert np.array_equal(keys, ref)


def test_occupied_voxel_keys_range_and_errors():
    pts = np.array([[0.0, 0.0, 0.0], [0.0001, 0.0002, 0.0003], [40000 * RES, 0, 0], [-0.0101, 0.0201, 0.7001]], np.float32)
    keys = mv.occupied_voxel_keys(pts, RES)
    assert keys.tolist() == [[-21, 40, 1400], [0, 0, 0]]
    assert mv.occupied_voxel_keys(np.zeros((0, 3)), RES).shape == (0, 3)
    with pytest.raises(ValueError):
        mv.occupied_voxel_keys(np.array([[np.nan, 0, 0]]), RES)


def test_dense_gripper_proxy():
    d = make_dense_gripper_proxy()
    for k in ("open", "enclosed"):
        V, F = d[k]["V"], d[k]["F"]
        assert len(F) >= 20000 and F.max() < len(V)
        n = np.cross(V[F[:, 1]] - V[F[:, 0]], V[F[:, 2]] - V[F[:, 1]])
        n /= np.linalg.norm(n, axis=1, keepdims=True)
        assert (np.abs(n).max(1) < 0.99).sum() >= 1000          # the chamfers: faces off every axis
        assert np.abs(np.linalg.norm(np.cross(V[F[:, 1]] - V[F[:, 0]], V[F[:, 2]] - V[F[:, 0]]), axis=1)).min() > 0


def touch_fixture():
    """Axis-aligned box gripper whose faces lie exactly on voxel faces (all coordinates power-of-two multiples of
    float32(res), identity rotations), posed at 0 and one float32 ulp either side per axis."""
    r = float(np.float32(RES))
    s = 4 * r
    C = np.array([[0, 0, 0], [s, 0, 0], [s, s, 0], [0, s, 0], [0, 0, s], [s, 0, s], [s, s, s], [0, s, s]], np.float64)
    V, F = _hexa_mesh(C, 2)
    u = float(np.spacing(np.float32(s)))
    poses = []
    for tx in (-u, 0.0, u):
        for ty in (-u, 0.0, u):
            for tz in (-u, 0.0, u):
                T = np.eye(4)
                T[:3, 3] = [tx, ty, tz]
                poses.append(T)
    c = lambda k: (np.asarray(k, np.float64) + 0.5) * r      # noqa: E731  a point at a voxel centre
    open_pts = np.array([c([4, 4, 4])], np.float32)                          # corner touch: hit iff t >= 0
    bg_pts = np.array([c([-1, 2, 2]), c([1, 4, -1])], np.float32)            # face x = 0 / edge y = s, z = 0
    return (V.astype(np.float32), F), np.stack(poses), open_pts, bg_pts


def test_touch_fixture_has_exact_touches():
    (V, F), poses, open_pts, bg_pts = touch_fixture()
    r = float(np.float32(RES))
    keys = mv.occupied_voxel_keys(np.concatenate([open_pts, bg_pts]), RES)
    m = mv.sat_margins(V.astype(np.float64), F, poses[13], keys, r)          # pose 13: no shift
    assert (np.abs(m) <= 1e-12).sum() >= 10
    st, _, _ = mv.filter_mesh_ref(poses, [EYE], EYE, EYE, EYE, False, False, (V, F), open_pts, (V, F), bg_pts, RES)
    assert (st == 0).any() and (st == 3).any()


# ------------------------------------------------------------------------------------------------------ GPU
def _mesh(V, F):
    from catgrasp_b200.mesh import GripperMesh
    return GripperMesh(V, F)


@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a B200; there is no CPU fallback")
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _run_both(case, fdir, adjust, split, res=RES):
    import torch
    p1, p2, poses, sym, nocs_pose, c2n, g = case
    mo, me = _mesh(g["open"]["V"], g["open"]["F"]), _mesh(g["enclosed"]["V"], g["enclosed"]["F"])
    st, off, out = my_cpp.filter_grasp_pose_mesh_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mo, p1,
                                                     me, p2, res, split_status=split)
    dst, doff, dout = my_cpp.filter_grasp_pose_mesh_raw(torch.from_numpy(poses).cuda(), sym, nocs_pose, c2n,
                                                        g["gripper_in_grasp"], fdir, adjust, mo, torch.from_numpy(p1).cuda(),
                                                        me, torch.from_numpy(p2).cuda(), res, split_status=split)
    assert np.array_equal(dst.cpu().numpy(), st) and np.array_equal(doff.cpu().numpy(), off)
    assert np.array_equal(dout.cpu().numpy().view(np.uint32), out.view(np.uint32))
    return st, off, out


CASES = [(1, True, True, False), (1, False, True, True), (1, False, False, False), (1, True, False, False),
         (2, True, True, False), (2, False, True, False), (2, False, False, True), (2, True, False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("proxy", ["box", "dense"])
@pytest.mark.parametrize("S,adjust,fdir,split,scale", [c + ((1, 1, 1),) for c in CASES] + [(2, True, True, False, (1.0, 1.1, 0.9))])
def test_mesh_filter_bit_exact_vs_oracle(cuda, proxy, S, adjust, fdir, split, scale):
    p1, p2, poses, sym, nocs_pose, c2n, g = make_filter_case(43, 256, S, scale)
    if proxy == "dense":
        g = make_dense_gripper_proxy()
        rng = np.random.RandomState(7)
        poses = poses.copy()
        for i in range(len(poses)):                      # random extra rotation of every candidate about its own origin
            poses[i, :3, :3] = poses[i, :3, :3] @ random_rotation(rng)
    case = (p1.astype(np.float32), p2.astype(np.float32), poses, sym, nocs_pose, c2n, g)
    st, off, out = _run_both(case, fdir, adjust, split)
    rst, roff, rout = mv.filter_mesh_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust,
                                         (g["open"]["V"], g["open"]["F"]), p1, (g["enclosed"]["V"], g["enclosed"]["F"]), p2,
                                         RES, split=split)
    assert np.array_equal(st, rst)
    assert np.array_equal(off, roff)
    assert np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    assert (st == 0).any() and (st >= 3).any()


@pytest.mark.gpu
def test_mesh_filter_touch_fixture(cuda):
    (V, F), poses, open_pts, bg_pts = touch_fixture()
    g = {"open": {"V": V, "F": F}, "enclosed": {"V": V, "F": F}, "gripper_in_grasp": EYE}
    case = (open_pts, bg_pts, poses, EYE[None], EYE, EYE, g)
    for split in (False, True):
        st, off, out = _run_both(case, False, False, split)
        rst, roff, rout = mv.filter_mesh_ref(poses, [EYE], EYE, EYE, EYE, False, False, (V, F), open_pts, (V, F), bg_pts, RES,
                                             split=split)
        assert np.array_equal(st, rst) and np.array_equal(off, roff)
        assert np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    assert (st == 0).any() and (st == 3).any() and (st == 4).any()


@pytest.mark.gpu
def test_voxel_keys_on_device(cuda):
    import torch
    from catgrasp_b200.mesh import VoxelSet
    p1, p2 = make_filter_case(43, 4, 1)[:2]
    pts = np.concatenate([p1, p1[:50], p2, [[40000 * RES, 0.0, 0.0], [0.0, -40000 * RES, 0.1]]]).astype(np.float32)
    for res in (0.0005, 0.001):
        for src in (pts, torch.from_numpy(pts).cuda()):
            v = VoxelSet(src, res)
            assert np.array_equal(v.keys(), mv.occupied_voxel_keys(pts, res))
    assert len(VoxelSet(np.zeros((0, 3), np.float32), RES)) == 0 and VoxelSet(np.zeros((0, 3)), RES).keys().shape == (0, 3)
    assert len(VoxelSet(pts[-2:], RES)) == 0
    with pytest.raises(ValueError):
        VoxelSet(np.array([[0.0, np.inf, 0.0]], np.float32), RES)
    with pytest.raises(ValueError):
        VoxelSet(pts, 0.0)


@pytest.mark.gpu
def test_bad_input_is_rejected(cuda):
    import ctypes as C
    from catgrasp_b200 import _lib
    from catgrasp_b200.mesh import GripperMesh
    g = make_dense_gripper_proxy()
    V, F = g["open"]["V"], g["open"]["F"]
    with pytest.raises(ValueError):
        GripperMesh(V, np.zeros((0, 3), np.int32))
    with pytest.raises(ValueError):
        GripperMesh(V, np.array([[0, 1, len(V)]]))
    with pytest.raises(ValueError):
        GripperMesh(np.where(np.arange(len(V))[:, None] == 5, np.nan, V), F)
    ctx = _lib.Context.get()
    k = C.c_int()
    assert ctx.lib.cg_voxels_count(None, C.byref(k)) == _lib.CG_EINVAL
    assert ctx.lib.cg_voxels_keys_host(None, None) == _lib.CG_EINVAL
    prm = _lib.FilterParams()
    out = np.zeros(16, np.float32)
    assert ctx.lib.cg_filter_grasp_pose_mesh_dev(ctx.h, C.byref(prm), _lib.ptr(out), 1, _lib.ptr(out), 1, None, None, None,
                                                 None, _lib.ptr(out), _lib.ptr(out), _lib.ptr(out)) == _lib.CG_EINVAL
    with pytest.raises(ValueError):
        my_cpp.filter_grasp_pose_mesh_raw(EYE[None], EYE[None], EYE, EYE, EYE, False, False, GripperMesh(V, F),
                                          np.zeros((1, 3)), None, np.zeros((0, 3)), -1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("with_ik", [False, True])
def test_filterGraspPose_mesh_mode_without_sdf(cuda, capsys, monkeypatch, with_ik):
    """COLLISION_PREDICATE = "mesh" with no SDF registered: the oracle's survivors and the oracle's counter line."""
    p1, p2, poses, sym, nocs_pose, c2n, g = make_filter_case(43, 128, 2)
    poses = poses.copy()
    poses[::3, :3, 3] += poses[::3, :3, 0] * 0.02      # every third candidate 2 cm sideways: a finger lands in the object
    monkeypatch.setattr(my_cpp, "_SDF_REGISTRY", {})
    monkeypatch.setattr(my_cpp, "COLLISION_PREDICATE", "mesh")
    ik = (lambda ee, up, lo: bool(ee[0, 3] < 0.0)) if with_ik else None      # a stub solver: half of the space reachable
    monkeypatch.setattr(my_cpp, "_IK_SOLVER", ik)
    cam = np.eye(4)
    cam[:3, 3] = [0.01, -0.02, 0.0]
    args = (list(poses), list(sym), nocs_pose, c2n, cam, EYE, g["gripper_in_grasp"], True, with_ik, False, np.zeros(7),
            np.zeros(7), g["open"]["V"], g["open"]["F"], g["enclosed"]["V"], g["enclosed"]["F"], p1, p2, RES, True)
    capsys.readouterr()
    got = my_cpp.filterGraspPose(*args)
    line = capsys.readouterr().out.strip().splitlines()[-1]
    st, _, out = mv.filter_mesh_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, False,
                                    (g["open"]["V"], g["open"]["F"]), p1, (g["enclosed"]["V"], g["enclosed"]["F"]), p2, RES,
                                    split=True)
    ik_fail = np.zeros(len(st), bool)
    if with_ik:
        un = my_cpp.grasp_in_cam_unshifted(poses, sym, nocs_pose, c2n)
        for q in np.nonzero(st != 1)[0]:
            ik_fail[q] = not ik(my_cpp._mm4_f32(my_cpp._mm4_f32(cam.astype(np.float32), un[q]), np.eye(4, dtype=np.float32)),
                                None, None)
        assert ik_fail.any() and not ik_fail.all()
    keep = (st == 0) & ~ik_fail
    assert line == "n_approach_dir_rej={}, n_ik_rej={}, n_open_gripper_rej={}, n_close_gripper_rej={}".format(
        int((st == 1).sum()), int(ik_fail.sum()), int(((st == 3) & ~ik_fail).sum()), int(((st == 4) & ~ik_fail).sum()))
    assert (st == 3).any() and (st == 4).any()
    assert len(got) == int(keep.sum())
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(got, out[keep]))


@pytest.mark.gpu
def test_collision_manager_mesh_mode(cuda, monkeypatch):
    p1, p2, poses, sym, nocs_pose, c2n, g = make_filter_case(43, 64, 1)
    monkeypatch.setattr(my_cpp, "_SDF_REGISTRY", {})
    monkeypatch.setattr(my_cpp, "COLLISION_PREDICATE", "mesh")
    un = my_cpp.grasp_in_cam_unshifted(poses, sym, nocs_pose, c2n)
    cm = my_cpp.CollisionManager()
    assert cm.registerMesh(g["open"]["V"], g["open"]["F"]) == 0
    cloud = np.concatenate([p1, p2])
    cm.registerPointCloud(cloud, RES)
    got, want = [], []
    for q in range(0, 64, 4):
        T = my_cpp._mm4_f32(un[q], g["gripper_in_grasp"].astype(np.float32))
        cm.setTransform(T, 0)
        got.append(cm.isAnyCollision())
        st, _, _ = mv.filter_mesh_ref(T[None], [EYE], EYE, EYE, EYE, False, False, (g["open"]["V"], g["open"]["F"]), cloud,
                                      None, np.zeros((0, 3)), RES)
        want.append(bool(st[0] == 3))
    assert got == want and any(want) and not all(want)
