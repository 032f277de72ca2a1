"""Drop-in for the reference's pybind module ``my_cpp`` (my_cpp/pybind.cpp:11-23).

``filterGraspPose`` keeps the reference's 20 positional arguments
(my_cpp/common.h:60) and returns the surviving grasp_in_cam matrices as a list
of (4,4) float32 arrays.  Differences, all documented in INTEGRATION.md:

* default geometry predicate = gripper SDF vs scene points (sdf.py:292-389)
  instead of FCL mesh-vs-octree; the SDFs of the two gripper meshes must be
  registered once with :func:`register_gripper_sdf` (the reference loads the
  same grids from ``gripper*.sdf``, dexnet/grasping/gripper.py:120-129).
  ``COLLISION_PREDICATE = "mesh"`` evaluates the reference's own mesh-vs-voxel
  test from the meshes alone, with no SDF;
* survivors come back in deterministic (pose, symmetry) order, not in OpenMP
  thread-arrival order (common.cpp:303-313);
* ``filter_ik=True`` needs a host IK predicate registered with
  :func:`set_ik_solver` (the generated ikfast solver stays on the CPU).
"""
import ctypes as C
import hashlib

import numpy as np
import torch

from . import _lib

_SDF_REGISTRY = {}
_MESH_REGISTRY = {}
_IK_SOLVER = None
DEFAULT_SDF_MODE = _lib.CG_SDF_TRILINEAR
# Which geometry predicate filterGraspPose uses for "the posed gripper touches a scene point":
#   "sdf"   -- the point lies inside the gripper solid (sd < 0): the predicate of meshpy's Sdf3D.is_any_points_inside;
#   "voxel" -- sd < octo_resolution * sqrt(3) / 2: conservative stand-in for the reference's FCL mesh-vs-octomap test
#              (collision_manager.cpp:93-111), where a point occupies a whole voxel cube of side octo_resolution -- every
#              cube that can touch the gripper surface has its generating point within half a cube diagonal of it.
#   "mesh"  -- the reference's own test: the posed gripper mesh touches an occupied voxel cube of side octo_resolution
#              (collision_manager.cpp:15-111, restated in oracle/mesh_voxel_ref.py); needs no SDF.
# Measured agreement with a restatement of the mesh-vs-voxel semantic: DESIGN.md, X2.
COLLISION_PREDICATE = "sdf"


def voxel_margin(octo_resolution):
    return float(np.float32(octo_resolution) * np.float32(np.sqrt(3.0) / 2.0))



def _digest(vertices, faces):
    h = hashlib.sha1()
    h.update(np.ascontiguousarray(vertices, dtype=np.float32).tobytes())
    h.update(np.ascontiguousarray(faces, dtype=np.int32).tobytes())
    return h.hexdigest()


def register_gripper_sdf(vertices, faces, sdf):
    """Associate a gripper mesh (as passed to filterGraspPose) with its Sdf3D."""
    _SDF_REGISTRY[_digest(vertices, faces)] = sdf


def set_ik_solver(fn):
    """fn(ee_in_base (4,4) float32, upper, lower) -> bool (True = some IK solution within limits)."""
    global _IK_SOLVER
    _IK_SOLVER = fn


def _sdf_for(vertices, faces):
    key = _digest(vertices, faces)
    if key not in _SDF_REGISTRY:
        raise _lib.CgError("no SDF registered for this gripper mesh: call "
                           "catgrasp_b200.my_cpp.register_gripper_sdf(vertices, faces, Sdf3D) first")
    return _SDF_REGISTRY[key]


def _mesh_for(vertices, faces):
    key = _digest(vertices, faces)
    if key not in _MESH_REGISTRY:
        from .mesh import GripperMesh
        _MESH_REGISTRY[key] = GripperMesh(vertices, faces)
    return _MESH_REGISTRY[key]


def _m16(m):
    a = np.ascontiguousarray(np.asarray(m, dtype=np.float64).astype(np.float32)).reshape(16)
    return (C.c_float * 16)(*[float(v) for v in a])


def filter_grasp_pose_raw(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs, gripper_in_grasp,
                          filter_approach_dir_face_camera, adjust_collision_pose, sdf_open, open_pts,
                          sdf_enclosed, enclosed_pts, sdf_mode=None, device_out=False, sdf_margin=0.0, split_status=False):
    """Array-level entry: returns (status (Q,) u8, offset (Q,) i8, poses (Q,4,4) f32) with Q = G*S.
    ``split_status`` (only meaningful without pose adjustment): CG_ST_REJ_COLL = open gripper vs object points,
    CG_ST_REJ_COLL_ENCL = enclosed gripper vs background (the reference's two verbose counters)."""
    ctx = sdf_open.ctx
    prm = _lib.FilterParams()
    prm.nocs_pose = _m16(nocs_pose)
    prm.canonical_to_nocs = _m16(canonical_to_nocs)
    prm.gripper_in_grasp = _m16(gripper_in_grasp)
    prm.filter_approach_dir_face_camera = int(bool(filter_approach_dir_face_camera))
    prm.adjust_collision_pose = int(bool(adjust_collision_pose))
    prm.sdf_mode = DEFAULT_SDF_MODE if sdf_mode is None else int(sdf_mode)
    prm.sdf_margin = float(sdf_margin)
    prm.split_coll_status = int(bool(split_status))
    if isinstance(grasp_poses, torch.Tensor) and grasp_poses.is_cuda:
        dev = grasp_poses.device
        gp = grasp_poses.to(torch.float32).contiguous().reshape(-1, 16)
        st = torch.as_tensor(np.asarray(symmetry_tfs)).to(device=dev, dtype=torch.float32).contiguous().reshape(-1, 16)
        p1 = torch.as_tensor(open_pts).to(device=dev, dtype=torch.float32).contiguous().reshape(-1, 3)
        p2 = torch.as_tensor(enclosed_pts).to(device=dev, dtype=torch.float32).contiguous().reshape(-1, 3)
        G, S = gp.shape[0], st.shape[0]
        Q = G * S
        status = torch.empty((Q,), dtype=torch.uint8, device=dev)
        offset = torch.empty((Q,), dtype=torch.int8, device=dev)
        poses = torch.empty((Q, 4, 4), dtype=torch.float32, device=dev)
        ctx.use_torch_stream()
        ctx.check(ctx.lib.cg_filter_grasp_pose_dev(
            ctx.h, C.byref(prm), _lib.ptr(gp), G, _lib.ptr(st), S, sdf_open.h, _lib.ptr(p1), p1.shape[0],
            sdf_enclosed.h if sdf_enclosed is not None else None, _lib.ptr(p2), p2.shape[0],
            _lib.ptr(status), _lib.ptr(offset), _lib.ptr(poses)))
        return status, offset, poses
    gp = np.ascontiguousarray(np.asarray(grasp_poses, dtype=np.float64).astype(np.float32)).reshape(-1, 16)
    st = np.ascontiguousarray(np.asarray(symmetry_tfs, dtype=np.float64).astype(np.float32)).reshape(-1, 16)
    p1 = np.ascontiguousarray(np.asarray(open_pts, dtype=np.float64).astype(np.float32)).reshape(-1, 3)
    p2 = np.ascontiguousarray(np.asarray(enclosed_pts, dtype=np.float64).astype(np.float32)).reshape(-1, 3)
    G, S = gp.shape[0], st.shape[0]
    Q = G * S
    status = np.empty((Q,), np.uint8)
    offset = np.empty((Q,), np.int8)
    poses = np.empty((Q, 4, 4), np.float32)
    ctx.use_own_stream()   # blocking host call
    ctx.check(ctx.lib.cg_filter_grasp_pose_host(
        ctx.h, C.byref(prm), _lib.ptr(gp), G, _lib.ptr(st), S, sdf_open.h, _lib.ptr(p1), p1.shape[0],
        sdf_enclosed.h if sdf_enclosed is not None else None, _lib.ptr(p2), p2.shape[0],
        _lib.ptr(status), _lib.ptr(offset), _lib.ptr(poses)))
    return status, offset, poses


def filter_grasp_pose_mesh_raw(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs, gripper_in_grasp,
                               filter_approach_dir_face_camera, adjust_collision_pose, mesh_open, open_pts, mesh_enclosed,
                               enclosed_pts, octo_resolution, split_status=False):
    """filter_grasp_pose_raw with the mesh-vs-voxel predicate: mesh_* are catgrasp_b200.mesh.GripperMesh handles;
    open_pts / enclosed_pts are (N,3) points (host arrays or CUDA tensors) or ready catgrasp_b200.mesh.VoxelSet handles
    at octo_resolution.  CUDA-tensor poses return device tensors, host poses host arrays."""
    from .mesh import VoxelSet, _check
    ctx = mesh_open.ctx
    prm = _lib.FilterParams()
    prm.nocs_pose = _m16(nocs_pose)
    prm.canonical_to_nocs = _m16(canonical_to_nocs)
    prm.gripper_in_grasp = _m16(gripper_in_grasp)
    prm.filter_approach_dir_face_camera = int(bool(filter_approach_dir_face_camera))
    prm.adjust_collision_pose = int(bool(adjust_collision_pose))
    prm.split_coll_status = int(bool(split_status))
    enc = mesh_enclosed.h if mesh_enclosed is not None else None
    on_device = isinstance(grasp_poses, torch.Tensor) and grasp_poses.is_cuda
    if on_device or isinstance(open_pts, VoxelSet) or isinstance(enclosed_pts, VoxelSet):
        dev = torch.device("cuda", ctx.device)
        gp = torch.as_tensor(np.asarray(grasp_poses) if not isinstance(grasp_poses, torch.Tensor) else grasp_poses)
        gp = gp.to(device=dev, dtype=torch.float32).contiguous().reshape(-1, 16)
        st = torch.as_tensor(np.asarray(symmetry_tfs)).to(device=dev, dtype=torch.float32).contiguous().reshape(-1, 16)
        vo = open_pts if isinstance(open_pts, VoxelSet) else VoxelSet(open_pts, octo_resolution, ctx=ctx)
        ve = enclosed_pts if isinstance(enclosed_pts, VoxelSet) else VoxelSet(enclosed_pts, octo_resolution, ctx=ctx)
        G, S = gp.shape[0], st.shape[0]
        Q = G * S
        status = torch.empty((Q,), dtype=torch.uint8, device=dev)
        offset = torch.empty((Q,), dtype=torch.int8, device=dev)
        poses = torch.empty((Q, 4, 4), dtype=torch.float32, device=dev)
        ctx.use_torch_stream()
        _check(ctx, ctx.lib.cg_filter_grasp_pose_mesh_dev(
            ctx.h, C.byref(prm), _lib.ptr(gp), G, _lib.ptr(st), S, mesh_open.h, vo.h, enc, ve.h,
            _lib.ptr(status), _lib.ptr(offset), _lib.ptr(poses)))
        if on_device:
            return status, offset, poses
        return status.cpu().numpy(), offset.cpu().numpy(), poses.cpu().numpy()
    gp = np.ascontiguousarray(np.asarray(grasp_poses, dtype=np.float64).astype(np.float32)).reshape(-1, 16)
    st = np.ascontiguousarray(np.asarray(symmetry_tfs, dtype=np.float64).astype(np.float32)).reshape(-1, 16)
    p1 = np.ascontiguousarray(np.asarray(open_pts, dtype=np.float64).astype(np.float32)).reshape(-1, 3)
    p2 = np.ascontiguousarray(np.asarray(enclosed_pts, dtype=np.float64).astype(np.float32)).reshape(-1, 3)
    G, S = gp.shape[0], st.shape[0]
    Q = G * S
    status = np.empty((Q,), np.uint8)
    offset = np.empty((Q,), np.int8)
    poses = np.empty((Q, 4, 4), np.float32)
    ctx.use_own_stream()   # blocking host call
    _check(ctx, ctx.lib.cg_filter_grasp_pose_mesh_host(
        ctx.h, C.byref(prm), _lib.ptr(gp), G, _lib.ptr(st), S, mesh_open.h, _lib.ptr(p1), p1.shape[0], enc,
        _lib.ptr(p2), p2.shape[0], C.c_float(float(np.float32(octo_resolution))),
        _lib.ptr(status), _lib.ptr(offset), _lib.ptr(poses)))
    return status, offset, poses


def _mm4_f32(A, B):
    """(...,4,4) x (...,4,4) in float32 with the accumulation order of the reference build's Eigen fixed-size product
    (sum over k = 0..3, one rounding per multiply and per add; my_cpp is built without FMA, CMakeLists.txt:5-6) --
    the same order as the CUDA kernel (csrc/cg_collide.cu) and oracle/filter_ref.c."""
    A = np.asarray(A, np.float32)
    B = np.asarray(B, np.float32)
    out = (A[..., :, 0:1] * B[..., 0:1, :]).astype(np.float32)
    for k in (1, 2, 3):
        out = (out + (A[..., :, k:k + 1] * B[..., k:k + 1, :]).astype(np.float32)).astype(np.float32)
    return out


def grasp_in_cam_unshifted(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs_transform):
    """common.cpp:159,190-197 on the host, bit-identical to the kernel: canonical_to_cam * (tf_j * pose_i) with the
    first three columns normalised, for every (i, j) -> (G*S, 4, 4) float32.  This is the pose the reference hands to
    the approach-direction and IK tests (:199-226), before any lateral offset."""
    f = lambda m: np.asarray(m, np.float64).astype(np.float32)      # noqa: E731  pybind narrows float64 -> float32
    gp = f(grasp_poses).reshape(-1, 1, 4, 4)
    st = f(symmetry_tfs).reshape(1, -1, 4, 4)
    c2c = _mm4_f32(f(nocs_pose), f(canonical_to_nocs_transform))
    g = _mm4_f32(c2c, _mm4_f32(st, gp)).reshape(-1, 4, 4)
    x, y, z = g[:, 0, :3], g[:, 1, :3], g[:, 2, :3]
    n = np.sqrt(((x * x).astype(np.float32) + (y * y).astype(np.float32)).astype(np.float32) + (z * z).astype(np.float32))
    g[:, :3, :3] = (g[:, :3, :3] / n[:, None, :]).astype(np.float32)
    return g


def filterGraspPose(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs_transform, cam_in_world, ee_in_grasp,
                    gripper_in_grasp, filter_approach_dir_face_camera, filter_ik, adjust_collision_pose, upper, lower,
                    gripper_vertices, gripper_faces, gripper_enclosed_vertices, gripper_enclosed_faces,
                    gripper_collision_pts, gripper_enclosed_collision_pts, octo_resolution, verbose):
    """my_cpp/common.cpp:156-321 (signature common.h:60).  Returns list[(4,4) float32]."""
    if len(grasp_poses) == 0 or len(symmetry_tfs) == 0:
        return []
    for name, a in (("gripper_collision_pts", gripper_collision_pts),
                    ("gripper_enclosed_collision_pts", gripper_enclosed_collision_pts)):
        a = np.asarray(a)
        if a.size and (a.ndim != 2 or a.shape[1] != 3):   # collision_manager.cpp:57-61 (reference exits)
            raise ValueError(f"{name} must be (N,3), got {a.shape}")
    if COLLISION_PREDICATE == "mesh":
        mesh_open = _mesh_for(gripper_vertices, gripper_faces)
        mesh_encl = _mesh_for(gripper_enclosed_vertices, gripper_enclosed_faces)
    else:
        sdf_open = _sdf_for(gripper_vertices, gripper_faces)
        sdf_encl = _sdf_for(gripper_enclosed_vertices, gripper_enclosed_faces)
    if filter_ik and _IK_SOLVER is None:
        raise NotImplementedError("filter_ik=True requires catgrasp_b200.my_cpp.set_ik_solver(fn); "
                                  "the generated ikfast solver is a host stage (INTEGRATION.md)")
    if COLLISION_PREDICATE == "mesh":
        status, offset, poses = filter_grasp_pose_mesh_raw(
            grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs_transform, gripper_in_grasp,
            filter_approach_dir_face_camera, adjust_collision_pose, mesh_open,
            np.asarray(gripper_collision_pts).reshape(-1, 3), mesh_encl,
            np.asarray(gripper_enclosed_collision_pts).reshape(-1, 3), octo_resolution, split_status=bool(verbose))
    else:
        status, offset, poses = filter_grasp_pose_raw(
            grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs_transform, gripper_in_grasp,
            filter_approach_dir_face_camera, adjust_collision_pose, sdf_open,
            np.asarray(gripper_collision_pts).reshape(-1, 3), sdf_encl,
            np.asarray(gripper_enclosed_collision_pts).reshape(-1, 3),
            sdf_margin=voxel_margin(octo_resolution) if COLLISION_PREDICATE == "voxel" else 0.0, split_status=bool(verbose))
    keep = status == _lib.CG_ST_ACCEPT
    ik_fail = np.zeros(status.shape[0], bool)
    if filter_ik:
        # common.cpp:214-226: IK is evaluated on the UN-shifted grasp_in_cam, after the approach test and before the
        # collision tests.  The rejections are independent, so running IK on the collision survivors only keeps the
        # same set; verbose mode evaluates it wherever the reference does, so that its counters come out the same.
        cam = np.asarray(cam_in_world, np.float64).astype(np.float32)
        eeg = np.asarray(ee_in_grasp, np.float64).astype(np.float32)
        unshifted = grasp_in_cam_unshifted(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs_transform)
        todo = np.nonzero(status != _lib.CG_ST_REJ_DIR)[0] if verbose else np.nonzero(keep)[0]
        for q in todo:
            ee_in_base = _mm4_f32(_mm4_f32(cam, unshifted[q]), eeg)      # common.cpp:216, left to right
            if not _IK_SOLVER(ee_in_base, upper, lower):
                ik_fail[q] = True
        keep &= ~ik_fail
    if verbose:
        # common.cpp:199-294: a pose is counted by the FIRST test that rejects it (approach, IK, open gripper, enclosed
        # gripper); with pose adjustment every collision rejection is counted as "open" (:290-294)
        coll_open = (status == _lib.CG_ST_REJ_COLL) & ~ik_fail
        coll_encl = (status == _lib.CG_ST_REJ_COLL_ENCL) & ~ik_fail
        print("n_approach_dir_rej={}, n_ik_rej={}, n_open_gripper_rej={}, n_close_gripper_rej={}".format(
            int((status == _lib.CG_ST_REJ_DIR).sum()), int(ik_fail.sum()), int(coll_open.sum()), int(coll_encl.sum())))
    return [poses[q].copy() for q in np.nonzero(keep)[0]]


def makeOccupancyGridFromCloudScan(pts, K, resolution):
    """my_cpp/common.cpp:324-431 (signature common.h:61): (P,3) scan points, camera K (unused by the reference's
    output as well), cell size -> (Q,3) float32 grid samples that lie on or behind the observed surface, in raster
    (x, y, z) order (the reference: OpenMP thread-arrival order)."""
    p = np.ascontiguousarray(np.asarray(pts, dtype=np.float64).astype(np.float32))
    if p.ndim != 2 or p.shape[1] != 3:
        raise ValueError(f"pts must be (N,3), got {p.shape}")     # assert(pts.cols()==3), common.cpp:329
    ctx = _lib.Context.get()
    res = float(np.float32(resolution))
    dims = (C.c_int * 3)()
    org = (C.c_float * 3)()
    ctx.check(ctx.lib.cg_occupancy_grid_geometry(_lib.ptr(p), p.shape[0], C.c_float(res), dims, org))
    nx, ny, nz = int(dims[0]), int(dims[1]), int(dims[2])
    if nx * ny * nz == 0:
        return np.zeros((0, 3), np.float32)
    flags = np.empty(nx * ny * nz, np.uint8)
    ctx.use_own_stream()   # blocking host call
    ctx.check(ctx.lib.cg_occupancy_from_scan_host(ctx.h, _lib.ptr(p), p.shape[0], C.c_float(res), _lib.ptr(flags)))
    idx = np.nonzero(flags)[0]
    xi, yi, zi = idx // (ny * nz), (idx // nz) % ny, idx % nz
    r32 = np.float32(res)
    out = np.stack([np.float32(org[0]) + xi.astype(np.float32) * r32, np.float32(org[1]) + yi.astype(np.float32) * r32,
                    np.float32(org[2]) + zi.astype(np.float32) * r32], axis=1).astype(np.float32)
    return out


def directionVecToRotation(direction, ref):
    """my_cpp/common.cpp:75-108 (twin of Utils.py:262-290): rotation taking ``ref`` onto ``direction``."""
    direction = np.asarray(direction, dtype=np.float32).reshape(3).copy()
    ref = np.asarray(ref, dtype=np.float32).reshape(3)
    direction /= np.linalg.norm(direction)
    v = np.cross(direction, ref)
    if np.linalg.norm(v) < 1e-5:
        return np.eye(3, dtype=np.float32)
    s = np.linalg.norm(v)
    c = float(np.dot(direction, ref))
    vs = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]], dtype=np.float32)
    R = (np.eye(3, dtype=np.float32) + vs + vs @ vs * (1 - c) / (s * s)).T
    u, _, vt = np.linalg.svd(R)
    return (u @ vt).astype(np.float32)


def augmentGraspPoses(R0, selected_point, sphere_pts, inplane_rot_step, hand_depth, approach_step, init_bite):
    """my_cpp/common.cpp:111-153 (exported by pybind.cpp:20, no Python caller in the reference): the cone enumeration
    R0 * R_sphere * R_inplane x approach depths.  The reference iterates ``sphere_pts.size()`` (rows*3, an
    out-of-bounds read, SURVEY.md 2.1 C4); this mirror iterates the rows."""
    R0 = np.asarray(R0, dtype=np.float32).reshape(3, 3)
    selected_point = np.asarray(selected_point, dtype=np.float32).reshape(3)
    sphere_pts = np.asarray(sphere_pts, dtype=np.float32).reshape(-1, 3)
    Rs = [R0]
    for sp in sphere_pts:
        R_sphere = directionVecToRotation(sp, np.array([1, 0, 0], np.float32))
        x_rot = np.float32(0)
        while x_rot < 180:                                   # for (float x_rot=0; x_rot<180; x_rot+=inplane_rot_step)
            a = float(x_rot) / 180.0 * np.pi
            ca, sa = np.cos(a), np.sin(a)
            R_inplane = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]], dtype=np.float32)
            Rs.append(R0 @ R_sphere @ R_inplane)
            x_rot = np.float32(x_rot + np.float32(inplane_rot_step))
    out = []
    for R in Rs:
        u, _, vt = np.linalg.svd(R)
        R = (u @ vt).astype(np.float32)
        approach_dir = R[:, 0]
        d = np.float32(0)
        while d < hand_depth:                                # for (float d=0; d<hand_depth; d+=approach_step)
            T = np.eye(4, dtype=np.float32)
            T[:3, :3] = R
            T[:3, 3] = selected_point + np.float32(init_bite) * approach_dir + approach_dir * d
            out.append(T)
            d = np.float32(d + np.float32(approach_step))
    return out


class CollisionManager:
    """my_cpp/collision_manager.h:33-52 (exported by pybind.cpp:13-18, no Python caller): one posed mesh against one
    point set.  The mesh is represented by its registered SDF (see register_gripper_sdf); isAnyCollision() evaluates
    the same predicate as filterGraspPose for the single transform set with setTransform().  With
    COLLISION_PREDICATE = "mesh" it is the reference class's own test: the registered mesh against the occupied voxels
    of the registered points at the registered resolution, and no SDF is needed."""

    def __init__(self):
        self._sdf = None
        self._mesh = None
        self._pts = np.zeros((0, 3), np.float32)
        self._res = None
        self._pose = np.eye(4, dtype=np.float32)

    def registerMesh(self, vertices, faces):
        vertices, faces = np.asarray(vertices), np.asarray(faces)
        if vertices.ndim != 2 or vertices.shape[1] != 3 or faces.ndim != 2 or faces.shape[1] != 3:
            raise ValueError("registerMesh: V,F must be (N,3)")                  # collision_manager.cpp:17-27 (exit(1))
        if COLLISION_PREDICATE == "mesh":
            self._mesh = _mesh_for(vertices, faces)
        else:
            self._sdf = _sdf_for(vertices, faces)
        return 0

    def registerPointCloud(self, pts, resolution):
        pts = np.asarray(pts)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError("registerPointCloud: pts must be (N,3)")            # collision_manager.cpp:57-61
        self._pts = np.ascontiguousarray(pts, dtype=np.float32)
        self._res = float(np.float32(resolution))
        return 1

    def setTransform(self, pose, ob_id):
        pose = np.asarray(pose)
        if pose.shape != (4, 4):
            raise ValueError("setTransform: pose must be (4,4)")                 # collision_manager.cpp:83-87
        self._pose = pose.astype(np.float32)

    def isAnyCollision(self):
        if COLLISION_PREDICATE == "mesh":
            if self._mesh is None or self._res is None:
                raise _lib.CgError("CollisionManager: registerMesh and registerPointCloud first")
            eye = np.eye(4)
            st, _, _ = filter_grasp_pose_mesh_raw(self._pose[None], eye[None], eye, eye, eye, False, False, self._mesh,
                                                  self._pts, None, np.zeros((0, 3), np.float32), self._res)
            return bool(st[0] == _lib.CG_ST_REJ_COLL)
        if self._sdf is None:
            raise _lib.CgError("CollisionManager: registerMesh first")
        eye = np.eye(4)
        st, _, _ = filter_grasp_pose_raw(self._pose[None], eye[None], eye, eye, eye, False, False, self._sdf, self._pts,
                                         None, np.zeros((0, 3), np.float32))
        return bool(st[0] == _lib.CG_ST_REJ_COLL)
