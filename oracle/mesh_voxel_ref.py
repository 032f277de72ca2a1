"""CPU ORACLE (test infrastructure only): the reference's own geometry predicate, "the posed gripper mesh touches an
occupied octree voxel" (my_cpp/collision_manager.cpp:15-111), with the reference's number types -- the semantic that
``my_cpp.COLLISION_PREDICATE = "mesh"`` (csrc/cg_mesh_collide.cu) computes bit for bit.

It restates oracle/fcl_semantic_ref.py with these conventions:

* occupied voxels (registerPointCloud, collision_manager.cpp:55-77): the points arrive as float32 (pybind narrows
  ``Eigen::MatrixXf``); ``res = double(float32(octo_resolution))``; ``key = floor(double(x) * (1.0 / res))`` per axis,
  deduplicated; keys outside octomap's 16-bit range (``-32768 <= key < 32768``) are dropped; a non-finite point is an
  error.  The key rule (``resolution_factor = 1.0 / resolution``, ``coordToKeyChecked``) is taken from octomap's
  source, which is not available here to check against;
* a voxel is the cube ``[key*res, (key+1)*res]`` per axis with centre ``(key + 0.5) * res`` (float64);
* the posed mesh uses the float32 ``gripper_in_cam`` of each (pose, symmetry, offset) widened to float64, and the
  float32 vertices widened to float64: ``Vc = ((R0*vx + R1*vy) + R2*vz) + t`` with one rounding per operation;
* collision = some cube overlaps some posed triangle under the 13-axis separating-axis test (3 box faces, the triangle
  normal cross(e0, e1), cross(eye[a], e_k) for e0 = v1-v0, e1 = v2-v1, e2 = v0-v2); projections
  ``(dx*ax + dy*ay) + dz*az`` of d = Vc - centre, radius ``half*((|ax| + |ay|) + |az|)``; an axis separates iff
  ``min > r`` or ``max < -r`` (touching collides).

Every sum is written out in scalar order so that the CUDA kernel can be compared bit for bit.  FCL itself (float32 leaf
boxes, GJK/EPA narrow phase) is not restated; agreement with it stays unpinned.
"""
import numpy as np

KEY_LIMIT = 32768          # octomap: tree_max_val, keys are 16 bits


def occupied_voxel_keys(points_f32, res):
    """Sorted unique (K,3) int64 keys of the registered points (x, then y, then z ascending)."""
    p = np.asarray(points_f32, np.float64).astype(np.float32).astype(np.float64).reshape(-1, 3)
    if not np.isfinite(p).all():
        raise ValueError("occupied_voxel_keys: non-finite point")
    r = float(np.float32(res))
    k = np.floor(p * (1.0 / r))
    k = k[((k >= -KEY_LIMIT) & (k < KEY_LIMIT)).all(1)].astype(np.int64)
    if len(k) == 0:
        return np.zeros((0, 3), np.int64)
    return np.unique(k, axis=0)


def posed_vertices(V, T):
    """((R0*vx + R1*vy) + R2*vz) + t per row, float64, one rounding per operation."""
    V = np.asarray(V, np.float64)
    T = np.asarray(T, np.float64)
    out = np.empty_like(V)
    for r in range(3):
        out[:, r] = ((T[r, 0] * V[:, 0] + T[r, 1] * V[:, 1]) + T[r, 2] * V[:, 2]) + T[r, 3]
    return out


def _axes(tri):
    """The 10 non-face SAT axes of (N,3,3) posed triangles -> list of (ax, ay, az): the normal cross(e0, e1), then
    cross(eye[a], e_k) = (0, -ez, ey), (ez, 0, -ex), (-ey, ex, 0) for k = 0, 1, 2 (the zero components contribute
    exactly +-0 to a projection, so leaving their products out changes no value)."""
    e = [tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 1], tri[:, 0] - tri[:, 2]]
    e0, e1 = e[0], e[1]
    out = [(e0[:, 1] * e1[:, 2] - e0[:, 2] * e1[:, 1], e0[:, 2] * e1[:, 0] - e0[:, 0] * e1[:, 2],
            e0[:, 0] * e1[:, 1] - e0[:, 1] * e1[:, 0])]
    zero = np.zeros(len(tri))
    for ek in e:
        out.append((zero, -ek[:, 2], ek[:, 1]))
        out.append((ek[:, 2], zero, -ek[:, 0]))
        out.append((-ek[:, 1], ek[:, 0], zero))
    return out


def box_triangle_sat(tri, centres, half, with_margin=False):
    """tri (N,3,3) posed triangles, centres (N,3) cube centres, half: cube half side.  Returns overlap (N,) bool and,
    with_margin, the SAT margin (N,): the largest separating gap over the non-degenerate axes, in metres
    (> 0 separated, <= 0 overlapping, 0 = touching)."""
    d = tri - centres[:, None, :]
    ov = np.ones(len(d), bool)
    margin = np.full(len(d), -np.inf)
    for a in range(3):
        lo, hi = d[:, :, a].min(1), d[:, :, a].max(1)
        ov &= ~((lo > half) | (hi < -half))
        if with_margin:
            margin = np.maximum(margin, np.maximum(lo - half, -half - hi))
    for ax, ay, az in _axes(tri):
        p = [(d[:, i, 0] * ax + d[:, i, 1] * ay) + d[:, i, 2] * az for i in range(3)]
        lo = np.minimum(np.minimum(p[0], p[1]), p[2])
        hi = np.maximum(np.maximum(p[0], p[1]), p[2])
        r = half * ((np.abs(ax) + np.abs(ay)) + np.abs(az))
        ov &= ~((lo > r) | (hi < -r))
        if with_margin:
            nrm = np.sqrt(ax * ax + ay * ay + az * az)
            ok = nrm > 0
            gap = np.where(ok, np.maximum(lo - r, -r - hi) / np.where(ok, nrm, 1.0), -np.inf)
            margin = np.maximum(margin, gap)
    return (ov, margin) if with_margin else ov


class _TriGrid:
    """Uniform grid over the gripper-frame mesh with per-cell triangle lists (triangle AABB, conservative): a broad
    phase only -- every pair it lets through is decided by the exact SAT above."""

    def __init__(self, V, F, cell=0.002):
        V = np.asarray(V, np.float64)
        F = np.asarray(F, np.int64)
        tri = V[F]
        self.lo = V.min(0) - cell
        self.cell = cell
        self.dims = np.floor((V.max(0) + cell - self.lo) / cell).astype(np.int64) + 1
        a = np.floor((tri.min(1) - self.lo) / cell).astype(np.int64)
        b = np.floor((tri.max(1) - self.lo) / cell).astype(np.int64)
        cells, tris = [], []
        span = (b - a).max(0) + 1
        for dx in range(span[0]):
            for dy in range(span[1]):
                for dz in range(span[2]):
                    c = a + np.array([dx, dy, dz])
                    m = (c <= b).all(1)
                    cells.append(self._lin(c[m]))
                    tris.append(np.nonzero(m)[0])
        cells, tris = np.concatenate(cells), np.concatenate(tris)
        o = np.argsort(cells, kind="stable")
        self.tris = tris[o]
        n = int(np.prod(self.dims))
        self.start = np.zeros(n + 1, np.int64)
        np.add.at(self.start, cells + 1, 1)
        self.start = np.cumsum(self.start)

    def _lin(self, c):
        return (c[:, 0] * self.dims[1] + c[:, 1]) * self.dims[2] + c[:, 2]

    def candidates(self, qlo, qhi):
        """(voxel, triangle) index pairs for gripper-frame query boxes (K,3) lo / hi."""
        a = np.clip(np.floor((qlo - self.lo) / self.cell).astype(np.int64), 0, self.dims - 1)
        b = np.clip(np.floor((qhi - self.lo) / self.cell).astype(np.int64), 0, self.dims - 1)
        inside = ((qhi >= self.lo) & (qlo <= self.lo + self.dims * self.cell)).all(1)
        vs, ts = [], []
        span = (b - a).max(0) + 1 if len(a) else np.zeros(3, np.int64)
        for dx in range(int(span[0])):
            for dy in range(int(span[1])):
                for dz in range(int(span[2])):
                    c = a + np.array([dx, dy, dz])
                    m = inside & (c <= b).all(1)
                    lin = self._lin(c[m])
                    s, e = self.start[lin], self.start[lin + 1]
                    cnt = e - s
                    if cnt.sum() == 0:
                        continue
                    vi = np.repeat(np.nonzero(m)[0], cnt)
                    off = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
                    vs.append(vi)
                    ts.append(self.tris[np.repeat(s, cnt) + off])
        if not vs:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        pair = np.unique(np.concatenate(vs) * (1 << 32) + np.concatenate(ts))
        return pair >> 32, pair & 0xFFFFFFFF


_GRIDS = {}


def _grid_for(V, F):
    key = (np.ascontiguousarray(V, np.float64).tobytes(), np.ascontiguousarray(F, np.int64).tobytes())
    if key not in _GRIDS:
        _GRIDS.clear() if len(_GRIDS) > 8 else None
        _GRIDS[key] = _TriGrid(V, F)
    return _GRIDS[key]


def mesh_voxel_pairs(V, F, gripper_in_cam, keys, res):
    """The triangle-cube pairs the oracle tests for one pose: (posed triangles (N,3,3), cube centres (N,3), half),
    float64.  V, gripper_in_cam, res are used as given (float64); filter_mesh_ref narrows them like the reference."""
    V = np.asarray(V, np.float64)
    F = np.asarray(F, np.int64)
    T = np.asarray(gripper_in_cam, np.float64)
    res = float(res)
    keys = np.asarray(keys, np.int64).reshape(-1, 3)
    half = 0.5 * res
    if len(keys) == 0:
        return np.zeros((0, 3, 3)), np.zeros((0, 3)), half
    centres = (keys.astype(np.float64) + 0.5) * res
    # broad phase in the gripper frame: cube -> parallelepiped, bounded by half * sum|Ainv| per axis, plus slack
    Ainv = np.linalg.inv(T)
    u = centres @ Ainv[:3, :3].T + Ainv[:3, 3]
    slack = 1e-6 * (1.0 + np.abs(centres).max(1, keepdims=True) + np.abs(T[:3, 3]).max())
    ext = half * np.abs(Ainv[:3, :3]).sum(1) + slack
    vi, ti = _grid_for(V, F).candidates(u - ext, u + ext)
    Vc = posed_vertices(V, T)
    return Vc[F[ti]], centres[vi], half


def mesh_hits_voxels(V, F, gripper_in_cam, keys, res, return_margin=False):
    """True iff some occupied cube overlaps some triangle of the posed mesh.  return_margin: also the smallest |SAT
    margin| (metres) over the tested pairs (inf when no pair is tested)."""
    tri, c, half = mesh_voxel_pairs(V, F, gripper_in_cam, keys, res)
    if not return_margin:
        return bool(box_triangle_sat(tri, c, half).any()) if len(tri) else False
    if len(tri) == 0:
        return False, np.inf
    ov, m = box_triangle_sat(tri, c, half, with_margin=True)
    return bool(ov.any()), float(np.abs(m).min())


def sat_margins(V, F, gripper_in_cam, keys, res):
    """SAT margins (metres) of every triangle-cube pair tested for one pose (see box_triangle_sat)."""
    tri, c, half = mesh_voxel_pairs(V, F, gripper_in_cam, keys, res)
    if len(tri) == 0:
        return np.zeros(0)
    return box_triangle_sat(tri, c, half, with_margin=True)[1]


def filter_mesh_ref(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs, gripper_in_grasp, filter_dir, adjust,
                    mesh_open, open_pts, mesh_encl, encl_pts, res, split=False):
    """filter_ref.filter_ref with the mesh-vs-voxel predicate: mesh_* = (V, F) of the open / enclosed gripper, res =
    octo_resolution.  Returns (status u8 (Q,), offset i8 (Q,), poses f32 (Q,4,4)), Q = G*S in (pose, symmetry) order."""
    from catgrasp_b200.my_cpp import _mm4_f32, grasp_in_cam_unshifted
    f32 = np.float32
    g = grasp_in_cam_unshifted(grasp_poses, symmetry_tfs, nocs_pose, canonical_to_nocs)
    gig = np.asarray(gripper_in_grasp, np.float64).astype(f32)
    r = float(np.float32(res))
    ko = occupied_voxel_keys(open_pts, r)
    ke = occupied_voxel_keys(encl_pts, r)
    Vo = np.asarray(mesh_open[0], np.float64).astype(f32).astype(np.float64)
    Ve = np.asarray(mesh_encl[0], np.float64).astype(f32).astype(np.float64) if mesh_encl is not None else None
    Q = g.shape[0]
    status = np.zeros(Q, np.uint8)
    offset = np.full(Q, -1, np.int8)
    poses = np.zeros((Q, 4, 4), f32)
    step1 = f32(0.001)
    step2 = f32(step1 + f32(0.001))
    n_off = 5 if adjust else 1
    use_split = split and not adjust
    for q in range(Q):
        x, y, z = g[q, 0, 0], g[q, 1, 0], g[q, 2, 0]
        n = np.sqrt(f32(f32(f32(x * x) + f32(y * y)) + f32(z * z)))
        if filter_dir and f32(z / n) < 0:
            status[q] = 1
            continue
        open_hit = False
        for k in range(n_off):
            step = f32(0) if k == 0 else (step1 if k <= 2 else step2)
            sign = f32(1) if (k == 0 or (k & 1)) else f32(-1)
            cur = g[q].copy()
            cur[:3, 3] = (g[q, :3, 3] + ((step * g[q, :3, 1]).astype(f32) * sign).astype(f32)).astype(f32)
            gic = _mm4_f32(cur, gig).astype(np.float64)
            hit_o = mesh_hits_voxels(Vo, mesh_open[1], gic, ko, r)
            hit_e = (not hit_o) and len(ke) > 0 and mesh_hits_voxels(Ve, mesh_encl[1], gic, ke, r)
            if not (hit_o or hit_e):
                offset[q] = k
                poses[q] = cur
                break
            open_hit = hit_o
        if offset[q] < 0:
            status[q] = 4 if (use_split and not open_hit) else 3
    return status, offset, poses
