"""Seeded synthetic assets for tests and bench (SURVEY.md 8d): the reference ships no weights,
meshes, SDFs or datasets (README.md:68-75), so parity and throughput run on these.

Everything here is numpy on the host and deterministic for a given seed.
"""
from collections import OrderedDict

import numpy as np

# ----------------------------------------------------------------------------- checkpoints
_ENC_SHAPES = [
    ("feat.stn.conv1", (64, 6, 1)), ("feat.stn.conv2", (128, 64, 1)), ("feat.stn.conv3", (1024, 128, 1)),
    ("feat.stn.fc1", (512, 1024)), ("feat.stn.fc2", (256, 512)), ("feat.stn.fc3", (9, 256)),
    ("feat.stn.bn1", 64), ("feat.stn.bn2", 128), ("feat.stn.bn3", 1024), ("feat.stn.bn4", 512), ("feat.stn.bn5", 256),
    ("feat.conv1", (64, 6, 1)), ("feat.conv2", (128, 64, 1)), ("feat.conv3", (1024, 128, 1)),
    ("feat.bn1", 64), ("feat.bn2", 128), ("feat.bn3", 1024),
    ("feat.fstn.conv1", (64, 64, 1)), ("feat.fstn.conv2", (128, 64, 1)), ("feat.fstn.conv3", (1024, 128, 1)),
    ("feat.fstn.fc1", (512, 1024)), ("feat.fstn.fc2", (256, 512)), ("feat.fstn.fc3", (4096, 256)),
    ("feat.fstn.bn1", 64), ("feat.fstn.bn2", 128), ("feat.fstn.bn3", 1024), ("feat.fstn.bn4", 512),
    ("feat.fstn.bn5", 256),
]


def _head_shapes(kind, n_out):
    if kind == "cls":   # pointnet2.py:281-286
        return [("fc1", (512, 1024)), ("fc2", (256, 512)), ("fc3", (n_out, 256)), ("bn1", 512), ("bn2", 256)]
    return [("conv1", (512, 1088, 1)), ("conv2", (256, 512, 1)), ("conv3", (128, 256, 1)),   # pointnet2.py:308-314
            ("conv4", (n_out, 128, 1)), ("bn1", 512), ("bn2", 256), ("bn3", 128)]


def make_state_dict(kind, n_out, seed=0, module_prefix=True, as_torch=True, logit_gain=1.0):
    """A PointNetCls ('cls') / PointNetSeg ('seg') state_dict with torch-default-like weight ranges
    (U(+-1/sqrt(fan_in))) and randomised BatchNorm statistics so that folding is exercised:
    running_mean ~ N(0,0.2), running_var ~ U(0.5,1.5), weight ~ U(0.5,1.5), bias ~ N(0,0.1)."""
    rng = np.random.RandomState(seed)
    sd = OrderedDict()
    for name, shp in _ENC_SHAPES + _head_shapes(kind, n_out):
        if isinstance(shp, tuple):
            fan_in = shp[1]
            bound = 1.0 / np.sqrt(fan_in)
            sd[name + ".weight"] = rng.uniform(-bound, bound, size=shp).astype(np.float32)
            sd[name + ".bias"] = rng.uniform(-bound, bound, size=(shp[0],)).astype(np.float32)
        else:
            sd[name + ".weight"] = rng.uniform(0.5, 1.5, size=(shp,)).astype(np.float32)
            sd[name + ".bias"] = rng.normal(0, 0.1, size=(shp,)).astype(np.float32)
            sd[name + ".running_mean"] = rng.normal(0, 0.2, size=(shp,)).astype(np.float32)
            sd[name + ".running_var"] = rng.uniform(0.5, 1.5, size=(shp,)).astype(np.float32)
            sd[name + ".num_batches_tracked"] = np.array(100, dtype=np.int64)
    if logit_gain != 1.0:   # a trained head separates its classes; default-range weights give near-uniform scores
        last = "fc3" if kind == "cls" else "conv4"
        sd[last + ".weight"] = (sd[last + ".weight"] * logit_gain).astype(np.float32)
        sd[last + ".bias"] = (sd[last + ".bias"] * logit_gain).astype(np.float32)
    if as_torch:
        import torch
        sd = OrderedDict((k, torch.from_numpy(np.asarray(v))) for k, v in sd.items())
    if module_prefix:   # checkpoints come from nn.DataParallel (trainer_grasp.py:33)
        sd = OrderedDict(("module." + k, v) for k, v in sd.items())
    return sd


def write_artifacts(artifact_dir, kind, n_pts, seed=0, with_normalizer=True, ce_loss_bins=100, logit_gain=1.0,
                    state_dict=None, normalizer=None):
    """Create an artifacts directory in the reference's layout (predicter.py:41-64, :101-132).  ``state_dict`` /
    ``normalizer=(mean, std)`` override the seeded defaults."""
    import os
    import pickle
    import torch
    import yaml
    os.makedirs(artifact_dir, exist_ok=True)
    if kind == "cls":
        classes = [float(v) for v in np.linspace(0, 1, 11)]   # config_grasp.yml: 11 edges -> 10 classes
        cfg = {"n_pts": int(n_pts), "input_channel": 6, "classes": classes, "batch_size": 240}
        n_out = 10
        cfg_name = "config_grasp.yml"
    else:
        cfg = {"n_pts": int(n_pts), "input_channel": 6, "ce_loss_bins": int(ce_loss_bins), "batch_size": 34}
        n_out = 3 * int(ce_loss_bins)
        cfg_name = "config_nunocs.yml"
    with open(os.path.join(artifact_dir, cfg_name), "w") as f:
        yaml.safe_dump(cfg, f)
    sd = state_dict if state_dict is not None else make_state_dict(kind, n_out, seed=seed, logit_gain=logit_gain)
    torch.save({"epoch": 1, "state_dict": sd, "best_res": 0.0}, os.path.join(artifact_dir, "best_val.pth.tar"))
    if normalizer is not None:
        with open(os.path.join(artifact_dir, "normalizer.pkl"), "wb") as f:
            pickle.dump({"mean": np.asarray(normalizer[0]), "std": np.asarray(normalizer[1])}, f)
    elif with_normalizer:
        rng = np.random.RandomState(seed + 7)
        if kind == "cls":   # grasp-frame coordinates in metres (dataset_grasp.py:84-85)
            mean = np.concatenate([rng.normal(0, 0.002, 3), rng.normal(0, 0.05, 3)])
            std = np.concatenate([rng.uniform(0.008, 0.012, 3), rng.uniform(0.5, 0.6, 3)])
        else:               # min/max-normalised coordinates in [0,1] (augmentations.py:70-75)
            mean = np.concatenate([rng.normal(0.5, 0.05, 3), rng.normal(0, 0.05, 3)])
            std = np.concatenate([rng.uniform(0.25, 0.35, 3), rng.uniform(0.5, 0.6, 3)])
        with open(os.path.join(artifact_dir, "normalizer.pkl"), "wb") as f:
            pickle.dump({"mean": mean, "std": std}, f)
    return artifact_dir


LATTICE_LEVELS = 26          # lattice positions per axis: normalised coordinate 0.04*g, NOCS bin 4*g
_LATTICE_HINGES = LATTICE_LEVELS + 2


def make_lattice_seg_state_dict(seed=0, mean=None, std=None, bins=100, beta=10.0, module_prefix=True, as_torch=True):
    """A PointNetSeg state_dict that *reads the NUNOCS bins off the input*: for a cloud whose min/max-normalised
    coordinates (augmentations.py:70-75) sit on the lattice {0, 0.04, ..., 1.0}, bin min(4*g, 99) wins with a logit gap of
    ``beta``, so every implementation (fp32 CPU, tcgen05 split precision) yields the same NOCS cloud and the full
    ``NunocsPredicter.predict`` success path (predicter.py:135-203) can be compared end to end.

    All other weights and every BatchNorm statistic stay as random as in :func:`make_state_dict`; the hand-set
    rows are solved *through* the random BatchNorm so folding is still exercised.  Construction: both STN heads
    output identity (fc3 = 0); three channels carry the un-normalised coordinate through feat.conv1 / conv1 /
    conv2; conv3 builds 28 hinges relu(x - 0.04 m) per axis; conv4 combines three hinges into a unit tent per
    lattice level.
    """
    assert bins == 100 and 3 * _LATTICE_HINGES <= 128
    sd = make_state_dict("seg", 3 * bins, seed=seed, module_prefix=False, as_torch=False)
    eps = 1e-5

    def through_bn(bn, rows, w_t, b_t):
        """conv rows such that BN(conv(x)) = w_t @ x + b_t."""
        s = np.sqrt(sd[bn + ".running_var"][rows].astype(np.float64) + eps) / sd[bn + ".weight"][rows]
        w = w_t * s[:, None]
        b = (b_t - sd[bn + ".bias"][rows]) * s + sd[bn + ".running_mean"][rows]
        return w.astype(np.float32), b.astype(np.float32)

    for stn in ("feat.stn.fc3", "feat.fstn.fc3"):
        sd[stn + ".weight"][:] = 0
        sd[stn + ".bias"][:] = 0
    rows = np.arange(3)
    # encoder conv1: channel j = input_j * std_j + mean_j (undoes the normalizer of dataset_nunocs.py:58-59)
    w_t = np.zeros((3, 6))
    w_t[rows, rows] = 1.0 if std is None else np.asarray(std, np.float64)[:3]
    b_t = np.zeros(3) if mean is None else np.asarray(mean, np.float64)[:3]
    w, b = through_bn("feat.bn1", rows, w_t, b_t)
    sd["feat.conv1.weight"][rows] = w[:, :, None]
    sd["feat.conv1.bias"][rows] = b
    # head conv1 (input = [1024 global | 64 point features]) and conv2: pass the three channels on
    for name, bn, cin, off in (("conv1", "bn1", 1088, 1024), ("conv2", "bn2", 512, 0)):
        w_t = np.zeros((3, cin))
        w_t[rows, off + rows] = 1.0
        w, b = through_bn(bn, rows, w_t, np.zeros(3))
        sd[name + ".weight"][rows] = w[:, :, None]
        sd[name + ".bias"][rows] = b
    # conv3: hinges h[a, m] = relu(x_a - 0.04 m), m = -1 .. LATTICE_LEVELS
    H = _LATTICE_HINGES
    hr = np.arange(3 * H)
    w_t = np.zeros((3 * H, 256))
    b_t = np.zeros(3 * H)
    for a in range(3):
        for i in range(H):
            w_t[a * H + i, a] = 1.0
            b_t[a * H + i] = -0.04 * (i - 1)
    w, b = through_bn("bn3", hr, w_t, b_t)
    sd["conv3.weight"][hr] = w[:, :, None]
    sd["conv3.bias"][hr] = b
    # conv4: tent_m = (h[m-1] - 2 h[m] + h[m+1]) / 0.04 on bin 4 m; every other bin sits at -beta
    W4 = np.zeros((3 * bins, 128), np.float32)
    b4 = np.full(3 * bins, -beta, np.float32)
    for a in range(3):
        for m in range(LATTICE_LEVELS):
            r = a * bins + min(4 * m, bins - 1)      # x = 1.0 (the far end of the largest extent) has no bin: use 99
            b4[r] = 0.0
            W4[r, a * H + m] += beta / 0.04
            W4[r, a * H + m + 1] -= 2 * beta / 0.04
            W4[r, a * H + m + 2] += beta / 0.04
    sd["conv4.weight"] = W4[:, :, None].copy()
    sd["conv4.bias"] = b4
    if as_torch:
        import torch
        sd = OrderedDict((k, torch.from_numpy(np.asarray(v))) for k, v in sd.items())
    if module_prefix:
        sd = OrderedDict(("module." + k, v) for k, v in sd.items())
    return sd


# ----------------------------------------------------------------------------- geometry
def random_rotation(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def sample_hex_nut(n, rng, across_flats=0.020, height=0.008, bore=0.010):
    """Surface samples + outward normals of a hex nut (SURVEY.md 8d: 20 mm AF, 8 mm high, 10 mm bore)."""
    R = across_flats / np.sqrt(3.0)            # circumradius
    a_side = 6 * R * height
    a_cap = 2 * (1.5 * np.sqrt(3) * R * R - np.pi * (bore / 2) ** 2)
    a_bore = np.pi * bore * height
    w = np.array([a_side, a_cap, a_bore])
    which = rng.choice(3, size=n, p=w / w.sum())
    pts = np.zeros((n, 3))
    nrm = np.zeros((n, 3))
    # sides
    m = which == 0
    k = rng.randint(0, 6, size=m.sum())
    t = rng.uniform(0, 1, size=m.sum())
    a0, a1 = k * np.pi / 3, (k + 1) * np.pi / 3
    p0 = np.stack([R * np.cos(a0), R * np.sin(a0)], 1)
    p1 = np.stack([R * np.cos(a1), R * np.sin(a1)], 1)
    xy = p0 + (p1 - p0) * t[:, None]
    am = (a0 + a1) / 2
    pts[m] = np.concatenate([xy, rng.uniform(-height / 2, height / 2, size=(m.sum(), 1))], 1)
    nrm[m] = np.stack([np.cos(am), np.sin(am), np.zeros_like(am)], 1)
    # caps (rejection sample the hexagon minus the bore)
    m = which == 1
    cnt = m.sum()
    xy = np.zeros((0, 2))
    while xy.shape[0] < cnt:
        c = rng.uniform(-R, R, size=(2 * cnt + 16, 2))
        ang = np.arctan2(c[:, 1], c[:, 0]) % (np.pi / 3) - np.pi / 6
        rad = np.linalg.norm(c, axis=1)
        ok = (rad * np.cos(ang) <= across_flats / 2) & (rad >= bore / 2)
        xy = np.concatenate([xy, c[ok]], 0)
    xy = xy[:cnt]
    s = rng.choice([-1.0, 1.0], size=cnt)
    pts[m] = np.concatenate([xy, (s * height / 2)[:, None]], 1)
    nrm[m] = np.stack([np.zeros(cnt), np.zeros(cnt), s], 1)
    # bore
    m = which == 2
    th = rng.uniform(0, 2 * np.pi, size=m.sum())
    pts[m] = np.stack([bore / 2 * np.cos(th), bore / 2 * np.sin(th), rng.uniform(-height / 2, height / 2, m.sum())], 1)
    nrm[m] = np.stack([-np.cos(th), -np.sin(th), np.zeros_like(th)], 1)
    return pts, nrm


def make_pile(n_points, n_objects=8, seed=0, bin_size=0.10, floor_z=0.70, max_tilt_deg=30.0):
    """A clutter pile of hex nuts in the camera frame (z >= 0.1 as required by dataset_grasp.py:64).

    Nuts lie roughly flat (tilt <= max_tilt_deg, random yaw) at rejection-sampled, mostly non-overlapping
    positions in a bin_size x bin_size bin whose floor is at camera z = floor_z; a second layer forms when
    the bin is full.  Returns dict(cloud_xyz (n_points,3) f64, cloud_normal (n_points,3) f64,
    object_id (n_points,), object_poses (n_objects,4,4)); only camera-facing samples are kept and normals
    point at the camera (Utils.py:205-213)."""
    rng = np.random.RandomState(seed)
    per = int(np.ceil(n_points * 2.6 / n_objects))
    P, Nn, ids, poses, centers = [], [], [], [], []
    for k in range(n_objects):
        p, n = sample_hex_nut(per, rng)
        tilt = np.deg2rad(rng.uniform(0, max_tilt_deg))
        phi = rng.uniform(0, 2 * np.pi)
        axis = np.array([np.cos(phi), np.sin(phi), 0.0])
        K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        Rt = np.eye(3) + np.sin(tilt) * K + (1 - np.cos(tilt)) * (K @ K)
        yaw = rng.uniform(0, 2 * np.pi)
        Rz = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
        Rm = Rt @ Rz
        layer = 0
        for attempt in range(200):
            c = rng.uniform(-bin_size / 2 + 0.012, bin_size / 2 - 0.012, size=2)
            if all(np.linalg.norm(c - q[:2]) > 0.025 or q[2] != layer for q in centers):
                break
            if attempt % 50 == 49:
                layer += 1
        centers.append(np.array([c[0], c[1], layer]))
        t = np.array([c[0], c[1], floor_z - 0.006 - 0.009 * layer - rng.uniform(0, 0.002)])
        T = np.eye(4)
        T[:3, :3] = Rm
        T[:3, 3] = t
        p = p @ Rm.T + t
        n = n @ Rm.T
        vis = np.einsum("ij,ij->i", n, p) < 0      # facing the camera at the origin
        P.append(p[vis]); Nn.append(n[vis]); ids.append(np.full(vis.sum(), k)); poses.append(T)
    P = np.concatenate(P); Nn = np.concatenate(Nn); ids = np.concatenate(ids)
    assert P.shape[0] >= n_points, "increase oversampling"
    sel = rng.choice(P.shape[0], size=n_points, replace=False)
    return {"cloud_xyz": P[sel].astype(np.float64), "cloud_normal": Nn[sel].astype(np.float64),
            "object_id": ids[sel], "object_poses": np.stack(poses)}


def _rot_x(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[1, 0, 0], [0, c, -s], [0, s, c]])


def make_candidates(cloud_xyz, cloud_normal, n_cand, seed=0, hand_depth=0.012, approach_step=0.002, init_bite=0.002,
                    cone_deg=35.0):
    """Grasp poses from the reference's cone parametrisation (grasp_sampler.py:269-289):
    approach = -normal, cone directions within ``cone_deg`` (reference: 60 deg), in-plane rotations 0..150 step 30 deg, depth steps."""
    rng = np.random.RandomState(seed)
    out = np.zeros((n_cand, 4, 4))
    sel = rng.randint(0, cloud_xyz.shape[0], size=n_cand)
    for i, s in enumerate(sel):
        approach = -cloud_normal[s] / np.linalg.norm(cloud_normal[s])
        tmp = rng.normal(size=3)
        minor = tmp - approach * np.dot(tmp, approach)
        minor /= np.linalg.norm(minor)
        major = np.cross(minor, approach)
        R0 = np.stack([approach, major, minor], 1)
        # cone direction: rotate about a random in-plane axis by up to 60 deg
        ang = rng.uniform(0, np.deg2rad(cone_deg))
        phi = rng.uniform(0, 2 * np.pi)
        axis = np.array([0, np.cos(phi), np.sin(phi)])
        K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        R_cone = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * (K @ K)
        R = R0 @ R_cone @ _rot_x(np.deg2rad(30.0 * rng.randint(0, 6)))
        d = approach_step * rng.randint(0, int(hand_depth / approach_step))
        T = np.eye(4)
        T[:3, :3] = R
        T[:3, 3] = cloud_xyz[s] + (init_bite + d) * R[:, 0]
        out[i] = T
    return out


# ----------------------------------------------------------------------------- gripper proxy
def _box_sdf(p, lo, hi):
    c = (lo + hi) / 2
    h = (hi - lo) / 2
    q = np.abs(p - c) - h
    return np.linalg.norm(np.maximum(q, 0), axis=-1) + np.minimum(q.max(axis=-1), 0)


def _box_mesh(lo, hi):
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    V = np.array([[x0, y0, z0], [x1, y0, z0], [x1, y1, z0], [x0, y1, z0],
                  [x0, y0, z1], [x1, y0, z1], [x1, y1, z1], [x0, y1, z1]], dtype=np.float64)
    F = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4],
                  [1, 2, 6], [1, 6, 5], [2, 3, 7], [2, 7, 6], [3, 0, 4], [3, 4, 7]], dtype=np.int32)
    return V, F


def make_gripper_proxy(res=0.001, pad_cells=5):
    """Two-finger box gripper (SURVEY.md 8d): palm 40x60x30 mm, fingers 45x8x20 mm, opening 50 mm.

    Gripper frame: +x is the approach axis (fingers extend from x=0 to x=0.045), +y the closing axis.
    Returns a dict with, for 'open' and 'enclosed': mesh (V,F), sdf grid (data[i][j][k] f32, origin, res),
    and ``gripper_in_grasp`` (4,4): the grasp centre sits 10 mm behind the finger tips."""
    palm = (np.array([-0.040, -0.030, -0.015]), np.array([0.0, 0.030, 0.015]))
    f1 = (np.array([0.0, 0.025, -0.010]), np.array([0.045, 0.033, 0.010]))
    f2 = (np.array([0.0, -0.033, -0.010]), np.array([0.045, -0.025, 0.010]))
    gap = (np.array([0.0, -0.025, -0.010]), np.array([0.045, 0.025, 0.010]))
    lo = np.array([-0.040, -0.033, -0.015]) - pad_cells * res
    hi = np.array([0.045, 0.033, 0.015]) + pad_cells * res
    dims = np.round((hi - lo) / res).astype(int) + 1
    gi, gj, gk = np.meshgrid(np.arange(dims[0]), np.arange(dims[1]), np.arange(dims[2]), indexing="ij")
    P = lo[None, None, None, :] + res * np.stack([gi, gj, gk], -1)

    def build(boxes):
        sd = np.min(np.stack([_box_sdf(P, b[0], b[1]) for b in boxes], 0), 0)
        Vs, Fs, off = [], [], 0
        for b in boxes:
            V, F = _box_mesh(b[0], b[1])
            Vs.append(V); Fs.append(F + off); off += V.shape[0]
        return {"V": np.concatenate(Vs), "F": np.concatenate(Fs).astype(np.int32),
                "sdf": sd.astype(np.float32), "origin": lo.astype(np.float32), "res": np.float32(res)}

    gig = np.eye(4)
    gig[0, 3] = -0.035
    return {"open": build([palm, f1, f2]), "enclosed": build([palm, f1, f2, gap]), "gripper_in_grasp": gig}


def _hexa_mesh(C, n):
    """Convex hexahedron with corners C (8,3) in _box_mesh order, every (planar) quad face split into an n x n grid
    of 2 n^2 outward-facing triangles."""
    faces = [(0, 3, 2, 1), (4, 5, 6, 7), (0, 1, 5, 4), (1, 2, 6, 5), (2, 3, 7, 6), (3, 0, 4, 7)]
    t = np.linspace(0.0, 1.0, n + 1)
    Vs, Fs, off = [], [], 0
    for a, b, c, d in faces:
        u, v = np.meshgrid(t, t, indexing="ij")
        u, v = u[..., None], v[..., None]
        P = (1 - u) * (1 - v) * C[a] + u * (1 - v) * C[b] + u * v * C[c] + (1 - u) * v * C[d]
        Vs.append(P.reshape(-1, 3))
        i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        p00 = (i * (n + 1) + j).ravel() + off
        p10, p01, p11 = p00 + (n + 1), p00 + 1, p00 + n + 2
        Fs.append(np.concatenate([np.stack([p00, p10, p11], 1), np.stack([p00, p11, p01], 1)]))
        off += (n + 1) ** 2
    return np.concatenate(Vs), np.concatenate(Fs).astype(np.int32)


def _hexa_sdf(p, C):
    """max over the six face planes of the signed plane distance: the exact sign of a convex hexahedron, exact
    distance inside and a lower bound outside."""
    faces = [(0, 3, 2), (4, 5, 6), (0, 1, 5), (1, 2, 6), (2, 3, 7), (3, 0, 4)]
    out = None
    for a, b, c in faces:
        nrm = np.cross(C[b] - C[a], C[c] - C[a])
        nrm /= np.linalg.norm(nrm)
        d = (p - C[a]) @ nrm
        out = d if out is None else np.maximum(out, d)
    return out


def make_dense_gripper_proxy(res=0.001, pad_cells=5, n=24, chamfer=0.004):
    """make_gripper_proxy's gripper finely triangulated (2 n^2 triangles per face: 20 736 for the open gripper and
    27 648 with the swept volume at n = 24, about the density of a real Hand-E mesh), with the inner edge of each
    finger tip chamfered by ``chamfer`` metres at 45 degrees in the x-y plane, so that some faces are not
    axis-aligned.  Same dictionary layout as make_gripper_proxy; the SDF grids are the signed plane-distance bound of
    the convex parts (exact sign)."""
    def box(lo, hi):
        V, _ = _box_mesh(np.asarray(lo, np.float64), np.asarray(hi, np.float64))
        return V

    palm = box([-0.040, -0.030, -0.015], [0.0, 0.030, 0.015])
    f1 = box([0.0, 0.025, -0.010], [0.045, 0.033, 0.010])
    f2 = box([0.0, -0.033, -0.010], [0.045, -0.025, 0.010])
    gap = box([0.0, -0.025, -0.010], [0.045, 0.025, 0.010])
    # tip corners on the inner (closing) side move back along x: corners 1, 5 of f1 (y = 0.025), 2, 6 of f2 (y = -0.025)
    f1[[1, 5], 0] -= chamfer
    f2[[2, 6], 0] -= chamfer
    lo = np.array([-0.040, -0.033, -0.015]) - pad_cells * res
    hi = np.array([0.045, 0.033, 0.015]) + pad_cells * res
    dims = np.round((hi - lo) / res).astype(int) + 1
    gi, gj, gk = np.meshgrid(np.arange(dims[0]), np.arange(dims[1]), np.arange(dims[2]), indexing="ij")
    P = lo[None, None, None, :] + res * np.stack([gi, gj, gk], -1)

    def build(parts):
        sd = np.min(np.stack([_hexa_sdf(P, C) for C in parts], 0), 0)
        Vs, Fs, off = [], [], 0
        for C in parts:
            V, F = _hexa_mesh(C, n)
            Vs.append(V); Fs.append(F + off); off += V.shape[0]
        return {"V": np.concatenate(Vs), "F": np.concatenate(Fs).astype(np.int32),
                "sdf": sd.astype(np.float32), "origin": lo.astype(np.float32), "res": np.float32(res)}

    gig = np.eye(4)
    gig[0, 3] = -0.035
    return {"open": build([palm, f1, f2]), "enclosed": build([palm, f1, f2, gap]), "gripper_in_grasp": gig}


def sample_lattice_nut(n, seed=0, origin=(-0.012, -0.011, 0.70), spacing=0.001):
    """A tilted hex nut snapped to a 1 mm lattice whose largest extent spans exactly LATTICE_LEVELS positions, in the
    camera frame (z ~ 0.7 m): returns (cloud_xyz (n,3) f64, cloud_normal (n,3) f64 with float32-representable values,
    lattice indices g (n,3) uint8).  Its min/max-normalised coordinates are 0.04*g (see make_lattice_seg_state_dict)."""
    rng = np.random.RandomState(seed)
    pts, nrm = sample_hex_nut(n, rng, across_flats=0.020, height=0.008, bore=0.010)
    R = _rot_x(np.deg2rad(25.0))
    pts = pts @ R.T
    nrm = nrm @ R.T
    lo = pts.min(0)
    step = (pts.max(0) - lo).max() / (LATTICE_LEVELS - 1)
    g = np.rint((pts - lo) / step).astype(np.int64)
    g -= g.min(0)
    assert g.max() == LATTICE_LEVELS - 1
    xyz = np.asarray(origin, np.float64)[None] + spacing * g.astype(np.float64)
    nrm = nrm.astype(np.float32).astype(np.float64)
    return xyz, nrm, g.astype(np.uint8)


def make_filter_case(seed, G, S, scale=(1, 1, 1), n_points=2400):
    """A sparse pile; the grasp target is object 3: its points feed the open-gripper check, all other
    points the enclosed (swept-volume) check; the canonical frame is the target's own frame, so the
    symmetry transforms spin the candidates about the object like Utils.py:79-84."""
    rng = np.random.RandomState(seed)
    scene = make_pile(n_points, n_objects=6, seed=seed)
    obj = scene["object_id"] == 3
    p1, p2 = scene["cloud_xyz"][obj], scene["cloud_xyz"][~obj]
    poses = make_candidates(p1, scene["cloud_normal"][obj], G, seed=seed + 1)
    sym = []
    for k in range(S):                                      # nut symmetry set (Utils.py:79-84)
        T = np.eye(4)
        a = k * np.pi / 3
        T[:3, :3] = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        if k >= 6:
            T[:3, :3] = T[:3, :3] @ np.diag([1, -1, -1])
        sym.append(T)
    nocs_pose = scene["object_poses"][3].copy()
    nocs_pose[:3, :3] = nocs_pose[:3, :3] @ np.diag(scale)   # 9-DoF pose: rotation x per-axis scale
    canonical_to_nocs = np.eye(4)
    canonical_to_nocs[:3, 3] = rng.normal(0, 0.0005, 3)
    inv = np.linalg.inv(nocs_pose @ canonical_to_nocs)
    poses_can = np.stack([inv @ p for p in poses])          # canonical_to_cam * pose_can == the camera-frame pose
    g = make_gripper_proxy()
    return p1, p2, poses_can, np.stack(sym), nocs_pose, canonical_to_nocs, g


def make_mlp_state_dict(dims, seed=0, conv2d=True):
    """Seeded weights of a PointNet++ shared-MLP stack in the upstream module layout: mlp_convs.{i} (Conv2d/Conv1d k=1)
    + mlp_bns.{i} with randomised running statistics (same ranges as make_state_dict)."""
    import torch
    rng = np.random.RandomState(seed)
    sd = OrderedDict()
    for i in range(len(dims) - 1):
        cin, cout = dims[i], dims[i + 1]
        bound = 1.0 / np.sqrt(cin)
        shp = (cout, cin, 1, 1) if conv2d else (cout, cin, 1)
        sd[f"mlp_convs.{i}.weight"] = rng.uniform(-bound, bound, size=shp).astype(np.float32)
        sd[f"mlp_convs.{i}.bias"] = rng.uniform(-bound, bound, size=(cout,)).astype(np.float32)
        sd[f"mlp_bns.{i}.weight"] = rng.uniform(0.5, 1.5, size=(cout,)).astype(np.float32)
        sd[f"mlp_bns.{i}.bias"] = rng.normal(0, 0.1, size=(cout,)).astype(np.float32)
        sd[f"mlp_bns.{i}.running_mean"] = rng.normal(0, 0.2, size=(cout,)).astype(np.float32)
        sd[f"mlp_bns.{i}.running_var"] = rng.uniform(0.5, 1.5, size=(cout,)).astype(np.float32)
    return OrderedDict((k, torch.from_numpy(v)) for k, v in sd.items())


# camera of the reference's shipped config (config.yml:1-3): 2064 x 1544 pixels
REF_CAMERA_K = np.array([[2257.7500557850776, 0, 1032], [0, 2257.4882391629421, 772], [0, 0, 1]], dtype=np.float64)
REF_CAMERA_HW = (1544, 2064)


def make_depth_scene(H, W, K, seed=0, floor_z=0.70, n_spheres=3, n_boxes=3):
    """Ray-cast depth image (H,W) float32 in metres of a bin floor at camera z = floor_z with a few spheres and
    axis-aligned boxes resting on it, seen by a pinhole camera K at the origin looking along +z.  Curved surfaces,
    flat faces and occlusion edges at any resolution (up to the reference camera's 2064 x 1544)."""
    rng = np.random.RandomState(seed)
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    v, u = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    dx = (u - K[0, 2]) / K[0, 0]                     # ray direction (dx, dy, 1): the hit's depth is its parameter t
    dy = (v - K[1, 2]) / K[1, 1]
    depth = np.full((H, W), floor_z)
    half = 0.6 * floor_z * min(K[0, 2] / K[0, 0], K[1, 2] / K[1, 1])   # objects stay inside the field of view
    for _ in range(n_spheres):
        R = rng.uniform(0.012, 0.030)
        c = np.array([rng.uniform(-half, half), rng.uniform(-half, half), floor_z - R])
        dd = dx * dx + dy * dy + 1.0
        b = dx * c[0] + dy * c[1] + c[2]
        disc = b * b - dd * (c @ c - R * R)
        hit = disc >= 0
        t = np.where(hit, (b - np.sqrt(np.where(hit, disc, 0.0))) / dd, np.inf)
        depth = np.minimum(depth, t)
    for _ in range(n_boxes):
        size = rng.uniform(0.015, 0.045, size=3)
        ctr = np.array([rng.uniform(-half, half), rng.uniform(-half, half)])
        lo = np.array([ctr[0] - size[0] / 2, ctr[1] - size[1] / 2, floor_z - size[2]])
        hi = np.array([ctr[0] + size[0] / 2, ctr[1] + size[1] / 2, floor_z])
        tmin = np.zeros((H, W))
        tmax = np.full((H, W), np.inf)
        for d, a in ((dx, 0), (dy, 1), (np.ones((H, W)), 2)):
            with np.errstate(divide="ignore", invalid="ignore"):
                t1 = (lo[a] - 0.0) / d
                t2 = (hi[a] - 0.0) / d
            inside = (lo[a] <= 0.0) & (0.0 <= hi[a])
            t1 = np.where(d == 0, np.where(inside, -np.inf, np.inf), t1)
            t2 = np.where(d == 0, np.where(inside, np.inf, -np.inf), t2)
            tmin = np.maximum(tmin, np.minimum(t1, t2))
            tmax = np.minimum(tmax, np.maximum(t1, t2))
        t = np.where(tmin <= tmax, tmin, np.inf)
        depth = np.minimum(depth, t)
    return depth.astype(np.float32)
