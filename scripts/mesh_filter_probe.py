"""Throughput of the mesh-vs-voxel collision predicate (COLLISION_PREDICATE = "mesh", csrc/cg_mesh_collide.cu) next to
the gripper-SDF predicate, on one GPU, in one run:

  (a) the K2 filter workload as bench.py builds it (20 000-pt pile, 4 096 cone candidates, pose adjustment on),
  (b) make_filter_case(43, 4096, 1) (mixed verdicts, no approach filter, no adjustment), plus the agreement of the
      mesh verdicts with the "sdf" and "voxel" predicates there (the device counterpart of r2_x2_agreement.json),
  (c) a K5-sized object-only run: ~1 M device-enumerated cone poses, adjustment off, no background,

each with the 36-triangle box proxy and the ~21 k-triangle dense proxy, plus cg_mesh_create / cg_voxels_create_dev
times.  Filter rates are CUDA-event timings over windows of at least one second with resident inputs (poses, voxel
sets, SDFs already on the device).

    python scripts/mesh_filter_probe.py [--out profiles/r4_mesh_filter.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
RES = 0.0005


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def rate(fn, pairs, min_s=1.0):
    """pairs per second of fn() over a CUDA-event window of >= min_s seconds (after one warm-up call)."""
    import torch
    fn()
    torch.cuda.synchronize()
    n, ms = 1, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000.0 * min_s:
            break
        n = max(n * 2, int(n * 1000.0 * min_s / max(ms, 1e-3) * 1.2))
    return {"pairs_per_s": pairs * n / (ms / 1e3), "ms_per_call": ms / n, "calls": n, "window_s": ms / 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_mesh_filter.json"))
    a = ap.parse_args()
    import torch
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.grasp_sampler import cone_frames, enumerate_poses
    from catgrasp_b200.mesh import GripperMesh, VoxelSet
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import (make_candidates, make_dense_gripper_proxy, make_filter_case, make_gripper_proxy,
                                         make_pile)
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    up = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)      # noqa: E731
    eye = np.eye(4)
    out = {"card": card(), "resolution_m": RES, "window": ">= 1 s of CUDA-event time per number, resident inputs"}

    proxies = {"box": make_gripper_proxy(), "dense": make_dense_gripper_proxy()}
    handles, create = {}, {}
    for name, g in proxies.items():
        h = {}
        for part in ("open", "enclosed"):
            torch.cuda.synchronize()
            t = time.perf_counter()
            h["mesh_" + part] = GripperMesh(g[part]["V"], g[part]["F"])
            dt = time.perf_counter() - t
            dims, cell, entries = h["mesh_" + part].info()
            create[f"cg_mesh_create_{name}_{part}"] = {"ms": dt * 1e3, "triangles": int(len(g[part]["F"])), "grid": dims,
                                                       "cell_m": cell, "entries": entries}
            h["sdf_" + part] = Sdf3D(g[part]["sdf"], g[part]["origin"], g[part]["res"])
        handles[name] = h
    out["create"] = create

    def run_pair(label, poses_d, sym, nocs_pose, c2n, p1, p2, fdir, adjust):
        d1, d2 = up(p1), up(p2)
        torch.cuda.synchronize()
        t = time.perf_counter()
        v1 = VoxelSet(d1, RES)
        v2 = VoxelSet(d2, RES)
        vox_ms = (time.perf_counter() - t) * 1e3
        Q = poses_d.shape[0] * len(sym)
        res = {"pairs": Q, "object_points": len(p1), "background_points": len(p2), "object_voxels": len(v1),
               "background_voxels": len(v2), "cg_voxels_create_dev_ms_both": vox_ms}
        for name, h in handles.items():
            g = proxies[name]
            f_mesh = lambda: my_cpp.filter_grasp_pose_mesh_raw(poses_d, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir,   # noqa: E731
                                                               adjust, h["mesh_open"], v1, h["mesh_enclosed"], v2, RES)
            f_sdf = lambda: my_cpp.filter_grasp_pose_raw(poses_d, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust,   # noqa: E731
                                                         h["sdf_open"], d1, h["sdf_enclosed"] if len(p2) else None, d2)
            r_mesh, r_sdf = rate(f_mesh, Q), rate(f_sdf, Q)
            st_m = f_mesh()[0].cpu().numpy()
            st_s = f_sdf()[0].cpu().numpy()
            res[name] = {"mesh": r_mesh, "sdf": r_sdf, "mesh_over_sdf_time": r_sdf["pairs_per_s"] / r_mesh["pairs_per_s"],
                         "accepted_mesh": int((st_m == 0).sum()), "accepted_sdf": int((st_s == 0).sum())}
            print(label, name, json.dumps(res[name]), flush=True)
        return res, (v1, v2, d1, d2)

    # (a) K2 filter workload (bench.py make_scene_job, config K2, rank 0)
    scene = make_pile(20000, n_objects=12, seed=0)
    obj = scene["object_id"] == 3
    if obj.sum() < 64:
        obj = scene["object_id"] == np.bincount(scene["object_id"]).argmax()
    poses = make_candidates(scene["cloud_xyz"][obj], scene["cloud_normal"][obj], 4096, seed=1)
    out["a_k2"], _ = run_pair("a_k2", up(poses), eye[None], eye, eye, scene["cloud_xyz"][obj], scene["cloud_xyz"][~obj],
                              True, True)

    # (b) make_filter_case(43, 4096, 1) + agreement of the three predicates
    p1, p2, poses, sym, nocs_pose, c2n, gbox = make_filter_case(43, 4096, 1)
    pd = up(poses)
    out["b_filter_case"], (v1, v2, d1, d2) = run_pair("b_filter_case", pd, sym, nocs_pose, c2n, p1, p2, False, False)
    h = handles["box"]
    mesh = my_cpp.filter_grasp_pose_mesh_raw(pd, sym, nocs_pose, c2n, gbox["gripper_in_grasp"], False, False, h["mesh_open"],
                                             v1, h["mesh_enclosed"], v2, RES)[0].cpu().numpy() == 3
    agree = {"workload": "make_filter_case(43, 4096, 1), box proxy, no approach filter, no adjustment, 0.5 mm voxels",
             "mesh_hits": int(mesh.sum())}
    for name, margin in (("sdf", 0.0), ("voxel", my_cpp.voxel_margin(RES))):
        v = my_cpp.filter_grasp_pose_raw(pd, sym, nocs_pose, c2n, gbox["gripper_in_grasp"], False, False, h["sdf_open"], d1,
                                         h["sdf_enclosed"], d2, sdf_margin=margin)[0].cpu().numpy() == 3
        agree[name] = {"agreement": float((v == mesh).mean()), "predicate_only_hits": int((v & ~mesh).sum()),
                       "mesh_only_hits": int((~v & mesh).sum()), "hits": int(v.sum())}
    out["b_agreement"] = agree
    print("agreement", json.dumps(agree), flush=True)

    # (c) K5-sized object-only run (bench.py run_k5: 10 000-pt single object, cone enumeration on the device)
    sc = make_pile(10000, n_objects=1, seed=0)
    pts, nrm = sc["cloud_xyz"], sc["cloud_normal"]
    hand_depth, step, n_dir = 0.042, 0.003, 30
    per_sample = (1 + n_dir * 6) * len(np.arange(0, hand_depth, step))
    np.random.seed(0)
    ids, R0s, sphere = cone_frames(pts.copy(), nrm.copy(), max_num_samples=-(-(1 << 20) // per_sample), n_sphere_dir=n_dir)
    _, p32 = enumerate_poses(pts[ids], R0s, sphere, hand_depth, step, 0.01, device=0)
    out["c_k5_object_only"], _ = run_pair("c_k5", p32, eye[None], eye, eye, pts, np.zeros((0, 3)), True, False)

    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
