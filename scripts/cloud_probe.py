"""Time the point-cloud front end (catgrasp_b200/cloud.py) on one GPU against the host path on the same inputs.

Device times: CUDA events around a warm loop whose timed region is >= 1 s.  Host times: scipy cKDTree plus the numpy
restatement (tests/cloud_oracle.py) -- what a user without this project runs minus open3d, which is not installed
and is not timed.  Inputs: the reference camera's full 2064 x 1544 synthetic depth scene, its 1 mm voxel scene, and
object crops of 5 k / 20 k / 50 k points.  Writes one JSON file (default profiles/r3_cloud_frontend.json).

    python scripts/cloud_probe.py [--out PATH] [--min-seconds 1.0]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.spatial import cKDTree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cloud_oracle as ref   # noqa: E402

from catgrasp_b200 import cloud, synthetic   # noqa: E402

GRIPPER_HALF = 0.085 / 2


def dev_time(fn, min_s):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    one = max(a.elapsed_time(b) / 1e3, 1e-6)
    reps = max(1, int(np.ceil(min_s / one)))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return {"ms": a.elapsed_time(b) / reps, "reps": reps, "region_s": a.elapsed_time(b) / 1e3}


def host_time(fn, min_s):
    t0 = time.perf_counter()
    fn()
    one = time.perf_counter() - t0
    reps = max(1, int(np.ceil(min_s / max(one, 1e-6)))) if one < min_s else 1
    if reps == 1 and one >= min_s:
        return {"ms": one * 1e3, "reps": 1, "region_s": one}
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    el = time.perf_counter() - t0
    return {"ms": el / reps * 1e3, "reps": reps, "region_s": el}


def crop(pts, n, seed=0):
    """The n scene points nearest (in x, y) to a seeded above-floor point: one object-sized crop."""
    rng = np.random.RandomState(seed)
    above = np.nonzero(pts[:, 2] < 0.699)[0]
    c = pts[above[rng.randint(len(above))]]
    return pts[np.argsort(np.linalg.norm(pts[:, :2] - c[:2], axis=1), kind="stable")[:n]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_cloud_frontend.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "cloud_probe measures on a GPU"
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "host_threads": os.cpu_count(), "rows": []}
    H, W = synthetic.REF_CAMERA_HW
    depth = synthetic.make_depth_scene(H, W, synthetic.REF_CAMERA_K, seed=0)
    K = synthetic.REF_CAMERA_K
    xyz = ref.depth2xyzmap(depth, K)
    full = xyz[xyz[:, :, 2] >= 0.1].reshape(-1, 3).astype(np.float64)
    scene1, _ = ref.voxel_down_sample(full, 0.001)
    full_d = torch.as_tensor(full, device=dev)
    scene1_d = torch.as_tensor(scene1, device=dev)
    depth_d = torch.as_tensor(depth, device=dev)
    ms = a.min_seconds

    def row(name, n, dfn, hfn):
        r = {"name": name, "n": int(n), "device": dev_time(dfn, ms), "host": host_time(hfn, ms)}
        r["speedup"] = r["host"]["ms"] / r["device"]["ms"]
        res["rows"].append(r)
        print(f"{name:40s} n={n:>8d}  device {r['device']['ms']:9.3f} ms  host {r['host']['ms']:10.1f} ms  x{r['speedup']:.0f}",
              flush=True)

    row("depth2xyzmap 2064x1544", H * W, lambda: cloud.depth2xyzmap(depth_d, K), lambda: ref.depth2xyzmap(depth, K))
    row("normals r=2mm nn=30 (full scan)", len(full), lambda: cloud.estimate_normals(full_d, 0.002, 30),
        lambda: ref.normals_from_neighbors(full, ref.hybrid_neighbors(cKDTree(full), full, 0.002, 30)[1]))
    row("voxel 1mm (full scan)", len(full), lambda: cloud.voxel_down_sample(full_d, 0.001),
        lambda: ref.voxel_down_sample(full, 0.001))
    row("normals r=3mm nn=30 (1mm scene)", len(scene1), lambda: cloud.estimate_normals(scene1_d, 0.003, 30),
        lambda: ref.normals_from_neighbors(scene1, ref.hybrid_neighbors(cKDTree(scene1), scene1, 0.003, 30)[1]))
    rng = np.random.RandomState(1)
    for n in (5000, 20000, 50000):
        ob = crop(full, n)
        ob_n = ref.correct_pcd_normal_direction(ob, rng.normal(size=ob.shape))
        ob_d, obn_d = torch.as_tensor(ob, device=dev), torch.as_tensor(ob_n, device=dev)
        down, _ = ref.voxel_down_sample(ob, 0.0005)
        down_d = torch.as_tensor(down, device=dev)
        bg = scene1[ref.any_within(ob, scene1, GRIPPER_HALF)]
        bg_d = torch.as_tensor(bg, device=dev)
        row(f"voxel 0.5mm (object {n})", n, lambda: cloud.voxel_down_sample(ob_d, 0.0005),
            lambda: ref.voxel_down_sample(ob, 0.0005))
        row(f"nearest voxel->object ({n})", len(down), lambda: cloud.CloudIndex(ob_d, 0.0005).query(down_d),
            lambda: cKDTree(ob).query(down))
        row(f"crop dist<=d/2 1mm scene ({n})", len(scene1), lambda: cloud.CloudIndex(ob_d, 0.005).any_within(scene1_d, GRIPPER_HALF),
            lambda: ref.any_within(ob, scene1, GRIPPER_HALF))
        row(f"cloudA_minus_cloudB ({n})", len(bg), lambda: cloud.cloudA_minus_cloudB(bg_d, ob_d, 0.005),
            lambda: ref.cloudA_minus_cloudB(bg, ob, 0.005))

        def dev_chain():
            d, _ = cloud.voxel_down_sample(ob_d, 0.0005)
            _, i = cloud.CloudIndex(ob_d, 0.0005).query(d)
            od, ond = ob_d[i], obn_d[i]
            near = cloud.CloudIndex(ob_d, 0.005).any_within(scene1_d, GRIPPER_HALF)
            b, _ = cloud.cloudA_minus_cloudB(scene1_d[near], ob_d, 0.005)
            cloud.voxel_down_sample(b, 0.001)
            vs = float(torch.linalg.norm(od.max(0).values - od.min(0).values)) / 10.0
            return cloud.voxel_down_sample(od, vs, normals=ond)

        def host_chain():
            d, _ = ref.voxel_down_sample(ob, 0.0005)
            _, i = cKDTree(ob).query(d)
            od, ond = ob[i], ob_n[i]
            b, _ = ref.cloudA_minus_cloudB(scene1[ref.any_within(ob, scene1, GRIPPER_HALF)], ob, 0.005)
            ref.voxel_down_sample(b, 0.001)
            return ref.voxel_down_sample(od, np.linalg.norm(od.max(0) - od.min(0)) / 10.0, ond)

        row(f"object chain :113-139+:171-175 ({n})", n, dev_chain, host_chain)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out, "|", res["gpu"], "|", res["nvidia_smi"])


if __name__ == "__main__":
    main()
