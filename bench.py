#!/usr/bin/env python
"""bench.py -- candidate grasps scored / second on the BASELINE.json configurations.

A "pass" scores every candidate of the configuration once: one grasp-Q PointNet forward on an n_pts-point subset of
the scene (fused per-candidate transform + softmax) AND one collision verdict (pose logic + gripper-SDF predicate over
object / background points) per candidate, plus one NUNOCS forward (8192 points) per scene.  A "step" is
`passes_per_step` back-to-back passes (chosen during warm-up so that the timed region lasts >= ~1 s; it is printed in
`config`), `value` = candidates scored / second over all ranks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config K1|K2|K3|K4|K5]
                    [--dump-outputs DIR]

Default configuration by GPU count (BASELINE.json `configs`):
    --gpus 1 -> K2  nut clutter pile, 20 000-pt scene, 4 096 candidates                       (weak when forced at N > 1)
    --gpus 2 -> K3  screw clutter pile, 40 000-pt scene, 16 384 candidates sharded by dist.shard_range
    --gpus 4/8 -> K4  8 scenes x 20 000 pts, 65 536 candidates, scenes dealt round-robin to the ranks
    --config K5     offline path (generate_grasp.py:81-97): cone pose enumeration on the device -> collision filter
                    (adjust_collision_pose off) -> grasp-Q on the survivors; ~1 M candidates over all ranks
N > 1 is launched by torchrun (one rank per GPU); no data-path collective, one NCCL all-gather of the 48-byte result
records per pass.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the timed path returned in its last pass as DIR/<name>.npy (see dump_outputs).  The
inputs are synthetic and seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_CAND = {1024: 880045568, 2048: 1754052096}     # SURVEY.md 8(d), exact from layer hooks on the reference
# MACs per point of the three fused trunk kernels (6*64 + [64*64] + 64*128 + 128*1024), SURVEY.md 8a N3-N5
TRUNK_MAC_PER_PT = [6 * 64 + 64 * 128 + 128 * 1024,            # STN3d trunk
                    6 * 64 + 64 * 64 + 64 * 128 + 128 * 1024,  # conv1 + STNkd trunk
                    6 * 64 + 64 * 64 + 64 * 128 + 128 * 1024]  # conv1 + @T64 + conv2 + conv3
ENGINE_NAMES = ["fp32-simt", "tcgen05-bf16x3", "tcgen05-f16x2", "tcgen05-f16x1-persistent"]
ENGINE_DTYPES = ["f32", "f32 (bf16 hi/lo x3 on tcgen05, f32 accumulate)", "f32 (f16 hi/lo x2 on tcgen05, f32 accumulate)",
                 "f32 (128->1024 layer f16 x f16 single pass on tcgen05, f32 accumulate; other layers bf16 hi/lo x3)"]
CONFIGS = {
    "K1": dict(name="K1 nut: single-object 1024-pt crop, 64 candidates", scenes=1, scene_pts=1024, total=64, objects=1),
    "K2": dict(name="K2 nut clutter pile: 20000-pt scene, 4096 candidates", scenes=1, scene_pts=20000, total=4096, objects=12),
    "K3": dict(name="K3 screw clutter pile: 40000-pt scene, 16384 candidates sharded across the ranks", scenes=1,
               scene_pts=40000, total=16384, objects=8),
    "K4": dict(name="K4 mixed-category batch: 8 scenes x 20000 pts, 65536 candidates", scenes=8, scene_pts=20000,
               total=65536, objects=12),
    "K5": dict(name="K5 offline generate_grasp path: cone enumeration -> collision filter -> grasp-Q on survivors", scenes=1,
               scene_pts=10000, total=1 << 20, objects=1),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS), help="default: K2 / K3 / K4 for 1 / 2 / >=4 GPUs")
    ap.add_argument("--n-pts", type=int, default=1024, help="points per candidate (config_grasp.yml n_pts)")
    ap.add_argument("--nunocs-pts", type=int, default=8192)
    ap.add_argument("--engine", type=int, default=None, help="0 fp32 SIMT, 1 tcgen05 3-pass bf16, 2 tcgen05 2-pass fp16, "
                    "3 persistent tcgen05 1-pass fp16 (default: library default = 3)")
    ap.add_argument("--passes-per-step", type=int, default=0, help="0 = calibrate so that the timed region is ~1.2 s")
    ap.add_argument("--cpu-sample", type=int, default=192, help="candidates in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api-leg", action="store_true", help="skip the e2e_api leg (GraspPredicter.predict_batch wall clock)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed pass to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.config is None:
        args.config = "K2" if args.gpus == 1 else ("K3" if args.gpus == 2 else "K4")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_MAX_ROWS = 1 << 16
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as <out_dir>/<name>.npy: float64 stays float64, everything else (probabilities, labels, status
    and offset codes, poses, NOCS coordinates and bins) becomes float32, which holds each of those integer codes exactly.
    An array with more than DUMP_MAX_ROWS rows keeps a fixed sample of rows (seeded, so the same rows every run for the
    same length), listed in <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.shape[0] > DUMP_MAX_ROWS:
            rows = np.sort(np.random.RandomState(0).choice(a.shape[0], DUMP_MAX_ROWS, replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
            total += rows.size * 8
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        total += a.nbytes
    assert total <= DUMP_MAX_BYTES, f"dumped {total} bytes, more than {DUMP_MAX_BYTES}"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ workload
def scene_assignment(cfg_name, rank, world):
    """Which scenes a rank works on and which candidates of each: [(scene_index, lo, hi, total_in_scene)]."""
    from catgrasp_b200.dist import shard_range
    c = CONFIGS[cfg_name]
    per_scene = c["total"] // c["scenes"]
    if cfg_name == "K2":                       # weak when forced at N > 1: every rank its own 4096 candidates
        return [(0, 0, per_scene, per_scene)]
    if c["scenes"] == 1:                       # K1 / K3: one scene, candidates sharded contiguously
        lo, hi = shard_range(per_scene, rank, world)
        return [(0, lo, hi, per_scene)]
    if world <= c["scenes"]:                   # K4: scenes dealt round-robin
        return [(s, 0, per_scene, per_scene) for s in range(c["scenes"]) if s % world == rank]
    out = []                                   # more ranks than scenes: shard inside the scene
    per = world // c["scenes"]
    s, r = rank // per, rank % per
    if s < c["scenes"]:
        lo, hi = shard_range(per_scene, r, per)
        out.append((s, lo, hi, per_scene))
    return out


def make_scene_job(cfg_name, scene_index, lo, hi, total, args, rank):
    """Host arrays of one scene's share of the work (synthetic; SURVEY.md 8d)."""
    from catgrasp_b200.synthetic import make_candidates, make_pile
    c = CONFIGS[cfg_name]
    M = c["scene_pts"]
    seed = {"K1": 3, "K2": 0, "K3": 1, "K4": 10 + scene_index, "K5": 0}[cfg_name]
    scene = make_pile(M, n_objects=c["objects"], seed=seed)
    ids_obj = scene["object_id"]
    target = 3 if c["objects"] > 3 else 0
    obj = ids_obj == target
    if obj.sum() < 64:
        obj = ids_obj == np.bincount(ids_obj).argmax()
    pose_seed = 1 + (rank if cfg_name == "K2" else 0) + 100 * scene_index
    poses = make_candidates(scene["cloud_xyz"][obj], scene["cloud_normal"][obj], total, seed=pose_seed)[lo:hi]
    rng = np.random.RandomState(100 + rank + 17 * scene_index)
    B = hi - lo
    n_pts = args.n_pts
    # per-candidate subsets like dataset_grasp.py:72-73 (without replacement when M >= n_pts)
    if M >= n_pts:
        ids = np.stack([rng.permutation(M)[:n_pts] for _ in range(B)]).astype(np.int32) if B else np.zeros((0, n_pts), np.int32)
    else:
        ids = rng.randint(0, M, size=(B, n_pts)).astype(np.int32)
    oxyz, onrm = scene["cloud_xyz"][obj], scene["cloud_normal"][obj]
    sel = rng.randint(0, oxyz.shape[0], size=args.nunocs_pts)
    x = oxyz[sel]
    x = (x - x.min(0)) / ((x.max(0) - x.min(0)).max() + 1e-15)
    nun_in = np.concatenate([x, onrm[sel]], -1).astype(np.float32)
    return {"scene": scene, "obj": obj, "poses": poses, "ids": ids, "nun_in": nun_in, "B": B, "M": M,
            "open_pts": oxyz.astype(np.float32), "bg_pts": scene["cloud_xyz"][~obj].astype(np.float32)}


def normalizer():
    norm = np.random.RandomState(7)
    mean = np.concatenate([norm.normal(0, 0.002, 3), norm.normal(0, 0.05, 3)])
    std = np.concatenate([norm.uniform(0.008, 0.012, 3), norm.uniform(0.5, 0.6, 3)])
    return mean, std


def workload_config(args, passes=None, world=None):
    c = CONFIGS[args.config]
    world = world or args.gpus
    per_gpu = c["total"] if args.config == "K2" else c["total"] // max(world, 1)
    d = {"workload": f"{c['name']}; n_pts={args.n_pts} per candidate; per pass: grasp-Q PointNetCls + SDF collision "
                     f"(5 lateral offsets, trilinear) per candidate + 1 NUNOCS PointNetSeg forward ({args.nunocs_pts} pts) per scene",
         "config": args.config, "scenes": c["scenes"], "scene_pts": c["scene_pts"], "n_pts": args.n_pts,
         "candidates_total": c["total"] * (world if args.config == "K2" else 1), "candidates_per_gpu": per_gpu,
         "l2": "flushed between timed passes (256 MiB write)",
         "parallelism": ("candidate-shard" if c["scenes"] == 1 else "scene round-robin") + f" x{world}",
         "streams": "single stream"}
    if passes is not None:
        d["passes_per_step"] = passes
    return d


# ------------------------------------------------------------------------------------------------ CPU arm
def pick_torch_threads(sd_cls, n_pts):
    """Quick sweep (a few hundred ms): torch intra-op thread count at which the reference network's forward is fastest
    on this host (the small conv1d / linear ops stop scaling long before all cores of a 128-core host are busy)."""
    import torch
    from oracle.pointnet_ref import pointnet_cls_forward
    x = np.random.RandomState(0).normal(0, 1, (24, n_pts, 6)).astype(np.float32)
    best, best_t = 8, 1e9
    ncpu = os.cpu_count() or 8
    for th in [t for t in (8, 16, 32, 64, 128) if t <= ncpu] or [ncpu]:
        torch.set_num_threads(th)
        pointnet_cls_forward(sd_cls, x)
        t0 = time.perf_counter()
        pointnet_cls_forward(sd_cls, x)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = th, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_pass(job, args, n_cand, sd_cls, sd_seg, mean, std, gripper, with_nunocs=True):
    """The reference's CPU path for n_cand candidates: per-candidate numpy transform loop + PointNetCls in
    micro-batches of 200 (predicter.py:67-94), C collision oracle with OpenMP, and (optionally) NUNOCS
    forwards (the first one is a warm-up, the second is the one timed)."""
    from oracle import filter_ref
    from oracle.transforms_ref import nunocs_predict, predict_batch
    scene = job["scene"]
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    cfg = {"n_pts": args.n_pts, "mean": mean, "std": std}
    t0 = time.perf_counter()
    predict_batch(sd_cls, cfg, data, job["poses"][:n_cand])
    t1 = time.perf_counter()
    eye = np.eye(4)
    # The C collision oracle runs on the same OpenMP runtime as torch.  With one OpenMP team of all 128 host cores every
    # later torch region of the process slowed down 4-30x (round 1 measured its NUNOCS forward right after such a region:
    # 5 s instead of ~0.2 s); the collision share is ~0.02 s per step either way, so it uses torch's thread count.
    import torch
    filter_ref.filter_ref(job["poses"][:n_cand], [eye], eye, eye, gripper["gripper_in_grasp"], True, True, 0, gripper["open"],
                          job["open_pts"], gripper["enclosed"], job["bg_pts"], nthreads=torch.get_num_threads())
    t2 = time.perf_counter()
    nun = 0.0
    if with_nunocs:
        ncfg = {"n_pts": args.nunocs_pts, "ce_loss_bins": 100}
        o = job["obj"]
        d = {"cloud_xyz": scene["cloud_xyz"][o], "cloud_normal": scene["cloud_normal"][o]}
        nunocs_predict(sd_seg, ncfg, dict(d))            # cold (first torch conv at this shape)
        t3 = time.perf_counter()
        nunocs_predict(sd_seg, ncfg, dict(d))            # warm: this is the one reported
        nun = time.perf_counter() - t3
    return {"net_s": t1 - t0, "collision_s": t2 - t1, "nunocs_s": nun}


def cpu_rate(r, n, cands_per_nunocs):
    """candidates/s of the CPU arm with the per-scene NUNOCS forward amortised like in the GPU pass."""
    return n / (r["net_s"] + r["collision_s"] + r["nunocs_s"] * n / cands_per_nunocs)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.  The reference is
    a script collection without an installer and my_cpp needs FCL/octomap, so the arm runs the pinned oracle PORT
    (oracle/: torch-CPU restatement of pointnet2.py + numpy transforms + C/OpenMP filter), each step a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from catgrasp_b200.synthetic import make_gripper_proxy, make_state_dict
    sd_cls, sd_seg = make_state_dict("cls", 10, seed=0), make_state_dict("seg", 300, seed=1)
    sc, lo, hi, tot = scene_assignment(args.config, 0, 1)[0]
    cap = min(tot, 512)
    job = make_scene_job(args.config, sc, 0, cap, tot, args, 0)
    mean, std = normalizer()
    g = make_gripper_proxy()
    th = pick_torch_threads(sd_cls, args.n_pts)
    per_scene = CONFIGS[args.config]["total"] // CONFIGS[args.config]["scenes"]
    n = max(16, min(args.cpu_sample, cap) // 2)
    r0 = cpu_reference_pass(job, args, n, sd_cls, sd_seg, mean, std, g, with_nunocs=True)    # warm-up; times NUNOCS warm
    nun_s = r0["nunocs_s"]
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        cpu_reference_pass(job, args, n, sd_cls, sd_seg, mean, std, g, with_nunocs=False)
    tot_s = {"net_s": 0.0, "collision_s": 0.0}
    for _ in range(args.steps):
        r = cpu_reference_pass(job, args, n, sd_cls, sd_seg, mean, std, g, with_nunocs=False)
        tot_s["net_s"] += r["net_s"]; tot_s["collision_s"] += r["collision_s"]
    dt = tot_s["net_s"] + tot_s["collision_s"] + nun_s * (n * args.steps) / per_scene
    v = n * args.steps / dt
    cores = os.cpu_count()
    sample = (f"{n} of {per_scene} candidates per step on a {job['M']}-pt scene (net {tot_s['net_s'] / args.steps:.2f} s, collision "
              f"{tot_s['collision_s'] / args.steps:.3f} s per step); warm NUNOCS forward ({nun_s:.2f} s) amortised 1 per {per_scene} "
              f"candidates; torch threads {th} (picked by a sweep), OpenMP collision threads {th}; PORT of the reference "
              f"(oracle/), not its own binaries; context: the reference's pointnet2.PointNetCls itself ran 134 cand/s on 8 cores "
              f"in the survey container (BASELINE.md section 2)")
    line = {"impl": "reference", "metric": "candidate grasps scored/sec", "value": v, "unit": "candidates/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak" if args.config == "K2" else "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args),
            "cpu_baseline": {"value": v, "unit": "candidates/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ e2e_api leg
def api_leg(dev_index, n_pts):
    """Wall clock of the calls a reference user makes: GraspPredicter.predict_batch(data, poses) with the subset draw
    INSIDE (both modes) at a 3 000-pt crop and a 20 000-pt scene, and NunocsPredicter.predict_nocs."""
    import contextlib
    import io
    from catgrasp_b200.predicter import GraspPredicter, NunocsPredicter
    from catgrasp_b200.synthetic import make_candidates, make_pile, write_artifacts
    out = {"predict_batch": []}
    with tempfile.TemporaryDirectory() as td:
        adir = write_artifacts(os.path.join(td, "artifacts-47"), "cls", n_pts=n_pts, seed=0)
        ndir = write_artifacts(os.path.join(td, "artifacts-78"), "seg", n_pts=8192, seed=1)
        with contextlib.redirect_stdout(io.StringIO()):
            gp = GraspPredicter("nut", artifact_dir=adir, device=dev_index)
            npred = NunocsPredicter("nut", artifact_dir=ndir, device=dev_index)
        for M, B in ((3000, 1024), (20000, 4096)):
            scene = make_pile(M, n_objects=4 if M < 10000 else 12, seed=5)
            data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
            poses = list(make_candidates(scene["cloud_xyz"], scene["cloud_normal"], B, seed=6))
            for mode in ("host", "device"):
                np.random.seed(0)
                gp.predict_batch(data, poses, subsample=mode)                       # warm-up (allocations, pinned buffer)
                reps = 3
                t0 = time.perf_counter()
                for _ in range(reps):
                    res = gp.predict_batch(data, poses, subsample=mode)
                dt = (time.perf_counter() - t0) / reps
                assert len(res) == B
                out["predict_batch"].append({"scene_pts": M, "candidates": B, "subsample": mode, "value": B / dt,
                                             "unit": "candidates/s", "ms": 1e3 * dt})
        scene = make_pile(20000, n_objects=12, seed=5)
        o = scene["object_id"] == 3
        d = {"cloud_xyz": scene["cloud_xyz"][o], "cloud_normal": scene["cloud_normal"][o]}
        npred.predict_nocs(dict(d))
        t0 = time.perf_counter()
        for _ in range(5):
            npred.predict_nocs(dict(d))
        out["nunocs_predict_nocs_ms"] = 1e3 * (time.perf_counter() - t0) / 5
    out["note"] = ("wall clock through catgrasp_b200.predicter (draw, H2D, forward, D2H, result list); 'host' = the reference's "
                   "numpy draw bit for bit (C continuation of MT19937, pipelined with the GPU), 'device' = counter-based "
                   "draw on the GPU (same distribution, not the reference's random stream); round 1 (numpy loop): 3.2k cand/s "
                   "at 20000 pts, 17.8k at 3000 pts")
    return out


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a B200; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"

    from catgrasp_b200 import _lib, my_cpp
    from catgrasp_b200.dist import all_gather_records, pack_records
    from catgrasp_b200.net import PointNetCls, PointNetSeg
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy, make_state_dict

    if args.config == "K5":
        return run_k5(args, rank, world, local, dev)
    sd_cls, sd_seg = make_state_dict("cls", 10, seed=0), make_state_dict("seg", 300, seed=1)
    cls = PointNetCls(sd_cls, device=local)
    seg = PointNetSeg(sd_seg, device=local)
    ctx = cls.ctx
    if args.engine is not None:
        ctx.set_engine(args.engine)
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"], device=local, ctx=ctx)
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"], device=local, ctx=ctx)
    N = args.n_pts
    mean, std = normalizer()
    assign = scene_assignment(args.config, rank, world)
    jobs = [make_scene_job(args.config, s, lo, hi, tot, args, rank) for (s, lo, hi, tot) in assign]
    B_local = sum(j["B"] for j in jobs)
    total_cands = CONFIGS[args.config]["total"] * (world if args.config == "K2" else 1)
    per_rank_max = max(1, -(-total_cands // world))

    # ---------------- device-resident inputs (the `value` leg)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    d_mean, d_std = up(mean), up(std)
    for j in jobs:
        j["d"] = {"xyz": up(j["scene"]["cloud_xyz"]), "nrm": up(j["scene"]["cloud_normal"]), "pose": up(j["poses"]),
                  "pose32": up(j["poses"].astype(np.float32)), "ids": up(j["ids"]), "nun": up(j["nun_in"]),
                  "open": up(j["open_pts"]), "bg": up(j["bg_pts"])}
    eye = np.eye(4)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def one_pass():
        recs, outs = [], []
        for j in jobs:
            d = j["d"]
            coords, conf, bins = seg.nunocs_dev(d["nun"], 100)
            outs.append({"nunocs_coords": coords, "nunocs_conf": conf, "nunocs_bins": bins})
            if j["B"] == 0:
                continue
            probs, label = cls.graspq_dev(d["xyz"], d["nrm"], d["pose"], d["ids"], d_mean, d_std)
            st, off, poses = my_cpp.filter_grasp_pose_raw(d["pose32"], eye[None], eye, eye, g["gripper_in_grasp"], True, True,
                                                          so, d["open"], se, d["bg"])
            outs[-1].update(graspq_probs=probs, graspq_label=label, filter_status=st, filter_offset=off, filter_poses=poses)
            recs.append(pack_records(probs, st, off))
        rec = torch.cat(recs) if len(recs) > 1 else (recs[0] if recs else torch.zeros((0, 12), device=dev))
        if world > 1:
            rec = all_gather_records(rec, per_rank_max * world)     # one ncclAllGather per pass, no host sync before it
        return rec, outs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up + calibration of passes_per_step
    for _ in range(2):
        flush.fill_(1)
        one_pass()
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        flush.fill_(1)
        one_pass()
    c1.record()
    barrier()
    pass_ms = torch.tensor([c0.elapsed_time(c1) / 3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(pass_ms, op=dist.ReduceOp.MAX)
    passes = args.passes_per_step or int(min(128, max(1, round(1200.0 / (float(pass_ms.item()) * max(args.steps, 1))))))

    def step_device():
        rec = outs = None
        for _ in range(passes):
            flush.fill_(1)                  # evict L2 between timed passes
            rec, outs = one_pass()
        return rec, outs

    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ctx.reset_launch_count()
    ctx.profile(True)
    ctx.profile_read()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        rec, outs = step_device()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count()
    trunk_ms, trunk_n = ctx.profile_read()
    ctx.profile(False)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        prefix = f"rank{rank}_" if world > 1 else ""
        dump_outputs(args.dump_outputs, {f"{prefix}scene{s}_{k}": v.cpu().numpy()
                                         for (s, _, _, _), o in zip(assign, outs) for k, v in o.items()})
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total_cands * passes * args.steps / (ms * 1e-3)
    checksum = float(rec[:, :10].sum().item())
    main_engine = ctx.get_engine()
    overflow = ctx.fp16_overflow()

    # ---------------- same workload on the 3-pass (near-fp32) tensor-core engine, for the record
    alt = None
    if main_engine >= 2:
        ctx.set_engine(1)
        for _ in range(2):
            one_pass()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        alt_passes = max(3, min(passes * args.steps // 8, 40))
        a0.record()
        for _ in range(alt_passes):
            flush.fill_(1)
            rec_alt, _ = one_pass()
        a1.record()
        barrier()
        t_alt = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_alt, op=dist.ReduceOp.MAX)
        alt = {"engine": ENGINE_NAMES[1], "value": total_cands * alt_passes / (float(t_alt.item()) * 1e-3),
               "unit": "candidates/s", "passes": alt_passes,
               "max_abs_dprob_vs_main_engine": float((rec_alt[:, :10] - rec[:, :10]).abs().max().item())}
        ctx.set_engine(main_engine)

    # ---------------- e2e leg: reference-facing C-ABI calls on pinned HOST buffers, H2D + D2H inside the timed region
    import ctypes as C
    lib = ctx.lib
    P = _lib.ptr
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()      # noqa: E731
    h_mean, h_std = pin(mean), pin(std)
    sym = pin(np.eye(4, dtype=np.float32))
    prm = _lib.FilterParams()
    for name, m in (("nocs_pose", eye), ("canonical_to_nocs", eye), ("gripper_in_grasp", g["gripper_in_grasp"])):
        setattr(prm, name, (C.c_float * 16)(*[float(v) for v in np.asarray(m, np.float32).reshape(16)]))
    prm.filter_approach_dir_face_camera, prm.adjust_collision_pose, prm.sdf_mode = 1, 1, 0
    h2d = d2h = 0
    for j in jobs:
        B = j["B"]
        j["h"] = {"xyz": pin(j["scene"]["cloud_xyz"]), "nrm": pin(j["scene"]["cloud_normal"]), "pose": pin(j["poses"]),
                  "ids": pin(j["ids"]), "nun": pin(j["nun_in"]), "pose32": pin(j["poses"].astype(np.float32)),
                  "open": pin(j["open_pts"]), "bg": pin(j["bg_pts"])}
        j["o"] = {"probs": torch.empty((B, 10), dtype=torch.float32).pin_memory(),
                  "label": torch.empty((B,), dtype=torch.int32).pin_memory(),
                  "coords": torch.empty((args.nunocs_pts, 3), dtype=torch.float32).pin_memory(),
                  "conf": torch.empty((args.nunocs_pts,), dtype=torch.float32).pin_memory(),
                  "bins": torch.empty((args.nunocs_pts, 3), dtype=torch.int32).pin_memory(),
                  "st": torch.empty((B,), dtype=torch.uint8).pin_memory(), "off": torch.empty((B,), dtype=torch.int8).pin_memory(),
                  "poses": torch.empty((B, 4, 4), dtype=torch.float32).pin_memory()}
        h2d += sum(v.numel() * v.element_size() for v in j["h"].values()) + 96 + 64
        d2h += sum(v.numel() * v.element_size() for v in j["o"].values())

    def pass_host():
        for j in jobs:
            h, o, B = j["h"], j["o"], j["B"]
            ctx.check(lib.cg_nunocs_forward_host(seg.h, P(h["nun"]), args.nunocs_pts, 100, P(o["coords"]), P(o["conf"]), P(o["bins"])))
            if B == 0:
                continue
            ctx.check(lib.cg_graspq_forward_host(cls.h, P(h["xyz"]), P(h["nrm"]), j["M"], P(h["pose"]), B, P(h["ids"]), N,
                                                 P(h_mean), P(h_std), P(o["probs"]), P(o["label"])))
            ctx.check(lib.cg_filter_grasp_pose_host(ctx.h, C.byref(prm), P(h["pose32"]), B, P(sym), 1, so.h, P(h["open"]),
                                                    h["open"].shape[0], se.h, P(h["bg"]), h["bg"].shape[0], P(o["st"]),
                                                    P(o["off"]), P(o["poses"])))

    ctx.use_own_stream()
    for _ in range(2):
        pass_host()
    barrier()
    e2e_passes = max(3, min(passes * args.steps // 4, 60))
    t0 = time.perf_counter()
    for _ in range(e2e_passes):
        pass_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = total_cands * e2e_passes / float(t.item())
    last = [j for j in jobs if j["B"]][-1] if B_local else None
    agree = None
    if last is not None:
        off = sum(j["B"] for j in jobs) - last["B"]
        base = rank * per_rank_max if world > 1 else 0
        agree = float(np.abs(last["o"]["probs"].numpy() - rec[base + off: base + off + last["B"], :10].cpu().numpy()).max())

    # ---------------- gather check: a sharded predict_batch equals the single-rank call (N > 1)
    gather_check = None
    if world > 1:
        gather_check = run_gather_check(args, local, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (fused shared-MLP + max "trunk")
    peaks = load_peaks()
    pts_per_pass = B_local * N + len(jobs) * args.nunocs_pts
    trunk_flops = 2.0 * sum(TRUNK_MAC_PER_PT) * pts_per_pass * passes * args.steps
    per_launch_ms = trunk_ms / max(trunk_n, 1)
    achieved = trunk_flops / (trunk_ms * 1e-3) / 1e12 if trunk_ms > 0 else 0.0
    long_region = ms > 500.0
    peak = peaks["bf16_tflops_sustained"] if long_region else peaks["bf16_tflops"]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "trunk_traffic.json")
    if os.path.exists(tpath):   # dram bytes per launch of the trunk from the committed ncu --set full capture
        traffic = json.load(open(tpath)).get("mean_bytes_per_launch")
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "trunk (fused shared-MLP 6-64-[64]-128-1024 + max)",
                "engine": ENGINE_NAMES[main_engine], "launches_timed": int(trunk_n), "avg_launch_ms": per_launch_ms,
                "share_of_step": trunk_ms / ms,
                "peak_source": f"{peaks['source']} bf16 dense, " + (f"sustained (timed region {ms / 1e3:.1f} s)" if long_region else "burst"),
                "frac_of_burst_peak": achieved / peaks["bf16_tflops"],
                "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"],
                "whole_step_tflops_per_gpu": (FLOP_PER_CAND[N] * value / world / 1e12) if N in FLOP_PER_CAND else None}

    line = {"metric": "candidate grasps scored/sec", "value": value, "unit": "candidates/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak" if args.config == "K2" else "strong", "vs_baseline": None,
            "dtype": ENGINE_DTYPES[main_engine], "data": "synthetic", "config": workload_config(args, passes, world),
            "e2e": {"value": e2e_value, "unit": "candidates/s", "h2d_bytes_per_step": int(h2d * passes),
                    "d2h_bytes_per_step": int(d2h * passes), "passes": e2e_passes, "max_abs_dprob_vs_device_leg": agree,
                    "through": "cg_nunocs_forward_host + cg_graspq_forward_host + cg_filter_grasp_pose_host (C ABI, pinned host buffers, "
                               "subset ids pre-drawn on the host; the draw-inclusive Python API is in e2e_api)",
                    "note": "every pass moves its inputs host->device and its results back inside the timed wall clock; the pinned "
                            "index buffer (the bulk of h2d_bytes) is read IN PLACE over the link by the three trunk launches "
                            "(3x its size crosses the link, hidden under the kernels) instead of being copied first; this leg has "
                            "no L2 flush (its inputs arrive from the host every pass) and a shorter region than `value` "
                            "(less time at the power cap), so it can come out above the device-resident figure"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "flop_per_candidate": FLOP_PER_CAND.get(N), "checksum": checksum, "fp16_clamp_seen": bool(overflow)}
    if alt is not None:
        line["alt_engine"] = alt
    if gather_check is not None:
        line["gather_check"] = gather_check
    if world == 1 and not args.no_api_leg:
        line["e2e_api"] = api_leg(local, N)
    if not args.no_cpu_baseline:
        n = min(args.cpu_sample, jobs[0]["B"])
        th = pick_torch_threads(sd_cls, N)
        r = cpu_reference_pass(jobs[0], args, n, sd_cls, sd_seg, mean, std, g)
        per_scene = CONFIGS[args.config]["total"] // CONFIGS[args.config]["scenes"]
        line["cpu_baseline"] = {"value": cpu_rate(r, n, per_scene), "unit": "candidates/s", "cores": os.cpu_count(),
                                "kind": "port", "sample": f"{n} of {per_scene} candidates (net {r['net_s']:.2f}s, collision "
                                f"{r['collision_s']:.2f}s) + 1 warm NUNOCS forward ({r['nunocs_s']:.2f}s, amortised 1 per {per_scene} "
                                f"candidates); torch threads {th} (sweep), OpenMP collision threads {th}; oracle PORT of the reference; "
                                f"the reference's own PointNetCls ran 134 cand/s on 8 cores in the survey container"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_gather_check(args, local, rank, world):
    """Rank 0 compares a 512-candidate dist.sharded_predict_batch (every rank scores its block, one all-gather) with its
    own single-rank predict_batch on the same candidates and the same subsets: must be bit-identical, in both draw modes,
    and leave numpy's generator in the same state."""
    import contextlib
    import io
    from catgrasp_b200.dist import sharded_predict_batch
    from catgrasp_b200.predicter import GraspPredicter
    from catgrasp_b200.synthetic import make_candidates, make_pile, write_artifacts
    td = tempfile.mkdtemp(prefix=f"cg_gc_{rank}_")
    adir = write_artifacts(os.path.join(td, "artifacts-47"), "cls", n_pts=args.n_pts, seed=0)
    with contextlib.redirect_stdout(io.StringIO()):
        gp = GraspPredicter("nut", artifact_dir=adir, device=local)
    scene = make_pile(20000, seed=0)
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    poses = list(make_candidates(scene["cloud_xyz"], scene["cloud_normal"], 512, seed=9))
    res = {}
    for mode in ("device", "host"):
        np.random.seed(5)
        full = sharded_predict_batch(gp, data, poses, subsample=mode)
        after_sharded = np.random.rand()
        np.random.seed(5)
        single = gp.predict_batch(data, poses, subsample=mode)
        after_single = np.random.rand()
        a = np.stack([o[2] for o in full])
        b = np.stack([o[2] for o in single])
        res[mode] = {"equal": bool(np.array_equal(a, b)), "max_abs_diff": float(np.abs(a - b).max()),
                     "same_numpy_stream": bool(after_sharded == after_single)}
    return {"candidates": 512, "ranks": world, **res}


def run_k5(args, rank, world, local, dev):
    """Offline path (generate_grasp.py:81-97): per object, surface samples -> cone pose enumeration ON THE DEVICE
    (cg_cone_poses_dev) -> collision filter with adjust_collision_pose off and no background (like :97) -> grasp-Q on
    the survivors with device-drawn subsets.  Surface samples shard across the ranks; ~1 M candidates in total."""
    import torch
    import torch.distributed as dist
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.dist import shard_range
    from catgrasp_b200.grasp_sampler import cone_frames, enumerate_poses
    from catgrasp_b200.net import PointNetCls
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy, make_pile, make_state_dict
    cls = PointNetCls(make_state_dict("cls", 10, seed=0), device=local)
    ctx = cls.ctx
    if args.engine is not None:
        ctx.set_engine(args.engine)
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"], device=local, ctx=ctx)
    scene = make_pile(CONFIGS["K5"]["scene_pts"], n_objects=1, seed=0)
    pts, nrm = scene["cloud_xyz"], scene["cloud_normal"]
    hand_depth, step, n_dir = 0.042, 0.003, 30
    per_sample = (1 + n_dir * 6) * len(np.arange(0, hand_depth, step))
    S_total = -(-CONFIGS["K5"]["total"] // per_sample)
    np.random.seed(0)
    sample_ids, R0s, sphere = cone_frames(pts.copy(), nrm.copy(), max_num_samples=S_total, n_sphere_dir=n_dir)   # host, not timed
    lo, hi = shard_range(len(sample_ids), rank, world)
    surf, R0 = pts[sample_ids[lo:hi]], R0s[lo:hi]
    eye = np.eye(4)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    d_xyz, d_nrm, d_obj = up(pts), up(nrm), up(pts.astype(np.float32))
    none_bg = torch.zeros((0, 3), dtype=torch.float32, device=dev)
    P_local = len(surf) * per_sample
    total = torch.tensor([P_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total)
    total = int(total.item())

    def one_pass():
        p64, p32 = enumerate_poses(surf, R0, sphere, hand_depth, step, 0.01, device=local)
        st, off, out = my_cpp.filter_grasp_pose_raw(p32, eye[None], eye, eye, g["gripper_in_grasp"], True, False, so, d_obj,
                                                    None, none_bg)
        keep = torch.nonzero(st == 0).flatten()
        n_keep = int(keep.numel())
        outs = {"filter_status": st, "filter_offset": off, "filter_poses": out}
        if n_keep:
            ids = cls.draw_ids_dev(pts.shape[0], args.n_pts, n_keep, seed=1234, first_candidate=0)
            outs["graspq_probs"], outs["graspq_label"] = cls.graspq_dev(d_xyz, d_nrm, p64[keep].contiguous(), ids)
        return n_keep, outs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(min(args.warmup, 3), 1)):
        one_pass()
    barrier()
    steps = args.steps
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        outs = None                     # drop the last pass's outputs first, so that this pass reuses their memory
        n_keep, outs = one_pass()
    ev1.record()
    barrier()
    if args.dump_outputs:
        prefix = f"rank{rank}_" if world > 1 else ""
        dump_outputs(args.dump_outputs, {prefix + k: v.cpu().numpy() for k, v in outs.items()})
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    k = torch.tensor([n_keep], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(k)
    if rank == 0:
        ms = float(t.item())
        line = {"metric": "candidate grasps scored/sec", "value": total * steps / (ms * 1e-3), "unit": "candidates/s",
                "n_gpus": world, "steps": steps, "warmup": max(min(args.warmup, 3), 1), "ms_per_step": ms / steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": ENGINE_DTYPES[ctx.get_engine()],
                "data": "synthetic",
                "config": {"workload": CONFIGS["K5"]["name"] + f"; {total} cone poses enumerated on the device per step "
                           f"({len(sample_ids)} surface samples x {per_sample}), every pose gets a collision verdict, the "
                           f"{int(k.item())} survivors a grasp-Q forward (n_pts={args.n_pts}, device-drawn subsets)",
                           "config": "K5", "candidates_total": total, "survivors": int(k.item()),
                           "parallelism": f"surface-sample shard x{world}",
                           "l2": "poses (128 MB / step / GPU at N=1) are regenerated every step: inputs larger than L2"},
                "gpu_launches": int(ctx.launch_count())}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
