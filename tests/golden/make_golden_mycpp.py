"""Golden vectors from the REFERENCE's own my_cpp/common.cpp, compiled by oracle/build_ref.py (FCL/octomap boundary
shimmed -- see that file for exactly what is and is not the reference in the library).

Run in the authoring container only (needs /root/reference):

    python tests/golden/make_golden_mycpp.py

Inputs are regenerated from catgrasp_b200.synthetic (seeded); the fixture stores a SHA-256 of the input bytes so a
drifting generator is detected, plus the reference outputs:
  mycpp_filter.npz      filterGraspPose survivors (sorted bit patterns) for 12 flag/symmetry/scale combinations
  mycpp_occupancy.npz   makeOccupancyGridFromCloudScan occupied samples (sorted bit patterns)
  mycpp_direction.npz   directionVecToRotation on random and degenerate directions
  mycpp_counters.npz    filterGraspPose's verbose rejection counters and survivor count per filter case, straight and
                        with every third pose shifted sideways (COUNTER_SIDEWAYS)
  mycpp_ik.npz          the ikfast solution count for every ee_in_base the IK stage can be asked about in IK_CASES,
                        so that tests replay the reference's IK verdicts without its compiled solver
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from catgrasp_b200 import synthetic      # noqa: E402
from oracle import mycpp_ref  # noqa: E402

FILTER_CASES = [(S, scale, mode, adjust, fdir)
                for (S, scale) in [(1, (1, 1, 1)), (12, (1.0, 1.1, 0.9))]
                for mode in (0, 1)
                for adjust, fdir in [(True, True), (False, True), (True, False)]]


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def filter_inputs(S, scale):
    p1, p2, poses, sym, nocs_pose, c2n, g = synthetic.make_filter_case(43, 128, S, scale)
    dg = digest(p1, p2, poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], g["open"]["sdf"], g["enclosed"]["sdf"])
    return (p1, p2, poses, sym, nocs_pose, c2n, g), dg


COUNTER_SIDEWAYS = (0.0, 0.02)       # metres along the gripper x axis, every third pose: makes the open gripper collide


def sideways_poses(poses, sideways):
    poses = poses.copy()
    poses[::3, :3, 3] += poses[::3, :3, 0] * sideways
    return poses


# filter_ik=True cases (common.cpp:214-226) run the reference's generated KUKA iiwa14 ikfast solver, compiled into oracle/_ref
IK_CASES = [(12, (1.0, 1.1, 0.9), 0, True, True), (1, (1, 1, 1), 1, False, False)]
IK_UPPER = np.deg2rad([170, 120, 170, 120, 170, 120, 175])
IK_LOWER = -IK_UPPER


def ik_frames():
    cam_in_world = np.eye(4)
    cam_in_world[:3, :3] = np.diag([1.0, -1.0, -1.0])            # camera looks down at the bin
    cam_in_world[:3, 3] = [0.6, 0.0, 0.85]
    ee_in_grasp = np.eye(4)
    ee_in_grasp[:3, :3] = np.array([[0, 0, 1], [0, 1, 0], [-1, 0, 0]], float).T
    ee_in_grasp[:3, 3] = [-0.17, 0, 0]
    return cam_in_world, ee_in_grasp


def ik_queries(k):
    """(G*S, 4, 4) float32: ee_in_base for every (pose, symmetry) of IK case k, computed the way
    catgrasp_b200.my_cpp.filterGraspPose hands it to the IK hook (common.cpp:216, left to right)."""
    from catgrasp_b200.my_cpp import _mm4_f32, grasp_in_cam_unshifted
    S, scale, _, _, _ = IK_CASES[k]
    (_, _, poses, sym, nocs_pose, c2n, _), _ = filter_inputs(S, scale)
    cam, ee = ik_frames()
    f = lambda m: np.asarray(m, np.float64).astype(np.float32)      # noqa: E731
    u = grasp_in_cam_unshifted(poses, sym, nocs_pose, c2n)
    return _mm4_f32(_mm4_f32(f(cam), u), f(ee))


def recorded_ik_solver(golden_dir, k):
    """IK hook for set_ik_solver: the reference's ikfast verdict recorded in mycpp_ik.npz for IK case k.  A pose that
    was not recorded, or other joint limits, raise instead of guessing."""
    g = np.load(os.path.join(golden_dir, "mycpp_ik.npz"))
    table = dict(zip((q.tobytes() for q in g[f"query_{k}"]), g[f"count_{k}"].tolist()))

    def solve(ee_in_base, upper, lower):
        assert np.array_equal(upper, IK_UPPER) and np.array_equal(lower, IK_LOWER)
        return table[np.ascontiguousarray(ee_in_base, np.float32).reshape(16).view(np.uint32).tobytes()] > 0
    return solve


def occupancy_inputs(n, seed):
    sc = synthetic.make_pile(n, n_objects=4, seed=seed)
    return sc["cloud_xyz"].astype(np.float32)


OCC_CASES = [(0.002, 3000, 5), (0.001, 6000, 5), (0.001, 20000, 6)]


def main():
    out = {}
    for k, (S, scale, mode, adjust, fdir) in enumerate(FILTER_CASES):
        (p1, p2, poses, sym, nocs_pose, c2n, g), dg = filter_inputs(S, scale)
        ref = mycpp_ref.filterGraspPose(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                        g["enclosed"], p2)
        out[f"survivors_{k}"] = mycpp_ref.sort_poses(ref).view(np.uint32)
        out[f"inputs_sha_{k}"] = dg
        print("filter case", k, (S, scale, mode, adjust, fdir), "survivors", len(ref))
    cam, ee = ik_frames()
    for k, (S, scale, mode, adjust, fdir) in enumerate(IK_CASES):
        (p1, p2, poses, sym, nocs_pose, c2n, g), dg = filter_inputs(S, scale)
        ref = mycpp_ref.filterGraspPose(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                        g["enclosed"], p2, cam_in_world=cam, ee_in_grasp=ee, filter_ik=True,
                                        upper=IK_UPPER, lower=IK_LOWER)
        out[f"ik_survivors_{k}"] = mycpp_ref.sort_poses(ref).view(np.uint32)
        out[f"ik_inputs_sha_{k}"] = digest(dg, cam, ee, IK_UPPER, IK_LOWER)
        print("filter+IK case", k, (S, scale, mode, adjust, fdir), "survivors", len(ref))
    np.savez_compressed(os.path.join(HERE, "mycpp_filter.npz"), **out)
    out = {}
    for k, (res, n, seed) in enumerate(OCC_CASES):
        pts = occupancy_inputs(n, seed)
        ref = mycpp_ref.makeOccupancyGridFromCloudScan(pts, np.eye(3), res)
        out[f"points_{k}"] = np.unique(ref.view(np.uint32), axis=0)        # sorted bit patterns of the (Q,3) float32 samples
        out[f"inputs_sha_{k}"] = digest(pts)
        print("occupancy case", k, (res, n, seed), "occupied samples", len(ref))
    np.savez_compressed(os.path.join(HERE, "mycpp_occupancy.npz"), **out)
    rng = np.random.RandomState(2)
    d = rng.normal(0, 1, (64, 3)).astype(np.float32)
    d[0] = [1, 0, 0]; d[1] = [-1, 0, 0]; d[2] = [3, 1e-7, 0]          # parallel / anti-parallel / nearly parallel to ref
    ref = np.array([1, 0, 0], np.float32)
    R = np.stack([mycpp_ref.directionVecToRotation(v, ref) for v in d])
    np.savez_compressed(os.path.join(HERE, "mycpp_direction.npz"), direction=d, ref=ref, R=R)
    print("direction cases", len(d))
    reference_counters_and_ik()


def reference_counters_and_ik():
    out = {}
    for k, (S, scale, mode, adjust, fdir) in enumerate(FILTER_CASES):
        (p1, p2, poses, sym, nocs_pose, c2n, g), _ = filter_inputs(S, scale)
        for j, sideways in enumerate(COUNTER_SIDEWAYS):
            ref, cnt = mycpp_ref.filterGraspPose(sideways_poses(poses, sideways), sym, nocs_pose, c2n, g["gripper_in_grasp"],
                                                 fdir, adjust, mode, g["open"], p1, g["enclosed"], p2, counters=True)
            out[f"counters_{k}_{j}"] = np.array([cnt["approach"], cnt["ik"], cnt["open"], cnt["close"], len(ref)], np.int64)
    np.savez_compressed(os.path.join(HERE, "mycpp_counters.npz"), **out)
    print("counter cases", len(out))
    out = {}
    for k in range(len(IK_CASES)):
        q = ik_queries(k)
        out[f"query_{k}"] = q.reshape(-1, 16).view(np.uint32)
        out[f"count_{k}"] = np.array([mycpp_ref.ik_solution_count(m, IK_UPPER, IK_LOWER) for m in q], np.int32)
        print("IK case", k, "queries", len(q), "with a solution", int((out[f"count_{k}"] > 0).sum()))
    np.savez_compressed(os.path.join(HERE, "mycpp_ik.npz"), **out)


if __name__ == "__main__":
    main()
