"""CPU: pin the C oracle (filter_ref.c, occupancy_ref.c) and the host helpers against outputs of the reference's own
my_cpp/common.cpp as compiled by oracle/build_ref.py (tests/golden/make_golden_mycpp.py wrote the fixtures; the
FCL / octomap boundary of that build is shimmed, see oracle/build_ref.py).  Everything the compiled reference answered
is recorded in tests/golden, so only test_ref_build_recipe_reproduces_fixture needs the reference sources."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_mycpp as mk  # noqa: E402  (case tables + input builders shared with the generator)

from oracle import build_ref, filter_ref, mycpp_ref  # noqa: E402


@pytest.mark.parametrize("k", range(len(mk.FILTER_CASES)))
def test_filter_oracle_equals_reference_build(golden_dir, k):
    g_ = np.load(os.path.join(golden_dir, "mycpp_filter.npz"))
    S, scale, mode, adjust, fdir = mk.FILTER_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), dg = mk.filter_inputs(S, scale)
    assert np.array_equal(dg, g_[f"inputs_sha_{k}"]), "synthetic inputs drifted: regenerate the fixture"
    st, off, out = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                         g["enclosed"], p2)
    mine = mycpp_ref.sort_poses(out[st == 0]).view(np.uint32)
    assert np.array_equal(mine, g_[f"survivors_{k}"])          # same survivors, bit for bit (poses include the winning offset)


@pytest.mark.parametrize("k", range(len(mk.FILTER_CASES)))
@pytest.mark.parametrize("sideways", mk.COUNTER_SIDEWAYS)
def test_filter_rejection_counters_equal_reference_build(golden_dir, k, sideways):
    """The reference's verbose counters (common.cpp:316-319), printed by the compiled reference itself and recorded in
    mycpp_counters.npz, equal the counts of the oracle's status codes with split=True: 1 approach direction, 3 open
    gripper, 4 enclosed gripper -- with pose adjustment every collision rejection is an "open" one.  sideways = 2 cm:
    cases where the open gripper does collide."""
    g_ = np.load(os.path.join(golden_dir, "mycpp_counters.npz"))
    S, scale, mode, adjust, fdir = mk.FILTER_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), dg = mk.filter_inputs(S, scale)
    assert np.array_equal(dg, np.load(os.path.join(golden_dir, "mycpp_filter.npz"))[f"inputs_sha_{k}"])
    poses = mk.sideways_poses(poses, sideways)
    st, off, out = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                         g["enclosed"], p2, split=True)
    approach, ik, open_, close, n_ref = g_[f"counters_{k}_{mk.COUNTER_SIDEWAYS.index(sideways)}"].tolist()
    assert (approach, ik, open_, close) == (int((st == 1).sum()), 0, int((st == 3).sum()), int((st == 4).sum()))
    assert n_ref == int((st == 0).sum())
    if sideways and not adjust:
        assert open_ > 0 and close > 0


@pytest.mark.parametrize("k", range(len(mk.OCC_CASES)))
def test_occupancy_oracle_equals_reference_build(golden_dir, k):
    g_ = np.load(os.path.join(golden_dir, "mycpp_occupancy.npz"))
    res, n, seed = mk.OCC_CASES[k]
    pts = mk.occupancy_inputs(n, seed)
    assert np.array_equal(mk.digest(pts), g_[f"inputs_sha_{k}"])
    flags, org, dims = filter_ref.occupancy_ref(pts, res)
    idx = np.argwhere(flags > 0)
    mine = (org[None, :] + idx.astype(np.float32) * np.float32(res)).astype(np.float32)
    assert np.array_equal(np.unique(mine.view(np.uint32), axis=0), g_[f"points_{k}"])


def test_direction_vec_to_rotation_matches_reference_build(golden_dir):
    from catgrasp_b200.my_cpp import directionVecToRotation
    g_ = np.load(os.path.join(golden_dir, "mycpp_direction.npz"))
    for d, R in zip(g_["direction"], g_["R"]):
        np.testing.assert_allclose(directionVecToRotation(d, g_["ref"]), R, rtol=0, atol=5e-6)


@pytest.mark.skipif(not build_ref.available(), reason="needs the reference sources")
def test_ref_build_recipe_reproduces_fixture(golden_dir):
    """Where the reference is present the recipe itself is exercised: build oracle/_ref and re-run one case live."""
    g_ = np.load(os.path.join(golden_dir, "mycpp_filter.npz"))
    k = 6
    S, scale, mode, adjust, fdir = mk.FILTER_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), _ = mk.filter_inputs(S, scale)
    ref = mycpp_ref.filterGraspPose(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                    g["enclosed"], p2)
    assert np.array_equal(mycpp_ref.sort_poses(ref).view(np.uint32), g_[f"survivors_{k}"])


@pytest.mark.parametrize("k", range(len(mk.IK_CASES)))
def test_filter_with_ik_stage_equals_reference_build(golden_dir, k):
    """filter_ik=True: oracle survivors, thinned by the reference's own get_ik_within_limits on the un-shifted pose
    (catgrasp_b200.my_cpp.grasp_in_cam_unshifted, bit-identical to the kernel; verdicts recorded in mycpp_ik.npz),
    equal the reference's survivors."""
    from catgrasp_b200.my_cpp import _mm4_f32, grasp_in_cam_unshifted
    g_ = np.load(os.path.join(golden_dir, "mycpp_filter.npz"))
    S, scale, mode, adjust, fdir = mk.IK_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), dg = mk.filter_inputs(S, scale)
    cam, ee = mk.ik_frames()
    assert np.array_equal(mk.digest(dg, cam, ee, mk.IK_UPPER, mk.IK_LOWER), g_[f"ik_inputs_sha_{k}"])
    ik_ok = mk.recorded_ik_solver(golden_dir, k)
    st, off, out = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode, g["open"], p1,
                                         g["enclosed"], p2)
    u = grasp_in_cam_unshifted(poses, sym, nocs_pose, c2n)
    f = lambda m: np.asarray(m, np.float64).astype(np.float32)      # noqa: E731
    keep = [q for q in np.nonzero(st == 0)[0] if ik_ok(_mm4_f32(_mm4_f32(f(cam), u[q]), f(ee)), mk.IK_UPPER, mk.IK_LOWER)]
    assert 0 < len(keep) < int((st == 0).sum())
    assert np.array_equal(mycpp_ref.sort_poses(out[keep]).view(np.uint32), g_[f"ik_survivors_{k}"])
