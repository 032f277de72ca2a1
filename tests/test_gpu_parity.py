"""GPU parity tests (-m gpu): CUDA path through the C ABI vs the CPU oracle / the reference's golden vectors.

Tolerances (north_star): collision/accept masks and all index work bit-exact; grasp-Q probabilities
within 1e-4; NUNOCS bins equal except where the top-2 logit gap is inside the logit tolerance.
"""
import copy
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-4          # north_star: scores within 1e-4 of the reference
LOGIT_TOL = 5e-4


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a B200; there is no CPU fallback")
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _engines():
    return [int(e) for e in os.environ.get("CG_TEST_ENGINES", "0,1,2,3").split(",")]


@pytest.fixture(scope="module")
def cls_net(cuda):
    from catgrasp_b200.net import PointNetCls
    from catgrasp_b200.synthetic import make_state_dict
    sd = make_state_dict("cls", 10, seed=0)
    return PointNetCls(sd, device=0), sd


@pytest.fixture(scope="module")
def seg_net(cuda):
    from catgrasp_b200.net import PointNetSeg
    from catgrasp_b200.synthetic import make_state_dict
    sd = make_state_dict("seg", 300, seed=1)
    return PointNetSeg(sd, device=0), sd


def _oracle_probs(sd, xyz, nrm, poses, ids, mean=None, std=None):
    """The reference's predict_batch arithmetic (dataset_grasp.py:69-85, predicter.py:84-86) for explicit subsets:
    float64 transform of the selected points, optional normaliser, fp32 PointNetCls, softmax."""
    from oracle.pointnet_ref import pointnet_cls_forward
    from oracle.transforms_ref import to_homo
    x = []
    for pose, sel in zip(poses, ids):
        p = (np.linalg.inv(pose) @ to_homo(xyz[sel]).T).T[:, :3]
        n = (np.linalg.inv(pose[:3, :3]) @ nrm[sel].T).T
        inp = np.concatenate((p, n), axis=-1)
        if mean is not None:
            inp = (inp - mean.reshape(1, -1)) / (std.reshape(1, -1) + 1e-15)
        x.append(inp)
    x = torch.from_numpy(np.stack(x)).float()
    return pointnet_cls_forward(sd, x)[0].softmax(dim=1).numpy()


# ------------------------------------------------------------------ networks
def test_tmem_fragment_layout(cuda):
    """The engine-3 max epilogue reads accumulators with tcgen05.ld.16x256b and reduces columns with FMNMX3 +
    a 3-step lane exchange.  TMEM is filled with lane*1000 + column; the column max over a warp's 32 lanes must be
    (32*warp + 31)*1000 + column, with thread t ending up with columns 2t and 2t+1."""
    import ctypes as C
    from catgrasp_b200 import _lib
    ctx = _lib.Context.get(0)
    out = np.zeros(768, np.float32)
    ctx.check(ctx.lib.cg_tmem_layout_selftest(ctx.h, C.c_void_p(out.ctypes.data)))
    red = out[:256].reshape(4, 32, 2)
    for w in range(4):
        for t in range(32):
            for k in range(2):
                assert red[w, t, k] == (32 * w + 31) * 1000 + 2 * t + k, (w, t, k, red[w, t, k])
    frag = out[256:].reshape(4, 32, 4)
    for w in range(4):
        for t in range(32):
            lane = 32 * w + t // 4
            exp = [lane * 1000 + 2 * (t % 4), lane * 1000 + 2 * (t % 4) + 1,
                   (lane + 8) * 1000 + 2 * (t % 4), (lane + 8) * 1000 + 2 * (t % 4) + 1]
            assert list(frag[w, t]) == exp, (w, t, frag[w, t], exp)


@pytest.mark.parametrize("engine", _engines())
def test_cls_vs_reference_golden(cls_net, golden_dir, engine):
    net, _ = cls_net
    net.ctx.set_engine(engine)
    g = np.load(os.path.join(golden_dir, "pointnet_cls.npz"))
    logits, probs = net.forward(g["x"], return_probs=True)
    assert np.abs(logits.cpu().numpy() - g["logits"]).max() < LOGIT_TOL * (1 if engine < 2 else 4)
    assert np.abs(probs.cpu().numpy() - g["probs"]).max() < PROB_TOL


@pytest.mark.parametrize("engine", _engines())
def test_seg_vs_reference_golden(seg_net, golden_dir, engine):
    net, _ = seg_net
    net.ctx.set_engine(engine)
    g = np.load(os.path.join(golden_dir, "pointnet_seg.npz"))
    logits = net.forward(g["x"]).cpu().numpy()
    assert np.abs(logits - g["logits"]).max() < (2e-4 if engine < 2 else 2e-3)
    # what the looser logit tolerance of the fp16 engines means for NUNOCS: a bin (argmax over 100 logits per axis,
    # predicter.py:144-146) may flip only where the reference's own top-2 gap is inside that tolerance
    ref = g["logits"].reshape(-1, 3, 100)
    got = logits.reshape(-1, 3, 100)
    flipped = ref.argmax(-1) != got.argmax(-1)
    top2 = np.sort(ref, axis=-1)[..., -2:]
    assert (top2[..., 1] - top2[..., 0])[flipped].max(initial=0.0) < (4e-4 if engine < 2 else 4e-3)
    assert flipped.mean() <= 0.01


def test_seg_bin_stability_8192_points(seg_net):
    """NUNOCS-sized cloud (8192 points): fraction of the 24 576 coordinate bins on which the fp16 engines (2, 3) differ
    from the near-fp32 engine 1 (CPU emulation of engine 3: 2 of 24 576), and every differing bin is a near-tie."""
    net, _ = seg_net
    rng = np.random.RandomState(1)
    x = np.concatenate([rng.uniform(0, 1, (1, 8192, 3)), rng.normal(0, 0.6, (1, 8192, 3))], -1).astype(np.float32)
    out = {}
    for e in (1, 2, 3):
        net.ctx.set_engine(e)
        out[e] = net.forward(x).cpu().numpy().reshape(-1, 3, 100)
    net.ctx.set_engine(3)
    top2 = np.sort(out[1], axis=-1)[..., -2:]
    gap = top2[..., 1] - top2[..., 0]
    for e in (2, 3):
        flipped = out[e].argmax(-1) != out[1].argmax(-1)
        assert flipped.mean() < 1e-3, (e, flipped.sum())
        assert gap[flipped].max(initial=0.0) < 2e-3
        assert np.abs(out[e] - out[1]).max() < 2e-3


@pytest.mark.parametrize("engine", _engines())
@pytest.mark.parametrize("B,N", [(1, 1), (3, 127), (5, 128), (2, 1000), (130, 64)])
def test_cls_ragged_shapes_vs_oracle(cls_net, engine, B, N):
    from oracle.pointnet_ref import pointnet_cls_forward
    net, sd = cls_net
    net.ctx.set_engine(engine)
    rng = np.random.RandomState(B * 1000 + N)
    x = rng.normal(0, 1, (B, N, 6)).astype(np.float32)
    ref = pointnet_cls_forward(sd, x)[0]
    logits, probs = net.forward(x, return_probs=True)
    assert np.abs(probs.cpu().numpy() - ref.softmax(1).numpy()).max() < PROB_TOL
    assert np.abs(logits.cpu().numpy() - ref.numpy()).max() < LOGIT_TOL * (4 if engine >= 2 else 1)


@pytest.mark.parametrize("engine", _engines())
@pytest.mark.parametrize("M,N,normalizer", [(3000, 512, True), (3000, 512, False), (300, 512, True), (1024, 1024, True)])
def test_graspq_fused_vs_oracle(cls_net, engine, M, N, normalizer):
    """Fused transform + forward == oracle predict_batch with the same numpy RNG stream
    (M < N exercises the replace=True draw, M == N the permutation draw)."""
    from catgrasp_b200.predicter import draw_subsample_ids
    from catgrasp_b200.synthetic import make_candidates, make_pile
    from oracle.transforms_ref import predict_batch
    net, sd = cls_net
    net.ctx.set_engine(engine)
    scene = make_pile(M, n_objects=4, seed=11)
    poses = make_candidates(scene["cloud_xyz"], scene["cloud_normal"], 12, seed=12)
    cfg = {"n_pts": N}
    rng = np.random.RandomState(5)
    mean = std = None
    if normalizer:
        mean = np.concatenate([rng.normal(0, 0.002, 3), rng.normal(0, 0.05, 3)])
        std = np.concatenate([rng.uniform(0.008, 0.012, 3), rng.uniform(0.5, 0.6, 3)])
        cfg["mean"], cfg["std"] = mean, std
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    np.random.seed(0)
    ref = predict_batch(sd, cfg, data, poses)
    np.random.seed(0)
    ids = draw_subsample_ids(M, N, count=len(poses))
    probs, _ = net.graspq_host(scene["cloud_xyz"], scene["cloud_normal"], poses, ids, mean, std)
    err = max(np.abs(probs[b] - ref[b][2]).max() for b in range(len(poses)))
    assert err < PROB_TOL, err


def test_predicter_dropin_surface(cuda, tmp_path):
    """GraspPredicter / NunocsPredicter keep the reference call surface (predicter.py:39-203)."""
    from catgrasp_b200.predicter import GraspPredicter, NunocsPredicter
    from catgrasp_b200.synthetic import make_candidates, make_pile, write_artifacts
    from catgrasp_b200.weights import load_checkpoint
    from oracle.transforms_ref import nunocs_predict, predict_batch
    adir = write_artifacts(str(tmp_path / "artifacts-47"), "cls", n_pts=256, seed=0)
    gp = GraspPredicter("nut", artifact_dir=adir)
    scene = make_pile(1500, n_objects=3, seed=21)
    scene["cloud_xyz"][:5, 2] = 0.05          # below the z >= 0.1 mask (dataset_grasp.py:64)
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    keep = copy.deepcopy(data)
    poses = list(make_candidates(scene["cloud_xyz"][5:], scene["cloud_normal"][5:], 7, seed=22))
    np.random.seed(3)
    out = gp.predict_batch(data, poses)
    assert all(np.array_equal(data[k], keep[k]) for k in data)          # not mutated (predicter.py:72)
    np.random.seed(3)
    ref = predict_batch(load_checkpoint(adir + "/best_val.pth.tar"), gp.cfg, keep, poses)
    assert len(out) == len(ref) == 7
    for o, r in zip(out, ref):
        assert isinstance(o[0], np.int64) and o[2].dtype == np.float32 and o[2].shape == (10,)
        assert np.abs(o[2] - r[2]).max() < PROB_TOL and abs(o[1] - r[1]) < PROB_TOL
    assert gp.predict_batch(data, []) == []
    # NUNOCS network half
    ndir = write_artifacts(str(tmp_path / "artifacts-78"), "seg", n_pts=512, seed=1)
    npred = NunocsPredicter("nut", artifact_dir=ndir)
    np.random.seed(4)
    nocs, conf = npred.predict_nocs(copy.deepcopy(keep))
    np.random.seed(4)
    rn, rc, rlogits, rdt = nunocs_predict(load_checkpoint(ndir + "/best_val.pth.tar"), npred.cfg, copy.deepcopy(keep))
    assert np.array_equal(npred.data_transformed["cloud_xyz_original"], rdt["cloud_xyz_original"])
    assert np.array_equal(npred.data_transformed["keep_ids"], rdt["keep_ids"])
    top2 = np.sort(rlogits, axis=-1)[..., -2:]
    tol = 2 * LOGIT_TOL * max(1.0, float(np.abs(rlogits).max()))
    decisive = (top2[..., 1] - top2[..., 0]) > tol                    # Appendix A6: bins equal where the gap is decisive
    assert np.array_equal(nocs[decisive], rn[decisive])
    assert decisive.mean() > 0.9
    assert (nocs.min() >= -0.5) and (nocs.max() <= 0.49 + 1e-6)
    assert np.abs(conf - rc).max() < PROB_TOL


@pytest.mark.parametrize("engine", _engines())
def test_graspq_full_size_properties(cls_net, engine):
    """BASELINE config K2 shape (20k-pt scene, 4096 candidates, 1024 pts each), every engine: size-independent
    properties -- probabilities are normalised, duplicated candidates agree bit-for-bit, a permutation of a candidate's
    point subset leaves its output bit-identical (max-pool invariance) -- AND a random sample of 256 of the 4096
    candidates re-scored by the CPU oracle (candidates are independent, so a sample pins the whole batch)."""
    from catgrasp_b200.synthetic import make_candidates, make_pile
    net, sd = cls_net
    net.ctx.set_engine(engine)
    M, B, N = 20000, 4096, 1024
    scene = make_pile(M, seed=0)
    poses = make_candidates(scene["cloud_xyz"], scene["cloud_normal"], B, seed=1)
    rng = np.random.RandomState(0)
    ids = np.stack([rng.permutation(M)[:N] for _ in range(64)]).astype(np.int32)
    ids = np.tile(ids, (B // 64, 1))
    poses[B // 2:] = poses[: B // 2]                      # second half duplicates the first
    ids[B // 2:] = ids[: B // 2][:, ::-1]                 # ... with its points in reverse order
    probs, label = net.graspq_host(scene["cloud_xyz"], scene["cloud_normal"], poses, np.ascontiguousarray(ids))
    assert np.isfinite(probs).all()
    assert np.abs(probs.sum(1) - 1).max() < 1e-5
    assert np.array_equal(probs[: B // 2].view(np.uint32), probs[B // 2:].view(np.uint32))
    assert np.array_equal(label, probs.argmax(1))
    sel = np.random.RandomState(engine).choice(B, 256, replace=False)
    ref = _oracle_probs(sd, scene["cloud_xyz"], scene["cloud_normal"], poses[sel], ids[sel])
    assert np.abs(probs[sel] - ref).max() < PROB_TOL


# ------------------------------------------------------------------ collision filter
def _filter_case(seed, G, S, scale=(1, 1, 1), n_points=2400):
    from catgrasp_b200.synthetic import make_filter_case
    return make_filter_case(seed, G, S, scale, n_points)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("adjust,fdir", [(True, True), (False, True), (True, False)])
@pytest.mark.parametrize("S,scale", [(1, (1, 1, 1)), (12, (1.0, 1.1, 0.9))])
def test_filter_bit_exact_vs_oracle(cuda, mode, adjust, fdir, S, scale):
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from oracle import filter_ref
    p1, p2, poses, sym, nocs_pose, c2n, g = _filter_case(43, 128, S, scale)
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    st, off, out = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, so, p1,
                                                se, p2, sdf_mode=mode)
    rst, roff, rout = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], fdir, adjust, mode,
                                            g["open"], p1, g["enclosed"], p2)
    assert np.array_equal(st, rst)
    assert np.array_equal(off, roff)
    assert np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    assert (st == 0).any() and (st == 3).any()      # the case exercises accept and collision-reject ...
    if adjust:
        assert len(set(off[st == 0].tolist())) >= 2  # ... and more than one winning lateral offset
    # device-pointer entry gives the same answer
    dst, doff, dout = my_cpp.filter_grasp_pose_raw(torch.from_numpy(poses).cuda(), sym, nocs_pose, c2n,
                                                   g["gripper_in_grasp"], fdir, adjust, so, p1, se, p2, sdf_mode=mode)
    assert np.array_equal(dst.cpu().numpy(), st) and np.array_equal(dout.cpu().numpy().view(np.uint32), out.view(np.uint32))


@pytest.mark.parametrize("mode", [0, 1])
def test_filter_split_collision_status_vs_oracle(cuda, mode, capsys):
    """split_coll_status without pose adjustment: which of the reference's two tests rejected a pose (open gripper vs
    object points -> 3, enclosed gripper vs background -> 4; common.cpp:228-249), bit-exact vs the oracle (whose counters
    equal the reference build's own, tests/test_mycpp_golden.py); the accept set does not depend on the switch, and
    filterGraspPose(verbose=True) prints the reference's counter line."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from oracle import filter_ref
    p1, p2, poses, sym, nocs_pose, c2n, g = _filter_case(43, 256, 2)
    poses = poses.copy()
    poses[::3, :3, 3] += poses[::3, :3, 0] * 0.02      # every third candidate 2 cm sideways: a finger lands in the object
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    st, off, out = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, False, so, p1, se, p2,
                                                sdf_mode=mode, split_status=True)
    rst, roff, rout = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, False, mode, g["open"], p1,
                                            g["enclosed"], p2, split=True)
    assert np.array_equal(st, rst) and np.array_equal(off, roff) and np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    assert (st == 3).any() and (st == 4).any() and (st == 0).any() and (st == 1).any()
    st0, _, out0 = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, False, so, p1, se, p2,
                                                sdf_mode=mode)
    assert np.array_equal(st0 == 0, st == 0) and np.array_equal(st0[st0 != 0] == 1, st[st != 0] == 1)
    assert not (st0 == 4).any() and np.array_equal(out0.view(np.uint32), out.view(np.uint32))
    # with pose adjustment the reference counts every collision rejection as "open" (common.cpp:290-294)
    sta, _, _ = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, True, so, p1, se, p2,
                                             sdf_mode=mode, split_status=True)
    assert not (sta == 4).any()
    if mode == 0:
        my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
        my_cpp.register_gripper_sdf(g["enclosed"]["V"], g["enclosed"]["F"], se)
        capsys.readouterr()
        got = my_cpp.filterGraspPose(list(poses), list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"], True,
                                     False, False, np.zeros(7), np.zeros(7), g["open"]["V"], g["open"]["F"], g["enclosed"]["V"],
                                     g["enclosed"]["F"], p1, p2, 0.0005, True)
        line = capsys.readouterr().out.strip().splitlines()[-1]
        assert line == "n_approach_dir_rej={}, n_ik_rej=0, n_open_gripper_rej={}, n_close_gripper_rej={}".format(
            int((st == 1).sum()), int((st == 3).sum()), int((st == 4).sum()))
        assert len(got) == int((st == 0).sum())


@pytest.mark.parametrize("mode", [0, 1])
def test_filter_voxel_margin_bit_exact_vs_oracle(cuda, mode):
    """sdf_margin = octo_resolution * sqrt(3)/2 (the conservative stand-in for the reference's mesh-vs-voxel test):
    GPU == oracle bit for bit, strictly more rejections than the plain SDF predicate, and the reference-facing
    filterGraspPose switches predicate through my_cpp.COLLISION_PREDICATE."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from oracle import filter_ref
    p1, p2, poses, sym, nocs_pose, c2n, g = _filter_case(43, 256, 2)
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    m = my_cpp.voxel_margin(0.0005)
    st, off, out = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, True, so, p1, se, p2,
                                                sdf_mode=mode, sdf_margin=m)
    rst, roff, rout = filter_ref.filter_ref(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, True, mode, g["open"], p1,
                                            g["enclosed"], p2, margin=m)
    assert np.array_equal(st, rst) and np.array_equal(off, roff)
    assert np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    st0, _, _ = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, True, so, p1, se, p2,
                                             sdf_mode=mode)
    assert (st == 0).sum() < (st0 == 0).sum() and not ((st == 0) & (st0 != 0)).any() or mode == 1
    if mode == 0:
        my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
        my_cpp.register_gripper_sdf(g["enclosed"]["V"], g["enclosed"]["F"], se)
        args = (list(poses), list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"], True, False, True,
                np.zeros(7), np.zeros(7), g["open"]["V"], g["open"]["F"], g["enclosed"]["V"], g["enclosed"]["F"], p1, p2,
                0.0005, False)
        try:
            my_cpp.COLLISION_PREDICATE = "voxel"
            got = my_cpp.filterGraspPose(*args)
        finally:
            my_cpp.COLLISION_PREDICATE = "sdf"
        assert len(got) == int((st == 0).sum())
        assert len(my_cpp.filterGraspPose(*args)) == int((st0 == 0).sum())


def test_filter_k2_size_bit_exact_and_offsets(cuda):
    """K2 shape: 4096 candidates x (20k-pt scene split into object / background points)."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_candidates, make_gripper_proxy, make_pile
    from oracle import filter_ref
    scene = make_pile(20000, seed=1)
    obj = scene["object_id"] == 3
    p1, p2 = scene["cloud_xyz"][obj], scene["cloud_xyz"][~obj]
    poses = make_candidates(p1, scene["cloud_normal"][obj], 4096, seed=1)
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    eye = np.eye(4)
    st, off, out = my_cpp.filter_grasp_pose_raw(poses, [eye], eye, eye, g["gripper_in_grasp"], True, True, so, p1, se, p2)
    rst, roff, rout = filter_ref.filter_ref(poses, [eye], eye, eye, g["gripper_in_grasp"], True, True, 0, g["open"], p1,
                                            g["enclosed"], p2)
    assert np.array_equal(st, rst) and np.array_equal(off, roff)
    assert np.array_equal(out.view(np.uint32), rout.view(np.uint32))
    acc = st == 0
    assert 0 < acc.sum() < len(st)
    # accepted poses are the normalised input shifted along their own y axis by exactly the winning step
    steps = np.array([0.0, 0.001, -0.001, 0.002, -0.002])
    g0 = poses.astype(np.float32)
    shift = np.einsum("ij,ij->i", out[acc][:, :3, 3] - g0[acc][:, :3, 3], out[acc][:, :3, 1])
    assert np.abs(shift - steps[off[acc]]).max() < 2e-6
    assert (out[~acc] == 0).all() and (off[~acc] == -1).all()


def test_my_cpp_filterGraspPose_signature(cuda):
    """The 20-positional-argument call of grasp_sampler.py:216 works unchanged."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    p1, p2, poses, sym, nocs_pose, c2n, g = _filter_case(43, 40, 2)
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
    my_cpp.register_gripper_sdf(g["enclosed"]["V"], g["enclosed"]["F"], se)
    res = my_cpp.filterGraspPose(list(poses), list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"],
                                 True, False, True, [3] * 7, [-3] * 7, g["open"]["V"], g["open"]["F"],
                                 g["enclosed"]["V"], g["enclosed"]["F"], p1, p2, 0.0005, False)
    st, _, out = my_cpp.filter_grasp_pose_raw(poses, sym, nocs_pose, c2n, g["gripper_in_grasp"], True, True, so, p1, se, p2)
    assert len(res) == int((st == 0).sum()) and all(r.shape == (4, 4) and r.dtype == np.float32 for r in res)
    assert all(np.array_equal(r, o) for r, o in zip(res, out[st == 0]))
    assert my_cpp.filterGraspPose([], list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"], True, False,
                                  True, [], [], g["open"]["V"], g["open"]["F"], g["enclosed"]["V"], g["enclosed"]["F"],
                                  p1, p2, 0.0005, False) == []
    with pytest.raises(ValueError):
        my_cpp.filterGraspPose(list(poses), list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"], True,
                               False, True, [], [], g["open"]["V"], g["open"]["F"], g["enclosed"]["V"],
                               g["enclosed"]["F"], p1[:, :2], p2, 0.0005, False)


@pytest.mark.parametrize("mode", [0, 1])
def test_sdf_lookup_vs_oracles(cuda, mode):
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy
    from oracle import filter_ref, sdf_ref
    g = make_gripper_proxy()["open"]
    s = Sdf3D(g["sdf"], g["origin"], g["res"])
    rng = np.random.RandomState(0)
    dims = np.array(g["sdf"].shape)
    gc = rng.uniform(-3, 1, (5000, 3)) * 0 + rng.uniform(-4, dims.max() + 4, (5000, 3))
    gc[:50] = np.round(gc[:50])                # exact lattice points
    gc[50:60] = dims - 1                       # the last cell (hi corner out of bounds)
    gc[60:80] += 0.5 - (gc[60:80] % 1)         # exact .5 ties for round-half-even
    gc = gc.astype(np.float32)
    out = s._signed_distance(gc.T, fast=(mode == 1)).cpu().numpy()
    ref32 = filter_ref.sdf_lookup_ref(g["sdf"], gc, mode)
    assert np.array_equal(out.view(np.uint32), ref32.view(np.uint32))
    ref64 = sdf_ref.signed_distance(g["sdf"], gc.T) if mode == 0 else sdf_ref.signed_distance_nearest(g["sdf"], gc.T)
    assert np.abs(out - ref64).max() < 1e-6


# ------------------------------------------------------------------ PointNet++ primitives
def test_pn2_primitives_vs_reference_golden(cuda, golden_dir):
    from catgrasp_b200 import pointnet2 as pn2
    g = np.load(os.path.join(golden_dir, "pn2_primitives.npz"))
    xyz = torch.from_numpy(g["xyz"]).cuda()
    S, K = g["fps"].shape[1], g["ball"].shape[2]
    fps = pn2.farthest_point_sample(xyz, S, start_idx=torch.from_numpy(g["start"]))
    assert fps.dtype == torch.int64 and np.array_equal(fps.cpu().numpy(), g["fps"])
    new_xyz = pn2.index_points(xyz, fps)
    assert np.array_equal(new_xyz.cpu().numpy(), g["new_xyz"])
    ball = pn2.query_ball_point(float(g["radius"]), K, xyz, new_xyz)
    assert np.array_equal(ball.cpu().numpy(), g["ball"])
    nx, npts, gxyz, fidx = pn2.sample_and_group(S, float(g["radius"]), K, xyz, torch.from_numpy(g["feats"]).cuda(),
                                                returnfps=True, start_idx=torch.from_numpy(g["start"]))
    assert np.array_equal(npts.cpu().numpy(), g["g_new_points"])
    assert np.array_equal(gxyz.cpu().numpy(), g["g_grouped_xyz"])
    sq = pn2.square_distance(new_xyz[:, :16], xyz[:, :256])
    assert np.array_equal(sq.cpu().numpy(), g["sq"])
    # camera-frame cloud: noisy expanded form, still identical to the reference
    cam = torch.from_numpy(g["cam"]).cuda()
    cfps = pn2.farthest_point_sample(cam, 64, start_idx=torch.from_numpy(g["cam_start"]))
    assert np.array_equal(cfps.cpu().numpy(), g["cam_fps"])
    cnew = pn2.index_points(cam, cfps)
    assert np.array_equal(pn2.square_distance(cnew, cam).cpu().numpy(), g["cam_sq"])
    assert np.array_equal(pn2.query_ball_point(0.004, 8, cam, cnew).cpu().numpy(), g["cam_ball"])
    # Appendix A1/A2 edge cases
    e = pn2.query_ball_point(1.0, 4, torch.from_numpy(g["e_xyz"]).cuda(), torch.from_numpy(g["e_new"]).cuda())
    assert np.array_equal(e.cpu().numpy(), g["e_ball"])
    a, b = pn2.sample_and_group_all(xyz, torch.from_numpy(g["feats"]).cuda())
    assert a.shape == (2, 1, 3) and b.shape == (2, 1, 2048, 6)


@pytest.mark.parametrize("N,npoint", [(20000, 1024), (40000, 256), (777, 777)])
def test_fps_ballquery_scene_sizes_vs_oracle(cuda, N, npoint):
    """BASELINE scene sizes (20k / 40k points): exact index parity with the numpy oracle; both
    shared-memory layouts of the FPS kernel (xyz resident for N <= 14080, streamed above)."""
    from catgrasp_b200 import pointnet2 as pn2
    from catgrasp_b200.synthetic import make_pile
    from oracle import pn2_ref
    scene = make_pile(N, n_objects=max(4, N // 900), seed=5)
    xyz = (scene["cloud_xyz"] - scene["cloud_xyz"].mean(0)).astype(np.float32)[None]
    start = np.array([N // 3])
    ref = pn2_ref.farthest_point_sample(xyz, npoint, start)
    got = pn2.farthest_point_sample(torch.from_numpy(xyz).cuda(), npoint, start_idx=torch.from_numpy(start))
    assert np.array_equal(got.cpu().numpy(), ref)
    assert len(set(ref[0].tolist())) == npoint or N == npoint
    S = min(npoint, 128)
    new_xyz = xyz[:, ref[0, :S]]
    rb = pn2_ref.query_ball_point(0.004, 32, xyz, new_xyz)
    gb = pn2.query_ball_point(0.004, 32, torch.from_numpy(xyz).cuda(), torch.from_numpy(new_xyz).cuda())
    assert np.array_equal(gb.cpu().numpy(), rb)
    # the reference's order: the in-ball indices ascend, then the pad repeats the first one (pointnet2.py:94-97)
    for row in rb.reshape(-1, rb.shape[-1]):
        k = 1
        while k < len(row) and row[k] > row[k - 1]:
            k += 1
        assert (row[k:] == row[0]).all()
    # cluster kernel (registers + DSMEM exchange) == round-1 single-CTA kernel (shared-memory distances), two clouds at once
    import ctypes as C  # noqa: F401
    from catgrasp_b200 import _lib
    ctx = _lib.Context.get(0)
    x2 = torch.from_numpy(np.concatenate([xyz, xyz[:, ::-1].copy()])).cuda().contiguous()
    st2 = torch.tensor([N // 3, 5 % N], dtype=torch.int32, device="cuda")
    o1 = torch.empty((2, npoint), dtype=torch.int32, device="cuda")
    o2 = torch.empty_like(o1)
    ctx.use_torch_stream()
    ctx.check(ctx.lib.cg_fps_dev(ctx.h, _lib.ptr(x2), 2, N, npoint, _lib.ptr(st2), _lib.ptr(o1)))
    ctx.check(ctx.lib.cg_fps_single_cta_dev(ctx.h, _lib.ptr(x2), 2, N, npoint, _lib.ptr(st2), _lib.ptr(o2)))
    assert torch.equal(o1, o2) and np.array_equal(o1[0].cpu().numpy(), ref[0])


def test_fps_large_cloud_no_cap(cuda):
    """60 000 points (beyond the round-1 shared-memory cap of 56 320, inside the cluster-size-8 cap of 65 536): equal to
    the numpy oracle on the first rounds and self-consistent (distinct indices, first index = start)."""
    from catgrasp_b200 import pointnet2 as pn2
    from oracle import pn2_ref
    rng = np.random.RandomState(0)
    xyz = rng.uniform(-1, 1, (1, 60000, 3)).astype(np.float32)
    got = pn2.farthest_point_sample(torch.from_numpy(xyz).cuda(), 512, start_idx=torch.tensor([77])).cpu().numpy()
    assert got[0, 0] == 77 and len(set(got[0].tolist())) == 512
    ref = pn2_ref.farthest_point_sample(xyz, 24, np.array([77]))
    assert np.array_equal(got[:, :24], ref)


# ------------------------------------------------------------------ occupancy grid (my_cpp.makeOccupancyGridFromCloudScan)
@pytest.mark.parametrize("res,n_points", [(0.002, 3000), (0.001, 6000)])
def test_occupancy_grid_bit_exact_vs_oracle(cuda, res, n_points):
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.synthetic import make_pile
    from oracle import filter_ref
    scene = make_pile(n_points, n_objects=4, seed=6)
    K = np.array([[2000.0, 0, 1032], [0, 2000.0, 772], [0, 0, 1]])
    out = my_cpp.makeOccupancyGridFromCloudScan(scene["cloud_xyz"], K, res)
    flags, org, dims = filter_ref.occupancy_ref(scene["cloud_xyz"], res)
    idx = np.argwhere(flags > 0)
    ref = (org[None, :] + idx.astype(np.float32) * np.float32(res)).astype(np.float32)
    assert out.dtype == np.float32 and out.shape == ref.shape and out.shape[0] > 100
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    with pytest.raises(ValueError):
        my_cpp.makeOccupancyGridFromCloudScan(scene["cloud_xyz"][:, :2], K, res)


# ------------------------------------------------------------------ NUNOCS 9-DoF RANSAC (aligning.py:83-119)
def test_ransac9d_vs_cv2_oracle(cuda):
    from catgrasp_b200.aligning import estimate9DTransform
    from catgrasp_b200.synthetic import random_rotation
    from oracle import aligning_ref
    rng = np.random.RandomState(0)
    N = 2000
    src = np.round(rng.uniform(-0.5, 0.5, (N, 3)) / 0.01) * 0.01            # NUNOCS coordinates live on a 0.01 grid
    scales = np.array([0.02, 0.02, 0.008])
    T_true = np.eye(4)
    T_true[:3, :3] = random_rotation(rng) @ np.diag(scales)
    T_true[:3, 3] = [0.01, -0.02, 0.69]
    tgt = (T_true @ np.c_[src, np.ones(N)].T).T[:, :3] + rng.normal(0, 0.0004, (N, 3))
    bad = rng.rand(N) < 0.3                                                 # wrong NUNOCS predictions (the target stays on the object)
    src[bad] = np.round(rng.uniform(-0.5, 0.5, (bad.sum(), 3)) / 0.01) * 0.01
    kw = dict(PassThreshold=0.003, max_iter=600, max_scale=[0.05, 0.05, 0.05], min_scale=[0.005, 0.005, 0.001],
              max_dimensions=np.array([1.2, 1.2, 1.2]))
    np.random.seed(1)
    Tg, ing = estimate9DTransform(source=src, target=tgt, **kw)
    after_g = np.random.rand()
    np.random.seed(1)
    Tr, inr = aligning_ref.estimate9DTransform(source=src, target=tgt, **kw)
    assert np.random.rand() == after_g                                     # identical RNG consumption
    assert Tg is not None and Tr is not None
    rg, rr = len(ing) / N, len(inr) / N
    assert rg > 0.6 and abs(rg - rr) <= 2.0 / N
    if np.array_equal(ing, inr):                                           # same hypothesis won: transforms agree
        assert np.abs(Tg - Tr).max() < 1e-7
    sc = np.linalg.norm(Tg[:3, :3], axis=0)
    assert np.abs(sc - scales).max() < 2e-3 and np.linalg.det(Tg[:3, :3]) > 0
    # nothing passes impossible gates -> (None, None), like aligning.py:105-106
    np.random.seed(1)
    assert estimate9DTransform(source=src, target=tgt, PassThreshold=0.003, max_iter=50, max_scale=[1e-6] * 3,
                               min_scale=[0, 0, 0]) == (None, None)


def test_nunocs_predict_full_surface(cuda, tmp_path):
    """NunocsPredicter.predict keeps the reference's return/attribute contract (predicter.py:135-203)."""
    from catgrasp_b200.predicter import NunocsPredicter
    from catgrasp_b200.synthetic import make_pile, write_artifacts
    ndir = write_artifacts(str(tmp_path / "artifacts-78"), "seg", n_pts=512, seed=1)
    npred = NunocsPredicter("nut", artifact_dir=ndir)
    npred.ransac_max_iter = 200
    scene = make_pile(1500, n_objects=3, seed=21)
    obj = scene["object_id"] == 1
    data = {"cloud_xyz": scene["cloud_xyz"][obj], "cloud_normal": scene["cloud_normal"][obj]}
    np.random.seed(0)
    nocs_cloud, transform = npred.predict(copy.deepcopy(data))
    assert "cloud_xyz_original" in npred.data_transformed
    if transform is None:                       # random weights rarely yield a consistent pose: the reference returns (None, None)
        assert nocs_cloud is None
    else:
        assert nocs_cloud.shape == (512, 3) and transform.shape == (4, 4)
        assert hasattr(npred, "best_ratio") and np.array_equal(npred.nocs_pose, transform)


# ------------------------------------------------------------------ BASELINE.json configs as parity cases
@pytest.mark.parametrize("engine", _engines())
@pytest.mark.parametrize("N", [1024, 2048])
def test_k1_single_object_crop_vs_oracle(cls_net, N, engine):
    """configs[0] (K1): 1024-pt crop, 64 candidates; N=2048 is the shipped config_grasp.yml n_pts (replace=True draw)."""
    from catgrasp_b200.predicter import draw_subsample_ids
    from catgrasp_b200.synthetic import make_candidates, make_pile
    from oracle.transforms_ref import predict_batch
    net, sd = cls_net
    net.ctx.set_engine(engine)
    scene = make_pile(1024, n_objects=1, seed=3)
    poses = make_candidates(scene["cloud_xyz"], scene["cloud_normal"], 64, seed=4)
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    np.random.seed(0)
    ref = predict_batch(sd, {"n_pts": N}, data, poses)
    np.random.seed(0)
    ids = draw_subsample_ids(1024, N, count=64)
    probs, _ = net.graspq_host(scene["cloud_xyz"], scene["cloud_normal"], poses, ids)
    assert max(np.abs(probs[b] - ref[b][2]).max() for b in range(64)) < PROB_TOL


def test_k3_k5_collision_scale_subset_exact(cuda):
    """configs[2] / configs[4] shapes for the collision half: 16 384 candidates against a 40 000-pt scene, and
    1 048 576 candidates (collision only, `adjust_collision_pose=False` like generate_grasp.py:97).  Poses are
    independent, so a random subset re-evaluated by the CPU oracle must agree bit for bit."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_candidates, make_gripper_proxy, make_pile
    from oracle import filter_ref
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    eye = np.eye(4)
    rng = np.random.RandomState(0)
    # K3
    scene = make_pile(40000, n_objects=8, seed=1)
    obj = scene["object_id"] == 3
    p1, p2 = scene["cloud_xyz"][obj], scene["cloud_xyz"][~obj]
    poses = make_candidates(p1, scene["cloud_normal"][obj], 16384, seed=2)
    st, off, out = my_cpp.filter_grasp_pose_raw(poses, [eye], eye, eye, g["gripper_in_grasp"], True, True, so, p1, se, p2)
    sel = rng.choice(16384, 384, replace=False)
    rst, roff, rout = filter_ref.filter_ref(poses[sel], [eye], eye, eye, g["gripper_in_grasp"], True, True, 0, g["open"],
                                            p1, g["enclosed"], p2)
    assert np.array_equal(st[sel], rst) and np.array_equal(off[sel], roff)
    assert np.array_equal(out[sel].view(np.uint32), rout.view(np.uint32))
    assert 0 < (st == 0).sum() < 16384
    # K5: 1M candidates = 4096 distinct poses x 256 jittered copies, object points only
    base = make_candidates(p1, scene["cloud_normal"][obj], 4096, seed=5)
    big = np.repeat(base, 256, axis=0)
    big[:, :3, 3] += rng.normal(0, 0.0005, (big.shape[0], 3))
    st, off, out = my_cpp.filter_grasp_pose_raw(big, [eye], eye, eye, g["gripper_in_grasp"], True, False, so, p1, None,
                                                np.zeros((0, 3)))
    assert st.shape == (1048576,)
    sel = rng.choice(big.shape[0], 512, replace=False)
    rst, roff, rout = filter_ref.filter_ref(big[sel], [eye], eye, eye, g["gripper_in_grasp"], True, False, 0, g["open"], p1,
                                            None, np.zeros((0, 3)))
    assert np.array_equal(st[sel], rst) and np.array_equal(off[sel], roff)
    assert np.array_equal(out[sel].view(np.uint32), rout.view(np.uint32))
    assert set(np.unique(off).tolist()) <= {-1, 0}          # no lateral search when adjust_collision_pose is off


def test_k3_k4_graspq_scale_properties(cls_net):
    """configs[2] / configs[3] shapes for the network half: 16 384 candidates on a 40 000-pt scene and a mixed batch of
    8 scenes; size-independent properties + agreement of the two tensor-core engines."""
    from catgrasp_b200.synthetic import make_candidates, make_pile
    net, net_sd = cls_net
    M, B, N = 40000, 16384, 1024
    scene = make_pile(M, n_objects=8, seed=1)
    poses = make_candidates(scene["cloud_xyz"], scene["cloud_normal"], B, seed=2)
    rng = np.random.RandomState(0)
    ids = np.stack([rng.permutation(M)[:N] for _ in range(128)]).astype(np.int32)
    ids = np.ascontiguousarray(np.tile(ids, (B // 128, 1)))
    out = {}
    for e in (1, 2, 3):
        net.ctx.set_engine(e)
        out[e], _ = net.graspq_host(scene["cloud_xyz"], scene["cloud_normal"], poses, ids)
        assert np.isfinite(out[e]).all() and np.abs(out[e].sum(1) - 1).max() < 1e-5
    assert np.abs(out[1] - out[2]).max() < PROB_TOL / 4
    assert np.abs(out[1] - out[3]).max() < PROB_TOL / 4
    sel = np.random.RandomState(3).choice(B, 128, replace=False)          # K3 sample against the CPU oracle
    ref = _oracle_probs(net_sd, scene["cloud_xyz"], scene["cloud_normal"], poses[sel], ids[sel])
    for e in (1, 2, 3):
        assert np.abs(out[e][sel] - ref).max() < PROB_TOL, e
    # K4: 8 independent scenes through the same handle give the same answers as one by one (no cross-call state)
    net.ctx.set_engine(3)
    scenes = [make_pile(20000, seed=10 + s) for s in range(8)]
    first = []
    for s, sc in enumerate(scenes):
        ps = make_candidates(sc["cloud_xyz"], sc["cloud_normal"], 256, seed=20 + s)
        first.append(net.graspq_host(sc["cloud_xyz"], sc["cloud_normal"], ps, ids[:256] % 20000)[0].copy())
    for s in (7, 0, 3):
        sc = scenes[s]
        ps = make_candidates(sc["cloud_xyz"], sc["cloud_normal"], 256, seed=20 + s)
        again = net.graspq_host(sc["cloud_xyz"], sc["cloud_normal"], ps, ids[:256] % 20000)[0]
        assert np.array_equal(again.view(np.uint32), first[s].view(np.uint32))


def test_my_cpp_module_surface(cuda):
    """Every name exported by my_cpp/pybind.cpp:11-23 exists and behaves: CollisionManager, augmentGraspPoses."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
    cm = my_cpp.CollisionManager()
    assert cm.registerMesh(g["open"]["V"], g["open"]["F"]) == 0
    inside = np.array([[-0.02, 0.0, 0.0], [0.5, 0.5, 0.5]])                 # first point sits in the palm
    cm.registerPointCloud(inside, 0.0005)
    cm.setTransform(np.eye(4), 0)
    assert cm.isAnyCollision() is True
    far = np.eye(4); far[:3, 3] = [1.0, 1.0, 1.0]
    cm.setTransform(far, 0)
    assert cm.isAnyCollision() is False
    with pytest.raises(ValueError):
        cm.registerPointCloud(inside[:, :2], 0.0005)
    R0 = np.eye(3)
    sph = np.array([[1.0, 0.2, 0.0], [0.9, 0.0, 0.3]])
    poses = my_cpp.augmentGraspPoses(R0, np.array([0.1, 0.2, 0.7]), sph, 30.0, 0.012, 0.003, 0.005)
    assert len(poses) == (1 + 2 * 6) * 4 and all(p.shape == (4, 4) and p.dtype == np.float32 for p in poses)
    P = np.stack(poses)
    assert np.abs(np.einsum("nij,nkj->nik", P[:, :3, :3], P[:, :3, :3]) - np.eye(3)).max() < 1e-5
    assert np.allclose(P[0, :3, 3], [0.105, 0.2, 0.7], atol=1e-6) and np.allclose(P[1, :3, 3] - P[0, :3, 3], [0.003, 0, 0], atol=1e-6)


def test_c_abi_error_codes_instead_of_exit(cuda):
    """Bad arguments come back as CG_E* codes with a message (the reference printf+exit(1)s, collision_manager.cpp:17-27)."""
    import ctypes as C
    from catgrasp_b200 import _lib
    ctx = _lib.Context.get(0)
    lib = ctx.lib
    h = C.c_void_p()
    blob = np.zeros(16, np.float32)
    assert lib.cg_net_create(ctx.h, _lib.CG_NET_CLS, 10, _lib.ptr(blob), blob.size, C.byref(h)) == _lib.CG_EINVAL
    assert b"blob" in lib.cg_last_error(ctx.h)
    assert lib.cg_ctx_set_engine(ctx.h, 7) == _lib.CG_EINVAL
    x = torch.zeros((4, 3), device="cuda")
    out = torch.zeros((4,), dtype=torch.int32, device="cuda")
    assert lib.cg_fps_dev(ctx.h, _lib.ptr(x), 1, 0, 4, None, _lib.ptr(out)) == _lib.CG_EINVAL
    assert lib.cg_fps_dev(ctx.h, _lib.ptr(x), 1, 1 << 20, 4, None, _lib.ptr(out)) == _lib.CG_EINVAL     # beyond 32 points per thread
    assert lib.cg_fps_single_cta_dev(ctx.h, _lib.ptr(x), 1, 100000, 4, None, _lib.ptr(out)) == _lib.CG_EINVAL
    org = (C.c_float * 3)(0, 0, 0)
    assert lib.cg_sdf_create(ctx.h, None, 4, 4, 4, org, C.c_float(0.001), C.byref(h)) == _lib.CG_EINVAL
    with pytest.raises(_lib.CgError):
        ctx.check(lib.cg_ctx_set_engine(ctx.h, -1))
    ctx.set_engine(3)


# ------------------------------------------------------------------ reference-generated host-path goldens
# (tests/golden/make_golden_hostpath.py ran the reference's predicter.py / dataset_*.py / aligning.py to make these)
@pytest.mark.parametrize("engine", _engines())
def test_predict_batch_vs_reference_run(cuda, golden_dir, tmp_path, engine):
    """GraspPredicter.predict_batch == the reference's own predict_batch on the same data, poses and numpy seed."""
    from catgrasp_b200 import _lib
    from catgrasp_b200.predicter import GraspPredicter
    from catgrasp_b200.synthetic import write_artifacts
    g = np.load(os.path.join(golden_dir, "host_predict_batch.npz"))
    adir = write_artifacts(str(tmp_path / "artifacts-47"), "cls", n_pts=1024, seed=int(g["artifact_seed"]),
                           logit_gain=float(g["logit_gain"]))
    gp = GraspPredicter("nut", artifact_dir=adir)
    assert gp.engine in (1, 3) and gp.engine_probe["max_abs_dprob"] < PROB_TOL      # load-time gate ran on this checkpoint
    gp.engine = engine                                                              # ... and can be overridden
    try:
        for tag in ("big", "small"):
            data = {"cloud_xyz": g[f"{tag}_cloud_xyz"].astype(np.float64), "cloud_normal": g[f"{tag}_cloud_normal"].astype(np.float64)}
            np.random.seed(0)
            out = gp.predict_batch(data, list(g[f"{tag}_poses"]))
            np.testing.assert_array_equal(np.random.rand(2), g[f"{tag}_next_rand"])
            np.testing.assert_array_equal([o[0] for o in out], g[f"{tag}_labels"])
            assert np.abs(np.stack([o[2] for o in out]) - g[f"{tag}_probs"]).max() < PROB_TOL
            assert np.abs(np.array([o[1] for o in out]) - g[f"{tag}_conf"]).max() < PROB_TOL
    finally:
        _lib.Context.get(0).set_engine(3)


def _nunocs_from_golden(g, tmp_path, sd):
    from catgrasp_b200.predicter import NunocsPredicter
    from catgrasp_b200.synthetic import write_artifacts
    ndir = write_artifacts(str(tmp_path / "artifacts-78"), "seg", n_pts=8192, state_dict=sd, normalizer=(g["mean"], g["std"]))
    return NunocsPredicter("nut", artifact_dir=ndir)


def test_nunocs_predict_vs_reference_run_no_pose(cuda, golden_dir, tmp_path):
    """Random weights: the reference's predict() found no pose; same subsample, same bins (up to logit ties), same
    (None, None), same numpy-RNG consumption through transform + 2 x 10 000 RANSAC draws."""
    from catgrasp_b200.synthetic import make_state_dict
    g = np.load(os.path.join(golden_dir, "host_nunocs_random.npz"))
    npred = _nunocs_from_golden(g, tmp_path, make_state_dict("seg", 300, seed=int(g["weight_seed"])))
    data = {"cloud_xyz": g["cloud_xyz"].astype(np.float64), "cloud_normal": g["cloud_normal"].astype(np.float64)}
    np.random.seed(0)
    nocs, tf = npred.predict(copy.deepcopy(data))
    assert bool(g["returned_none"]) and nocs is None and tf is None
    np.testing.assert_array_equal(np.random.rand(2), g["next_rand"])
    np.testing.assert_array_equal(npred.data_transformed["keep_ids"], g["keep_ids"])
    np.testing.assert_array_equal(npred.data_transformed["input"].astype(np.float32), g["input"])
    assert (npred.pred_bins.reshape(-1, 3) != g["nocs_bins"]).mean() < 1e-2


def test_nunocs_predict_vs_reference_run_success_path(cuda, golden_dir, tmp_path):
    """Lattice weights: bins identical to the reference run, and predict() returns the reference's NOCS cloud, pose,
    best_ratio and nocs_pose (predicter.py:135-203)."""
    from catgrasp_b200.synthetic import make_lattice_seg_state_dict
    g = np.load(os.path.join(golden_dir, "host_nunocs_lattice.npz"))
    npred = _nunocs_from_golden(g, tmp_path, make_lattice_seg_state_dict(seed=int(g["weight_seed"]), mean=g["mean"], std=g["std"]))
    data = {"cloud_xyz": g["cloud_xyz"], "cloud_normal": g["cloud_normal"].astype(np.float64)}
    np.random.seed(0)
    nocs, tf = npred.predict(copy.deepcopy(data))
    np.testing.assert_array_equal(np.random.rand(2), g["next_rand"])
    np.testing.assert_array_equal(npred.data_transformed["keep_ids"], g["keep_ids"])
    np.testing.assert_array_equal(npred.pred_bins.reshape(-1, 3), g["nocs_bins"])
    np.testing.assert_array_equal(np.asarray(nocs, np.float32), g["nocs_cloud"])
    assert npred.best_ratio == float(g["best_ratio"])
    np.testing.assert_allclose(tf, g["transform"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(npred.nocs_pose, g["nocs_pose"], rtol=0, atol=1e-9)


def test_ransac9d_vs_reference_run(cuda, golden_dir):
    from catgrasp_b200.aligning import estimate9DTransform
    g = np.load(os.path.join(golden_dir, "host_ransac9d.npz"))
    np.random.seed(3)
    tf, inl = estimate9DTransform(source=g["source"], target=g["target"], PassThreshold=0.003, max_iter=3000,
                                  max_scale=[0.05] * 3, min_scale=[0.005, 0.005, 0.001], max_dimensions=np.array([1.2] * 3))
    np.testing.assert_array_equal(np.random.rand(2), g["next_rand"])
    np.testing.assert_allclose(tf, g["transform"], rtol=0, atol=1e-9)
    np.testing.assert_array_equal(inl, g["inliers"])


# ------------------------------------------------------------------ goldens from the compiled reference my_cpp (oracle/build_ref.py)
def _mk():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_mycpp as mk
    return mk


@pytest.mark.parametrize("k", range(12))
def test_filterGraspPose_equals_reference_build(cuda, golden_dir, k):
    """my_cpp.filterGraspPose (20 positional args, survivors only) returns exactly the survivor set the reference's own
    compiled filterGraspPose returned (pose logic = reference code, geometry predicate = gripper SDF on both sides)."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from oracle import mycpp_ref
    mk = _mk()
    g_ = np.load(os.path.join(golden_dir, "mycpp_filter.npz"))
    S, scale, mode, adjust, fdir = mk.FILTER_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), dg = mk.filter_inputs(S, scale)
    assert np.array_equal(dg, g_[f"inputs_sha_{k}"])
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
    my_cpp.register_gripper_sdf(g["enclosed"]["V"], g["enclosed"]["F"], se)
    old = my_cpp.DEFAULT_SDF_MODE
    my_cpp.DEFAULT_SDF_MODE = mode
    try:
        res = my_cpp.filterGraspPose(list(poses), list(sym), nocs_pose, c2n, np.eye(4), np.eye(4), g["gripper_in_grasp"],
                                     fdir, False, adjust, [3] * 7, [-3] * 7, g["open"]["V"], g["open"]["F"],
                                     g["enclosed"]["V"], g["enclosed"]["F"], p1, p2, 0.0005, False)
    finally:
        my_cpp.DEFAULT_SDF_MODE = old
    assert np.array_equal(mycpp_ref.sort_poses(np.stack(res)).view(np.uint32), g_[f"survivors_{k}"])


@pytest.mark.parametrize("k", range(3))
def test_occupancy_equals_reference_build(cuda, golden_dir, k):
    from catgrasp_b200 import my_cpp
    mk = _mk()
    g_ = np.load(os.path.join(golden_dir, "mycpp_occupancy.npz"))
    res, n, seed = mk.OCC_CASES[k]
    pts = mk.occupancy_inputs(n, seed)
    assert np.array_equal(mk.digest(pts), g_[f"inputs_sha_{k}"])
    out = my_cpp.makeOccupancyGridFromCloudScan(pts, np.eye(3), res)
    assert np.array_equal(np.unique(out.view(np.uint32), axis=0), g_[f"points_{k}"])


@pytest.mark.parametrize("k", range(2))
def test_filterGraspPose_with_ik_equals_reference_build(cuda, golden_dir, k):
    """filter_ik=True through the 20-argument call, the IK hook answering with the reference's own ikfast verdicts
    (recorded in tests/golden/mycpp_ik.npz)."""
    from catgrasp_b200 import my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from oracle import mycpp_ref
    mk = _mk()
    g_ = np.load(os.path.join(golden_dir, "mycpp_filter.npz"))
    S, scale, mode, adjust, fdir = mk.IK_CASES[k]
    (p1, p2, poses, sym, nocs_pose, c2n, g), dg = mk.filter_inputs(S, scale)
    cam, ee = mk.ik_frames()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    my_cpp.register_gripper_sdf(g["open"]["V"], g["open"]["F"], so)
    my_cpp.register_gripper_sdf(g["enclosed"]["V"], g["enclosed"]["F"], se)
    old = my_cpp.DEFAULT_SDF_MODE
    my_cpp.DEFAULT_SDF_MODE = mode
    my_cpp.set_ik_solver(mk.recorded_ik_solver(golden_dir, k))
    try:
        res = my_cpp.filterGraspPose(list(poses), list(sym), nocs_pose, c2n, cam, ee, g["gripper_in_grasp"], fdir, True, adjust,
                                     list(mk.IK_UPPER), list(mk.IK_LOWER), g["open"]["V"], g["open"]["F"], g["enclosed"]["V"],
                                     g["enclosed"]["F"], p1, p2, 0.0005, False)
    finally:
        my_cpp.DEFAULT_SDF_MODE = old
        my_cpp.set_ik_solver(None)
    assert np.array_equal(mycpp_ref.sort_poses(np.stack(res)).view(np.uint32), g_[f"ik_survivors_{k}"])


# ------------------------------------------------------------------ cone pose enumeration (grasp_sampler.py:131-298), SURVEY 8f F3
@pytest.mark.parametrize("k", range(3))
def test_cone_grasp_poses_vs_reference_run(cuda, golden_dir, k):
    """cone_grasp_poses == the poses the reference's own PointConeGraspSampler.sample_grasps handed to filterGraspPose
    (tests/golden/make_golden_cone.py), same numpy-RNG consumption; float64 to 1e-13, float32 copy = narrowed values."""
    import test_cone_golden as tc
    from catgrasp_b200 import grasp_sampler as gs
    g = np.load(os.path.join(golden_dir, "cone_poses.npz"))
    c = tc.CASES[k]
    pts, nrm = tc.case_inputs(c)
    np.random.seed(7)
    p64, p32 = gs.cone_grasp_poses(pts, nrm, tc.HAND_DEPTH, tc.INIT_BITE, max_num_samples=c["max_num_samples"],
                                   n_sphere_dir=c["n_sphere_dir"], approach_step=c["approach_step"],
                                   center_ob_between_gripper=c["center"])
    np.testing.assert_array_equal(np.random.rand(2), g[f"next_rand_{k}"])
    ref = g[f"poses_{k}"]
    assert tuple(p64.shape) == ref.shape and p64.is_cuda and p32.dtype == torch.float32
    assert np.abs(p64.cpu().numpy() - ref).max() < 1e-13
    assert np.abs(p32.cpu().numpy().astype(np.float64) - ref.astype(np.float32)).max() < 1.3e-7   # <= 1 ulp at |x| < 1


def test_cone_poses_feed_filter_on_device(cuda):
    """The device-resident float32 poses go straight into the collision filter and give the same verdicts as the same
    poses passed from the host (the reference's route: list of numpy 4x4 -> pybind -> float32)."""
    from catgrasp_b200 import grasp_sampler as gs, my_cpp
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy, make_pile
    scene = make_pile(2400, n_objects=6, seed=43)
    obj = scene["object_id"] == 3
    p1, p2 = scene["cloud_xyz"][obj], scene["cloud_xyz"][~obj]
    np.random.seed(1)
    p64, p32 = gs.cone_grasp_poses(p1.copy(), scene["cloud_normal"][obj].copy(), 0.012, 0.002, max_num_samples=12,
                                   n_sphere_dir=6, approach_step=0.004)
    g = make_gripper_proxy()
    so = Sdf3D(g["open"]["sdf"], g["open"]["origin"], g["open"]["res"])
    se = Sdf3D(g["enclosed"]["sdf"], g["enclosed"]["origin"], g["enclosed"]["res"])
    eye = np.eye(4)
    dst, doff, dout = my_cpp.filter_grasp_pose_raw(p32, [eye], eye, eye, g["gripper_in_grasp"], True, True, so, p1, se, p2)
    hst, hoff, hout = my_cpp.filter_grasp_pose_raw(p64.cpu().numpy(), [eye], eye, eye, g["gripper_in_grasp"], True, True, so,
                                                   p1, se, p2)
    assert np.array_equal(dst.cpu().numpy(), hst) and np.array_equal(doff.cpu().numpy(), hoff)
    assert np.array_equal(dout.cpu().numpy().view(np.uint32), hout.view(np.uint32))
    assert p32.shape[0] > 0 and p32.shape[0] % ((1 + 6 * 6) * 3) == 0 and (hst == 0).any() and (hst != 0).any()


def test_sdf_lookups_vs_reference_run(cuda, golden_dir):
    """Sdf3D lookups on the GPU vs values computed by the reference's own meshpy Sdf3D (tests/golden/make_golden_sdf.py)."""
    from catgrasp_b200.sdf import Sdf3D
    from catgrasp_b200.synthetic import make_gripper_proxy
    g_ = np.load(os.path.join(golden_dir, "sdf_lookup.npz"))
    g = make_gripper_proxy()["open"]
    s = Sdf3D(g["sdf"], g["origin"], g["res"])
    gc = g_["coords"]
    tri = s._signed_distance(gc.T, fast=False).cpu().numpy()
    near = s._signed_distance(gc.T, fast=True).cpu().numpy()
    assert np.abs(tri - g_["trilinear"]).max() < 1e-6
    np.testing.assert_allclose(near, g_["nearest_clamped"], rtol=0, atol=1e-7)


# ------------------------------------------------------------------ affordance transfer (run_grasp_simulation.py:50-107), SURVEY 8f F4
def test_grasp_affordance_vs_reference_run(cuda, golden_dir):
    """compute_grasp_affordance on the GPU vs the reference's own worker (tests/golden/make_golden_affordance.py): same
    dropped grasps, same contact-patch sizes, scores equal up to nearest-neighbour ties (<= 1e-3) and equal to the
    tie-free oracle formulation to 1e-12."""
    import test_affordance_golden as ta
    from scipy.spatial import cKDTree
    from catgrasp_b200.affordance import compute_grasp_affordance
    from oracle import affordance_ref
    g = np.load(os.path.join(golden_dir, "affordance.npz"))
    full, affordance, down, down_n, boxes, fmig, poses = ta.affordance_case()
    p, ncon = compute_grasp_affordance(poses, fmig, down, down_n, full, affordance, boxes, [[0, 1, 0], [0, -1, 0]], 0.005)
    assert np.array_equal(np.isnan(p), np.isnan(g["p_T_given_G"]))
    np.testing.assert_array_equal(ncon, g["n_contacts"])
    ok = ~np.isnan(p)
    assert np.abs(p[ok] - g["p_T_given_G"][ok]).max() < 1e-3
    _, nn = cKDTree(full).query(down)
    po, _ = affordance_ref.grasp_affordance_pointwise_nn(poses, fmig, down, down_n, affordance[nn], boxes, [1, -1], 0.005)
    assert np.abs(p[ok] - po[ok]).max() < 1e-12
    with pytest.raises(RuntimeError):
        compute_grasp_affordance(poses[:1], fmig, down, down_n, full, affordance, boxes, [[1, 0, 0], [0, -1, 0]], 0.005)


# ------------------------------------------------------------------ subset draws (round 2)
@pytest.mark.parametrize("M,n_pts,count", [(20000, 1024, 96), (3000, 1024, 17), (1024, 1024, 5), (700, 1024, 9), (1, 1, 4),
                                           (40000, 2048, 8)])
def test_device_draw_vs_oracle(cls_net, M, n_pts, count):
    """cg_draw_ids_dev == oracle/draw_ref.py bit for bit (integer work), including a non-zero first candidate."""
    from oracle.draw_ref import draw_ids
    net, _ = cls_net
    got = net.draw_ids_dev(M, n_pts, count, seed=0x1234_5678_9abc, first_candidate=5).cpu().numpy()
    assert np.array_equal(got, draw_ids(M, n_pts, count, 0x1234_5678_9abc, 5))


def test_device_draw_statistics(cuda, tmp_path):
    """subsample="device" is NOT the reference's random stream (documented) but the same distribution:
    (1) every candidate gets n_pts distinct in-range indices; (2) pooled index frequencies are uniform (chi-square);
    (3) the grasp-Q expectation p_G = sum_k k p_k / 10 (run_grasp_simulation.py:311) of device-drawn subsets is
    distributed like that of numpy-drawn subsets (two-sample KS test over 512 candidates, p > 1e-3);
    (4) it consumes exactly one value of the global numpy generator and is reproducible under np.random.seed."""
    from scipy import stats
    from catgrasp_b200.predicter import GraspPredicter
    from catgrasp_b200.synthetic import make_candidates, make_pile, write_artifacts
    adir = write_artifacts(str(tmp_path / "artifacts-47"), "cls", n_pts=512, seed=0, logit_gain=6.0)
    gp = GraspPredicter("nut", artifact_dir=adir)
    scene = make_pile(6000, n_objects=4, seed=31)
    data = {"cloud_xyz": scene["cloud_xyz"], "cloud_normal": scene["cloud_normal"]}
    poses = list(make_candidates(scene["cloud_xyz"], scene["cloud_normal"], 8, seed=32)) * 64       # 8 poses x 64 draws each
    ids = gp.model.draw_ids_dev(6000, 512, 4096, seed=7).cpu().numpy()
    assert ids.min() >= 0 and ids.max() < 6000 and all(len(set(r.tolist())) == 512 for r in ids[:256])
    cnt = np.bincount(ids.ravel(), minlength=6000)
    e = ids.size / 6000
    assert 0.8 < ((cnt - e) ** 2 / e).sum() / 5999 < 1.1
    np.random.seed(1)
    host = gp.predict_batch(data, poses, subsample="host")
    np.random.seed(1)
    dev = gp.predict_batch(data, poses, subsample="device")
    after = np.random.rand()
    np.random.seed(1)
    dev2 = gp.predict_batch(data, poses, subsample="device")
    assert all(np.array_equal(a[2], b[2]) for a, b in zip(dev, dev2))
    np.random.seed(1)
    np.random.randint(0, 2 ** 63 - 1, dtype=np.int64)
    assert np.random.rand() == after                                  # one draw consumed
    pg = lambda out: np.array([(np.arange(10) * o[2]).sum() / 10 for o in out]).reshape(64, 8)   # noqa: E731
    ph, pd = pg(host), pg(dev)
    for k in range(8):                                                # per pose: same sampling distribution of p_G
        assert stats.ks_2samp(ph[:, k], pd[:, k]).pvalue > 1e-3, k
    assert np.abs(ph.mean(0) - pd.mean(0)).max() < 4 * (ph.std(0).max() / 8 + 1e-6)


def test_predict_batch_pipeline_chunks_equal_single_call(cuda, golden_dir, tmp_path):
    """The pipelined host draw (C continuation of numpy's MT19937 on a worker thread, chunk by chunk) returns the
    reference run's probabilities and leaves numpy's generator where the reference leaves it, for any chunk size."""
    from catgrasp_b200.predicter import GraspPredicter
    from catgrasp_b200.synthetic import write_artifacts
    g = np.load(os.path.join(golden_dir, "host_predict_batch.npz"))
    adir = write_artifacts(str(tmp_path / "artifacts-47"), "cls", n_pts=1024, seed=int(g["artifact_seed"]),
                           logit_gain=float(g["logit_gain"]))
    gp = GraspPredicter("nut", artifact_dir=adir)
    for chunk in (5, 1, 512):
        gp.chunk = chunk
        for tag in ("big", "small"):
            data = {"cloud_xyz": g[f"{tag}_cloud_xyz"].astype(np.float64), "cloud_normal": g[f"{tag}_cloud_normal"].astype(np.float64)}
            np.random.seed(0)
            out = gp.predict_batch(data, list(g[f"{tag}_poses"]))
            np.testing.assert_array_equal(np.random.rand(2), g[f"{tag}_next_rand"])
            np.testing.assert_array_equal([o[0] for o in out], g[f"{tag}_labels"])
            assert np.abs(np.stack([o[2] for o in out]) - g[f"{tag}_probs"]).max() < PROB_TOL
