"""Set-abstraction / feature-propagation stacks.

CPU: oracle/pn2_modules_ref.py driven by the numpy primitive oracle (oracle/pn2_ref.py) reproduces the golden file
that was generated with the REFERENCE's own primitives (tests/golden/make_golden_modules.py).
GPU (-m gpu): catgrasp_b200.pointnet2.PointNetSetAbstraction / PointNetFeaturePropagation through the C ABI:
sampled / grouped indices and 3-NN indices bit-exact, features within 2e-5 (+1e-5 relative).
"""
import os
import types

import numpy as np
import pytest
import torch

from catgrasp_b200.synthetic import make_mlp_state_dict

SPECS = dict(sa1=([6, 64, 64, 128], 11, True), sa2=([131, 128, 128, 256], 12, True), sa3=([259, 256, 512], 13, True),
             fp3=([768, 256, 256], 14, False), fp2=([384, 256, 128], 15, False), fp1=([131, 128, 128, 64], 16, False))


def _sd(name):
    dims, seed, c2 = SPECS[name]
    return make_mlp_state_dict(dims, seed=seed, conv2d=c2), len(dims) - 1


def _numpy_prims(starts):
    """Stand-in for the reference's pointnet2 module built from the numpy oracle; FPS starts are explicit."""
    from oracle import pn2_ref
    it = iter(starts)

    def sample_and_group(npoint, radius, nsample, xyz, points):
        nx, npts, _, _ = pn2_ref.sample_and_group(npoint, radius, nsample, xyz.numpy(), None if points is None else points.numpy(),
                                                  next(it))
        return torch.from_numpy(nx), torch.from_numpy(npts)

    def sample_and_group_all(xyz, points):
        B, N, C = xyz.shape
        new_xyz = torch.zeros(B, 1, C)
        g = xyz.view(B, 1, N, C)
        return new_xyz, (torch.cat([g, points.view(B, 1, N, -1)], dim=-1) if points is not None else g)

    return types.SimpleNamespace(
        sample_and_group=sample_and_group, sample_and_group_all=sample_and_group_all,
        square_distance=lambda a, b: torch.from_numpy(pn2_ref.square_distance(a.numpy(), b.numpy())),
        index_points=lambda p, i: torch.from_numpy(pn2_ref.index_points(p.numpy(), i.numpy())))


def test_module_oracle_reproduces_reference_primitive_run(golden_dir):
    from oracle.pn2_modules_ref import feature_propagation, set_abstraction
    g = np.load(os.path.join(golden_dir, "pn2_modules.npz"))
    prims = _numpy_prims([g["start1"], g["start2"]])
    xyz, nrm = torch.from_numpy(g["xyz"]), torch.from_numpy(g["nrm"])
    sd, n = _sd("sa1")
    l1_xyz, l1_pts, grouped = set_abstraction(prims, sd, n, 256, 0.2, 32, False, xyz, nrm)
    assert np.array_equal(l1_xyz.numpy(), g["l1_xyz"]) and np.array_equal(grouped.numpy()[:, :8], g["grouped1"])
    assert np.abs(l1_pts.numpy() - g["l1_pts"]).max() < 1e-5
    sd, n = _sd("sa2")
    l2_xyz, l2_pts, _ = set_abstraction(prims, sd, n, 64, 0.4, 16, False, torch.from_numpy(g["l1_xyz"]), torch.from_numpy(g["l1_pts"]))
    assert np.array_equal(l2_xyz.numpy(), g["l2_xyz"]) and np.abs(l2_pts.numpy() - g["l2_pts"]).max() < 1e-5
    sd, n = _sd("fp2")
    f1, idx2, w2 = feature_propagation(prims, sd, n, torch.from_numpy(g["l1_xyz"]), torch.from_numpy(g["l2_xyz"]),
                                       torch.from_numpy(g["l1_pts"]), torch.from_numpy(g["f2"]))
    assert np.array_equal(idx2.numpy(), g["idx2"]) and np.abs(w2.numpy() - g["w2"]).max() < 1e-6
    assert np.abs(f1.numpy() - g["f1"]).max() < 1e-5
    f0, idx1, w1 = _fp1_oracle(g)
    assert np.array_equal(idx1.numpy(), g["idx1"]) and np.abs(w1.numpy() - g["w1"]).max() < 1e-6
    assert np.abs(f0.numpy()[:, :, g["f0_cols"]] - g["f0_sample"]).max() < 1e-5


def _fp1_oracle(g):
    """FP1 (256 -> 3000 points) by the module oracle on the golden inputs; the golden file keeps a sample of its output."""
    from oracle.pn2_modules_ref import feature_propagation
    sd, n = _sd("fp1")
    return feature_propagation(_numpy_prims([]), sd, n, torch.from_numpy(g["xyz"]), torch.from_numpy(g["l1_xyz"]),
                               torch.from_numpy(g["nrm"]), torch.from_numpy(g["f1"]))


@pytest.mark.gpu
def test_sa_fp_stack_vs_golden(golden_dir):
    from catgrasp_b200.pointnet2 import PointNetFeaturePropagation, PointNetSetAbstraction
    assert torch.cuda.is_available(), "GPU tests need a B200; there is no CPU fallback"
    dev = torch.device("cuda", 0)
    g = np.load(os.path.join(golden_dir, "pn2_modules.npz"))
    t = lambda k: torch.from_numpy(g[k]).to(dev)   # noqa: E731
    tol = lambda a, ref: np.abs(a.cpu().numpy() - ref).max() < 2e-5 + 1e-5 * np.abs(ref).max()   # noqa: E731
    sa1 = PointNetSetAbstraction(256, 0.2, 32, 6, [64, 64, 128], False, _sd("sa1")[0], device=0)
    l1_xyz, l1_pts = sa1(t("xyz"), t("nrm"), start_idx=g["start1"])
    assert np.array_equal(l1_xyz.cpu().numpy(), g["l1_xyz"])               # FPS indices exact -> coordinates exact
    assert tol(l1_pts, g["l1_pts"])
    sa2 = PointNetSetAbstraction(64, 0.4, 16, 131, [128, 128, 256], False, _sd("sa2")[0], device=0)
    l2_xyz, l2_pts = sa2(t("l1_xyz"), t("l1_pts"), start_idx=g["start2"])   # golden inputs: layers are tested one by one
    assert np.array_equal(l2_xyz.cpu().numpy(), g["l2_xyz"]) and tol(l2_pts, g["l2_pts"])
    sa3 = PointNetSetAbstraction(None, None, None, 259, [256, 512], True, _sd("sa3")[0], device=0)
    _, l3_pts = sa3(t("l2_xyz"), t("l2_pts"))
    assert tol(l3_pts, g["l3_pts"])
    fp3 = PointNetFeaturePropagation(768, [256, 256], _sd("fp3")[0], device=0)
    f2 = fp3(t("l2_xyz"), torch.zeros((2, 3, 1), device=dev), t("l2_pts"), t("l3_pts"))
    assert tol(f2, g["f2"])
    fp2 = PointNetFeaturePropagation(384, [256, 128], _sd("fp2")[0], device=0)
    f1, idx2, w2 = fp2(t("l1_xyz"), t("l2_xyz"), t("l1_pts"), t("f2"), return_nn=True)
    assert np.array_equal(idx2.cpu().numpy(), g["idx2"]) and np.abs(w2.cpu().numpy() - g["w2"]).max() < 1e-6
    assert tol(f1, g["f1"])
    fp1 = PointNetFeaturePropagation(131, [128, 128, 64], _sd("fp1")[0], device=0)
    f0, idx1, w1 = fp1(t("xyz"), t("l1_xyz"), t("nrm"), t("f1"), return_nn=True)
    assert np.array_equal(idx1.cpu().numpy(), g["idx1"]) and np.abs(w1.cpu().numpy() - g["w1"]).max() < 1e-6
    assert tol(f0[:, :, torch.from_numpy(g["f0_cols"]).to(dev)], g["f0_sample"])
    assert tol(f0, _fp1_oracle(g)[0].numpy())                              # every point, against the oracle
    # chained end to end (own outputs feed the next layer): same answer
    l1x, l1p = sa1(t("xyz"), t("nrm"), start_idx=g["start1"])
    l2x, l2p = sa2(l1x, l1p, start_idx=g["start2"])
    assert np.array_equal(l2x.cpu().numpy(), g["l2_xyz"]) and tol(l2p, g["l2_pts"])


@pytest.mark.gpu
def test_three_interp_error_paths():
    import ctypes as C
    from catgrasp_b200 import _lib
    ctx = _lib.Context.get(0)
    x = torch.zeros((1, 8, 3), device="cuda")
    f = torch.zeros((1, 2, 4), device="cuda")
    out = torch.zeros((1, 8, 4), device="cuda")
    rc = ctx.lib.cg_three_interp_dev(ctx.h, _lib.ptr(x), _lib.ptr(x), None, 0, _lib.ptr(f), 4, 1, 8, 2, _lib.ptr(out), None, None)
    assert rc == _lib.CG_EINVAL and b"S >= 3" in ctx.lib.cg_last_error(ctx.h)
    h = C.c_void_p()
    assert ctx.lib.cg_mlp_create(ctx.h, 0, None, None, None, C.byref(h)) == _lib.CG_EINVAL
