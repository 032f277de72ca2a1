"""Golden vectors for the set-abstraction / feature-propagation stacks (tests/golden/pn2_modules.npz).

Run in the authoring container only (needs /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_modules.py

The reference ships no SA/FP module (SURVEY.md section 0, D1); oracle/pn2_modules_ref.py restates the upstream forward
passes.  Here that composition is EXECUTED WITH THE REFERENCE'S OWN PRIMITIVES (sample_and_group, square_distance,
index_points imported from /root/reference/pointnet2.py) so that everything the reference does define is the real
thing; the conv/BN/ReLU/max/interpolation glue is torch.  Weights come from catgrasp_b200.synthetic.make_mlp_state_dict.
"""
import os
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, "/root/reference")

import pointnet2 as ref  # noqa: E402  the reference itself

from catgrasp_b200.synthetic import make_mlp_state_dict  # noqa: E402
from oracle.pn2_modules_ref import feature_propagation, set_abstraction  # noqa: E402


def main():
    torch.set_num_threads(1)
    rng = np.random.RandomState(3)
    B, N = 2, 3000
    xyz = rng.uniform(-0.5, 0.5, (B, 3, N)).astype(np.float32)
    nrm = rng.normal(0, 1, (B, 3, N)).astype(np.float32)
    out = {"xyz": xyz, "nrm": nrm}
    # SA1(npoint 256, r 0.2, k 32, 3+3 -> [64,64,128]); the FPS start is whatever torch.randint draws (:66)
    sd1 = make_mlp_state_dict([6, 64, 64, 128], seed=11)
    torch.manual_seed(5)
    start1 = torch.randint(0, N, (B,), dtype=torch.long)
    torch.manual_seed(5)
    l1_xyz, l1_pts, grouped1 = set_abstraction(ref, sd1, 3, 256, 0.2, 32, False, torch.from_numpy(xyz), torch.from_numpy(nrm))
    # SA2 on top of it (npoint 64, r 0.4, k 16, 128+3 -> [128,128,256]): widths that are not tensor-core shapes at the input
    sd2 = make_mlp_state_dict([131, 128, 128, 256], seed=12)
    torch.manual_seed(6)
    start2 = torch.randint(0, 256, (B,), dtype=torch.long)
    torch.manual_seed(6)
    l2_xyz, l2_pts, _ = set_abstraction(ref, sd2, 3, 64, 0.4, 16, False, l1_xyz, l1_pts)
    # SA3: group_all (3+256 -> [256,512])
    sd3 = make_mlp_state_dict([259, 256, 512], seed=13)
    l3_xyz, l3_pts, _ = set_abstraction(ref, sd3, 2, None, None, None, True, l2_xyz, l2_pts)
    # FP3: S == 1 broadcast path (256 + 512 -> [256,256])
    sdf3 = make_mlp_state_dict([768, 256, 256], seed=14, conv2d=False)
    f2, _, _ = feature_propagation(ref, sdf3, 2, l2_xyz, l3_xyz, l2_pts, l3_pts)
    # FP2: 64 -> 256 points (128 + 256 -> [256,128])
    sdf2 = make_mlp_state_dict([384, 256, 128], seed=15, conv2d=False)
    f1, idx2, w2 = feature_propagation(ref, sdf2, 2, l1_xyz, l2_xyz, l1_pts, f2)
    # FP1: 256 -> 3000 points, skip = the normals (3 + 128 -> [128,128,64])
    sdf1 = make_mlp_state_dict([131, 128, 128, 64], seed=16, conv2d=False)
    f0, idx1, w1 = feature_propagation(ref, sdf1, 3, torch.from_numpy(xyz), l1_xyz, torch.from_numpy(nrm), f1)
    # f0 in full would put the file over 1 MB: keep a fixed, seeded sample of 512 of its N points
    f0_cols = np.sort(np.random.RandomState(0).choice(N, 512, replace=False))
    out.update(start1=start1.numpy(), start2=start2.numpy(), l1_xyz=l1_xyz.numpy(), l1_pts=l1_pts.numpy(),
               grouped1=grouped1.numpy()[:, :8], l2_xyz=l2_xyz.numpy(), l2_pts=l2_pts.numpy(), l3_pts=l3_pts.numpy(),
               f2=f2.numpy(), f1=f1.numpy(), idx2=idx2.numpy(), w2=w2.numpy(), f0_cols=f0_cols,
               f0_sample=np.ascontiguousarray(f0.numpy()[:, :, f0_cols]), idx1=idx1.numpy(), w1=w1.numpy())
    np.savez_compressed(os.path.join(HERE, "pn2_modules.npz"), **out)
    print({k: v.shape for k, v in out.items()}, os.path.getsize(os.path.join(HERE, "pn2_modules.npz")))


if __name__ == "__main__":
    main()
