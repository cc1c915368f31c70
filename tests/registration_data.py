"""Synthetic registration pairs shared by the registration tests and tools/bench_registration.py: ground-truth
transforms from the KITTI test list (tests/golden/kitti_reg_correct_gt.txt, rows seq,anc,pos,tx,ty,tz,qw,qx,qy,qz)."""
import os

import numpy as np

GT_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kitti_reg_correct_gt.txt")


def quat2rotm(q):
    """unit quaternion (w, x, y, z) -> rotation matrix (quat2rotm)"""
    w, x, y, z = np.asarray(q, np.float64) / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def kitti_gt_transforms():
    """(2831, 3, 4) float64: T_gt = [quat2rotm(q), t] per test pair (evaluate_kitti.m:88-90)"""
    rows = np.loadtxt(GT_PATH, delimiter=",")
    return np.stack([np.concatenate([quat2rotm(r[6:10]), r[3:6, None]], 1) for r in rows])


def synth_pairs(T, M, inlier_ratio, C=32, noise=0.05, desc_noise=0.05, seed=0):
    """Keypoint pairs related by T (B,3,4): pos keypoints y, anc keypoints x = R y + t (+ noise) for the first
    round(inlier_ratio * M) of them, unrelated points for the rest; descriptors shared (+ noise) by the related pairs,
    random otherwise.  Rows are shuffled on the pos side.  -> anc_xyz, pos_xyz (B,M,3), anc_desc, pos_desc (B,M,C) float32."""
    rng = np.random.default_rng(seed)
    B = len(T)
    ratios = np.broadcast_to(np.asarray(inlier_ratio, np.float64), (B,))
    pos = rng.uniform(-30, 30, (B, M, 3)) * np.array([1.0, 1.0, 0.1])
    anc = np.einsum("bij,bmj->bmi", T[:, :, :3], pos) + T[:, None, :, 3] + rng.normal(0, noise, (B, M, 3))
    pd = rng.normal(0, 1, (B, M, C))
    ad = pd + rng.normal(0, desc_noise, (B, M, C))
    for b in range(B):
        n_in = int(round(ratios[b] * M))
        anc[b, n_in:] = rng.uniform(-30, 30, (M - n_in, 3)) * np.array([1.0, 1.0, 0.1])
        ad[b, n_in:] = rng.normal(0, 1, (M - n_in, C))
        perm = rng.permutation(M)
        pos[b] = pos[b, perm]; pd[b] = pd[b, perm]
    f = lambda v: np.ascontiguousarray(v, np.float32)
    return f(anc), f(pos), f(ad), f(pd)
