"""Registration and repeatability evaluation -- the numbers the USIP paper reports for a trained detector + descriptor,
computed on the GPU instead of in MATLAB.  Restates the original project's evaluation/matlab/:

  eval_outdoor/kitti/evaluate_kitti.m    1-NN anc -> pos matching, RANSAC, RTE / RRE, failure count
  eval_outdoor/oxford/evaluate_oxford.m  5-NN in both directions, union of the matches, then the same
  eval_outdoor/external/*.m              ransacfitRt / ransac / estimateRigidTransform (the RANSAC rigid fit)
  eval_repeatability/eval_rep.m          keypoint repeatability

Matching, the correspondence list and RANSAC run in libusip_b200 (csrc/registration.cu); repeatability uses the
transform and nearest-point kernels of the losses.  compare_transform and the summary are float64 host bookkeeping.

Frames: all points and T_gt are in one frame per pair, and T_gt maps pos-frame points into the anc frame (the same
direction as the estimated Rt).  Dataset-specific conversions (KITTI cam2velodyne, Oxford's axis swap) stay with the
caller.  Points, descriptors and keypoints are rows: padded (B, M, D) tensors with per-pair counts, or lists of (M_b, D)
arrays (what select_keypoints and read_descriptors_bin return).

Known deviation: MATLAB draws RANSAC samples with rng(0); randsample per pair, a stream that cannot be reproduced here.
Trials draw from a counter-based Philox generator keyed by (seed, pair, trial) instead, so per-pair results are
statistically comparable with MATLAB runs, not identical to them."""
import collections

import numpy as np
import torch

from .. import ops

RansacResult = collections.namedtuple(
    "RansacResult", ["Rt", "n_inliers", "trialcount", "best_trial", "inlier_mask", "status", "samples"])

STATUS_OK, STATUS_TOO_FEW_CORRESPONDENCES, STATUS_TOO_FEW_INLIERS = 0, 1, 2


# ----------------------------------------------------------------------------- descriptor files
def write_descriptors_bin(path, xyz, desc):
    """Rows of 3 + C float32 (xyz then descriptor), the layout Utils.load_descriptors reads (Utils.m:56-73)."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    desc = np.asarray(desc, np.float32).reshape(len(xyz), -1)
    np.ascontiguousarray(np.concatenate([xyz, desc], 1), np.float32).tofile(path)


def read_descriptors_bin(path, feature_dim=128):
    """-> (xyz (M,3), desc (M,feature_dim)) float32 from a file written by write_descriptors_bin."""
    a = np.fromfile(path, dtype=np.float32)
    m = 3 + int(feature_dim)
    if a.size % m:
        raise ValueError("%s: %d floats is not a whole number of rows of 3 + %d" % (path, a.size, feature_dim))
    a = a.reshape(-1, m)
    return a[:, :3].copy(), a[:, 3:].copy()


# ----------------------------------------------------------------------------- batching
def _device(device):
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def _rows(x, counts, dtype, device, fill=0.0):
    """A list of (M_b, D) arrays or a padded (B, M, D) tensor -> (padded (B, M, D) contiguous on device, counts (B) i32)."""
    if isinstance(x, (list, tuple)):
        ts = [torch.as_tensor(np.asarray(t) if not torch.is_tensor(t) else t) for t in x]
        D = ts[0].shape[1]
        M = max([t.shape[0] for t in ts] + [1])
        out = torch.full((len(ts), M, D), fill, dtype=dtype, device=device)
        for b, t in enumerate(ts):
            out[b, :t.shape[0]] = t.to(device=device, dtype=dtype)
        cnt = torch.tensor([t.shape[0] for t in ts], dtype=torch.int32, device=device)
        return out, cnt
    out = torch.as_tensor(x).to(device=device, dtype=dtype).contiguous()
    if counts is None:
        cnt = torch.full((out.shape[0],), out.shape[1], dtype=torch.int32, device=device)
    else:
        cnt = torch.as_tensor(counts).to(device=device, dtype=torch.int32).contiguous()
        if fill != 0.0:
            pad = torch.arange(out.shape[1], device=device)[None, :] >= cnt[:, None].long()
            out = out.masked_fill(pad[:, :, None], fill)
    return out, cnt


def _T34(T_gt):
    T = np.asarray(T_gt.detach().cpu().numpy() if torch.is_tensor(T_gt) else T_gt, np.float64)
    T = T.reshape(-1, T.shape[-2], 4)
    return T[:, :3, :]


# ----------------------------------------------------------------------------- the three stages
def match_descriptors(anc_desc, pos_desc, k=1, both_directions=False, anc_count=None, pos_count=None, device=None):
    """Correspondences from descriptor matching.  k = 1, one direction: [i, nn(i)] for every anc keypoint i in order
    (evaluate_kitti.m:53-54).  both_directions: the unique (anc, pos) rows of the k-NN matches anc -> pos and pos -> anc
    in ascending order (union(..., 'rows'), evaluate_oxford.m:63-72).  k in [1, 8]; at most 1024 keypoints per frame.
    -> (corr (B, nmax, 2) int32 cuda, rows past counts[b] are -1; counts (B) int32 cuda)."""
    dev = _device(device)
    a, na = _rows(anc_desc, anc_count, torch.float32, dev)
    b, nb = _rows(pos_desc, pos_count, torch.float32, dev)
    a = a.transpose(1, 2).contiguous()           # (B, C, M): the kernels' channel-major layout
    b = b.transpose(1, 2).contiguous()
    nn12 = ops.desc_knn(a, b, k, na, nb)
    nn21 = ops.desc_knn(b, a, k, nb, na) if both_directions else None
    return ops.corr_build(nn12, b.shape[2], nn21, na, nb)


def ransac_fit_rt(anc_xyz, pos_xyz, corr, counts, threshold=1.0, max_trials=10001, p=0.99, seed=0, samples=None,
                  anc_count=None, pos_count=None, return_samples=False, device=None):
    """RANSAC for the rigid transform x = R y + t over correspondences (x = anc_xyz[corr[:, 0]], y = pos_xyz[corr[:, 1]]),
    ransacfitRt.m with s = 3, inlier iff ||x - (R y + t)|| < threshold, adaptive trial count for probability p, at most
    max_trials + 1 trials, then a least-squares refit on the best hypothesis's inliers.
    samples: optional (B, max_trials + 1, 3) int32 table of 0-based correspondence indices used instead of the generator.
    -> RansacResult of cuda tensors: Rt (B,3,4) float64 (NaN when empty), n_inliers, trialcount, best_trial (-1 when no
    loop ran), inlier_mask (B, nmax) uint8, status (STATUS_*), samples (the table used, with return_samples; -1 for
    trials never scored)."""
    dev = _device(device)
    ax, _ = _rows(anc_xyz, anc_count, torch.float64, dev)
    px, _ = _rows(pos_xyz, pos_count, torch.float64, dev)
    corr = torch.as_tensor(corr).to(device=dev, dtype=torch.int32).contiguous()
    counts = torch.as_tensor(counts).to(device=dev, dtype=torch.int32).contiguous()
    if samples is not None:
        samples = torch.as_tensor(samples).to(device=dev, dtype=torch.int32).contiguous()
    r = ops.ransac_rt(ax, px, corr, counts, threshold, max_trials, p, seed, samples=samples, want_samples=return_samples)
    return RansacResult(r["Rt"], r["n_inliers"], r["trialcount"], r["best_trial"], r["inlier_mask"], r["status"],
                        r.get("samples"))


def rotm2eul_zyx(R):
    """rotm2eul(R) in its default ZYX order for a batch (B,3,3): [atan2(r21, r11), atan2(-r31, hypot(r11, r21)),
    atan2(r32, r33)].  At the gimbal singularity (hypot(r11, r21) < 10 eps) the first angle is 0 and the third is
    atan2(-r23, r22); such a relative rotation is ~90 degrees off and fails the 5 degree test either way."""
    R = np.asarray(R, np.float64)
    sy = np.hypot(R[:, 0, 0], R[:, 1, 0])
    sing = sy < 10 * np.finfo(np.float64).eps
    z = np.where(sing, 0.0, np.arctan2(R[:, 1, 0], R[:, 0, 0]))
    y = np.arctan2(-R[:, 2, 0], sy)
    x = np.where(sing, np.arctan2(-R[:, 1, 2], R[:, 1, 1]), np.arctan2(R[:, 2, 1], R[:, 2, 2]))
    return np.stack([z, y, x], 1)


def compare_transform(T_gt, Rt):
    """Utils.compareTransform (Utils.m:320-325) per pair: delta_t = ||t_gt - t||, delta_deg = sum |rotm2eul(R_gt^T R)| in
    degrees.  T_gt (B,3,4) or (B,4,4), Rt (B,3,4); an empty Rt (any NaN) scores 3 m / 6 degrees, the catch of
    evaluate_kitti.m:92-97.  -> (delta_t (B), delta_deg (B)) float64 numpy."""
    T = _T34(T_gt)
    E = _T34(Rt)
    empty = ~np.isfinite(E).all(axis=(1, 2))
    E = np.where(empty[:, None, None], 0.0, E)
    dt = np.linalg.norm(T[:, :, 3] - E[:, :, 3], axis=1)
    dR = np.einsum("bji,bjk->bik", T[:, :, :3], E[:, :, :3])
    deg = np.abs(rotm2eul_zyx(dR)).sum(1) * 180.0 / np.pi
    return np.where(empty, 3.0, dt), np.where(empty, 6.0, deg)


def _std1(v):
    return float(np.std(v, ddof=1)) if len(v) > 1 else (0.0 if len(v) == 1 else float("nan"))


def _mean(v):
    return float(np.mean(v)) if len(v) else float("nan")


def evaluate_registration(anc_xyz, anc_desc, pos_xyz, pos_desc, T_gt, protocol="kitti", threshold=1.0, max_trials=10001,
                          p=0.99, seed=0, anc_count=None, pos_count=None, device=None):
    """evaluate_kitti.m / evaluate_oxford.m for a batch of pairs.  protocol "kitti": 1-NN anc -> pos; "oxford": 5-NN in
    both directions, union.  A pair fails if delta_t > 2 m or delta_deg > 5 degrees; inlier ratio, trial count and
    RTE / RRE mean and std (N-1) are over the successful pairs only (evaluate_kitti.m:104-131).
    -> dict: wrong_counter, inlier_ratio, trial_count, rte_mean, rte_std, rre_mean, rre_std, and per pair: delta_t,
    delta_deg, success, n_inliers, n_corr, trialcount, status, Rt (numpy)."""
    if protocol == "kitti":
        k, both = 1, False
    elif protocol == "oxford":
        k, both = 5, True
    else:
        raise ValueError("protocol must be 'kitti' or 'oxford', got %r" % (protocol,))
    corr, counts = match_descriptors(anc_desc, pos_desc, k=k, both_directions=both, anc_count=anc_count,
                                     pos_count=pos_count, device=device)
    r = ransac_fit_rt(anc_xyz, pos_xyz, corr, counts, threshold=threshold, max_trials=max_trials, p=p, seed=seed,
                      anc_count=anc_count, pos_count=pos_count, device=device)
    return summarize_registration(T_gt, r, counts)


def summarize_registration(T_gt, r, counts):
    """The tail of evaluate_*.m over a RansacResult and the correspondence counts (see evaluate_registration)."""
    Rt = r.Rt.cpu().numpy()
    n_inl = r.n_inliers.cpu().numpy().astype(np.int64)
    n_corr = torch.as_tensor(counts).cpu().numpy().astype(np.int64)
    tc = r.trialcount.cpu().numpy().astype(np.int64)
    dt, deg = compare_transform(T_gt, Rt)
    ok = ~((dt > 2) | (deg > 5))
    ratio = n_inl / np.maximum(n_corr, 1)
    return dict(wrong_counter=int((~ok).sum()), inlier_ratio=_mean(ratio[ok]), trial_count=_mean(tc[ok]),
                rte_mean=_mean(dt[ok]), rte_std=_std1(dt[ok]), rre_mean=_mean(deg[ok]), rre_std=_std1(deg[ok]),
                delta_t=dt, delta_deg=deg, success=ok, n_inliers=n_inl, n_corr=n_corr, trialcount=tc,
                status=r.status.cpu().numpy(), Rt=Rt)


def repeatability(anc_kp, pos_kp, T_gt, radius=0.5, anc_count=None, pos_count=None, device=None):
    """eval_rep.m:143-146: per pair, the fraction of anc keypoints whose nearest pos keypoint, after applying T_gt to
    the pos keypoints, is closer than radius.  Computed in float32 (MATLAB: float64), so a keypoint can only be counted
    differently when its distance is within rounding of the radius.
    -> dict: per_pair (B), mean, min, max (as eval_rep.m prints them), keypoint_mean (mean anc keypoint count)."""
    dev = _device(device)
    a, na = _rows(anc_kp, anc_count, torch.float32, dev)
    b, _ = _rows(pos_kp, pos_count, torch.float32, dev, fill=float("nan"))   # NaN rows are never the nearest
    T = torch.from_numpy(_T34(T_gt)).to(device=dev, dtype=torch.float32)
    B = a.shape[0]
    R = T[:, :, :3].contiguous()
    shift = T[:, :, 3].contiguous()
    scale = torch.ones((B,), dtype=torch.float32, device=dev)
    pt = ops.transform_points(b.transpose(1, 2).contiguous(), R, scale, shift)
    d, _ = ops.pairwise_min(a.transpose(1, 2).contiguous(), pt, method="brute")
    valid = torch.arange(a.shape[1], device=dev)[None, :] < na[:, None].long()
    hits = ((d < radius) & valid).sum(1).double()
    per = (hits / na.double()).cpu().numpy()
    return dict(per_pair=per, mean=float(per.mean()), min=float(per.min()), max=float(per.max()),
                keypoint_mean=float(na.double().mean().item()))
