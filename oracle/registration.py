"""float64 numpy restatement of the original project's MATLAB registration evaluation (test infrastructure only; the
package never imports it).  Paths are relative to the original project's evaluation/matlab/:

  eval_outdoor/kitti/evaluate_kitti.m, eval_outdoor/oxford/evaluate_oxford.m   matching, scoring, summary
  eval_outdoor/external/ransacfitRt.m, ransac.m                               RANSAC loop and final refit
  eval_outdoor/external/estimateRigidTransform.m, quat2rot.m, crossTimesMatrix.m   the rigid fit
  eval_outdoor/Utils.m                                                        compareTransform, apply_transform
  eval_repeatability/eval_rep.m                                               repeatability

RANSAC runs over an explicit sample table (T, 3) of 0-based indices instead of MATLAB's rng(0) / randsample stream."""
import numpy as np

EPS = 2.0 ** -52          # MATLAB eps


def knn(a, b, k):
    """pdist2(b, a, 'euclidean', 'smallest', k) (evaluate_kitti.m:53): a (C,Ma), b (C,Mb) -> idx (Ma,k), d2 (Ma,Mb).
    Ascending distance, ties to the smaller index (stable sort)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    d2 = ((a[:, :, None] - b[:, None, :]) ** 2).sum(0)
    return np.argsort(d2, axis=1, kind="stable")[:, :k], d2


def correspondences(nn12, nn21=None):
    """evaluate_kitti.m:53-54: [i, nn12(i)] in anc order (k = 1, one direction); evaluate_oxford.m:63-72: the unique rows
    of union(matches12, matches21, 'rows') in ascending (anc, pos) order.  nn12 (Ma,k), nn21 (Mb,k) -> (n, 2)."""
    nn12 = np.asarray(nn12)
    rows = [np.stack([np.repeat(np.arange(nn12.shape[0]), nn12.shape[1]), nn12.reshape(-1)], 1)]
    if nn21 is not None:
        nn21 = np.asarray(nn21)
        rows.append(np.stack([nn21.reshape(-1), np.repeat(np.arange(nn21.shape[0]), nn21.shape[1])], 1))
    return np.unique(np.concatenate(rows).astype(np.int64), axis=0).reshape(-1, 2)


def cross_times(v):
    """crossTimesMatrix.m:18-26 for one vector"""
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def quat2rot(q):
    """quat2rot.m:10-25, w first"""
    q0, q1, q2, q3 = q
    return np.array([[q0 * q0 + q1 * q1 - q2 * q2 - q3 * q3, 2 * (q1 * q2 - q0 * q3), 2 * (q1 * q3 + q0 * q2)],
                     [2 * (q1 * q2 + q0 * q3), q0 * q0 - q1 * q1 + q2 * q2 - q3 * q3, 2 * (q2 * q3 - q0 * q1)],
                     [2 * (q1 * q3 - q0 * q2), 2 * (q2 * q3 + q0 * q1), q0 * q0 - q1 * q1 - q2 * q2 + q3 * q3]])


def estimate_rigid_transform(x, y):
    """estimateRigidTransform.m:43-71 / estimateRt.m: x, y (3,n), n >= 3 -> Rt (3,4) with x = R y + t (Taati's quaternion
    form: B = sum A_i^T A_i, quaternion = last right-singular vector of B)."""
    x = np.asarray(x, np.float64); y = np.asarray(y, np.float64)
    n = x.shape[1]
    xc = x.sum(1) / n; yc = y.sum(1) / n
    xs = x - xc[:, None]; ys = y - yc[:, None]
    B = np.zeros((4, 4))
    for i in range(n):
        A = np.zeros((4, 4))
        A[0, 1:] = ys[:, i] - xs[:, i]
        A[1:, 0] = xs[:, i] - ys[:, i]
        A[1:, 1:] = cross_times(ys[:, i] + xs[:, i])
        B += A.T @ A
    _, _, vh = np.linalg.svd(B)
    R = quat2rot(vh[3])
    return np.concatenate([R, (xc - R @ yc)[:, None]], 1)


def residuals(Rt, x, y):
    """ransacfitRt.m:73-74, in the op order the GPU kernel uses: p_r = ((R_r0 y0 + R_r1 y1) + R_r2 y2) + t_r,
    d = sqrt((dx^2 + dy^2) + dz^2)"""
    e = [x[r] - (((Rt[r, 0] * y[0] + Rt[r, 1] * y[1]) + Rt[r, 2] * y[2]) + Rt[r, 3]) for r in range(3)]
    return np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2])


def ransac_rt(x, y, samples, threshold=1.0, max_trials=10001, p=0.99):
    """ransacfitRt.m:20-51 + ransac.m:113-232 (s = 3, isdegenerate = 0) over the explicit sample table samples (>= max_trials+1,
    3).  x, y (3,n).  Returns dict Rt (3,4) or None, inliers (0-based indices of the best hypothesis), trialcount,
    best_trial (-1 without a loop), counts (inliers per trial scored), margin (min |d - threshold| over every residual
    of every scored trial)."""
    x = np.asarray(x, np.float64); y = np.asarray(y, np.float64)
    n = x.shape[1]
    res = dict(Rt=None, inliers=np.zeros(0, np.int64), trialcount=0, best_trial=-1, counts=[], margin=np.inf)
    if n < 3:                                                     # ransacfitRt.m:25-29
        return res
    if n == 3:                                                    # ransacfitRt.m:30-34
        res.update(Rt=estimate_rigid_transform(x, y), inliers=np.arange(3))
        return res
    N, trialcount, bestscore = 1.0, 0, 0                          # ransac.m:131-133
    best_inl, best_trial = None, -1
    lp = np.log(1.0 - p)
    while N > trialcount:                                         # ransac.m:140
        ind = np.asarray(samples[trialcount])
        M = estimate_rigid_transform(x[:, ind], y[:, ind])
        d = residuals(M, x, y)
        res["margin"] = min(res["margin"], float(np.abs(d - threshold).min()))
        inl = np.nonzero(d < threshold)[0]
        res["counts"].append(len(inl))
        if len(inl) >= bestscore:                                 # ransac.m:195, ties to the later trial
            bestscore, best_inl, best_trial = len(inl), inl, trialcount
            f = len(inl) / n
            pno = min(1.0 - EPS, max(EPS, 1.0 - f * f * f))       # ransac.m:202-205 (f^3 as f*f*f, as the kernel)
            N = max(lp / np.log(pno), 10.0)                       # ransac.m:206-207
        trialcount += 1
        if trialcount > max_trials:                               # ransac.m:216-218
            break
    res.update(trialcount=trialcount, best_trial=best_trial)
    if len(best_inl) >= 3:                                        # ransacfitRt.m:45-50
        res.update(Rt=estimate_rigid_transform(x[:, best_inl], y[:, best_inl]), inliers=best_inl)
    return res


def rotm2eul_zyx(R):
    """rotm2eul(R) in its default ZYX order: [atan2(r21, r11), asin(-r31), atan2(r32, r33)] (r31 clamped to [-1, 1])"""
    return np.array([np.arctan2(R[1, 0], R[0, 0]), np.arcsin(np.clip(-R[2, 0], -1.0, 1.0)), np.arctan2(R[2, 1], R[2, 2])])


def compare_transform(T_gt, Rt):
    """Utils.m:320-325 with the catch of evaluate_kitti.m:92-97 (empty Rt -> 3 m / 6 degrees)"""
    if Rt is None:
        return 3.0, 6.0
    T_gt = np.asarray(T_gt, np.float64); Rt = np.asarray(Rt, np.float64)
    dt = float(np.linalg.norm(T_gt[:3, 3] - Rt[:3, 3]))
    return dt, float(np.abs(rotm2eul_zyx(T_gt[:3, :3].T @ Rt[:3, :3])).sum() * 180.0 / np.pi)


def summarize(delta_t, delta_deg, inlier_ratio, trialcount):
    """evaluate_kitti.m:104-131: failure if delta_t > 2 or delta_deg > 5; means / std (N-1) over successful pairs"""
    delta_t = np.asarray(delta_t, np.float64); delta_deg = np.asarray(delta_deg, np.float64)
    ok = ~((delta_t > 2) | (delta_deg > 5))
    std = lambda v: float(np.std(v, ddof=1)) if len(v) > 1 else (0.0 if len(v) == 1 else float("nan"))
    mean = lambda v: float(np.mean(v)) if len(v) else float("nan")
    return dict(wrong_counter=int((~ok).sum()), inlier_ratio=mean(np.asarray(inlier_ratio)[ok]),
                trial_count=mean(np.asarray(trialcount)[ok]), rte_mean=mean(delta_t[ok]), rte_std=std(delta_t[ok]),
                rre_mean=mean(delta_deg[ok]), rre_std=std(delta_deg[ok]), success=ok)


def repeatability(anc_kp, pos_kp, T_gt, radius=0.5):
    """eval_rep.m:143-146: fraction of anc keypoints whose nearest pos keypoint (after apply_transform(pos, T_gt),
    Utils.m:127-134) is closer than radius.  anc_kp (Ma,3), pos_kp (Mb,3) -> (repeatability, nearest distances)."""
    anc = np.asarray(anc_kp, np.float64); pos = np.asarray(pos_kp, np.float64); T = np.asarray(T_gt, np.float64)
    pt = pos @ T[:3, :3].T + T[:3, 3]
    d = np.sqrt(((anc[:, None, :] - pt[None, :, :]) ** 2).sum(-1)).min(1)
    return float((d < radius).sum() / len(anc)), d
