"""CPU checks of the registration evaluation: the float64 oracle (oracle/registration.py) against closed-form cases, the
RANSAC loop's termination rules, and the host-side parts of usip_b200.evaluation.registration."""
import numpy as np
import pytest

from oracle import registration as orc
from tests.registration_data import kitti_gt_transforms, quat2rotm


def _rand_rigid(rng):
    q = rng.normal(size=4)
    return quat2rotm(q), rng.uniform(-10, 10, 3)


def test_fit_recovers_exact_transform_and_agrees_with_kabsch():
    rng = np.random.default_rng(0)
    for _ in range(20):
        R, t = _rand_rigid(rng)
        y = rng.uniform(-20, 20, (3, 50))
        x = R @ y + t[:, None]
        Rt = orc.estimate_rigid_transform(x, y)
        assert np.abs(Rt[:, :3] - R).max() <= 1e-9 and np.abs(Rt[:, 3] - t).max() <= 1e-9
        # noisy data: Horn / Taati quaternion fit == SVD (Kabsch) least-squares fit
        xn = x + rng.normal(0, 0.3, x.shape)
        Rt = orc.estimate_rigid_transform(xn, y)
        xc, yc = xn.mean(1, keepdims=True), y.mean(1, keepdims=True)
        U, _, Vt = np.linalg.svd((xn - xc) @ (y - yc).T)
        D = np.diag([1, 1, np.sign(np.linalg.det(U @ Vt))])
        Rk = U @ D @ Vt
        assert np.abs(Rt[:, :3] - Rk).max() <= 1e-9
        assert np.abs(Rt[:, 3] - (xc - Rk @ yc)[:, 0]).max() <= 1e-9


def _table(n, T, seed=0):
    rng = np.random.default_rng(seed)
    return np.stack([rng.choice(n, 3, replace=False) for _ in range(T)])


def test_ransac_all_inliers_stops_at_ten_trials():
    rng = np.random.default_rng(1)
    R, t = _rand_rigid(rng)
    y = rng.uniform(-20, 20, (3, 40)); x = R @ y + t[:, None]
    r = orc.ransac_rt(x, y, _table(40, 10002), 1.0, 10001)
    assert r["trialcount"] == 10 and len(r["inliers"]) == 40 and r["best_trial"] == 9   # '>=': the last tie wins
    assert np.abs(r["Rt"][:, :3] - R).max() <= 1e-9


def test_ransac_all_outliers_and_max_trials_cap():
    rng = np.random.default_rng(2)
    x = rng.uniform(-100, 100, (3, 30)); y = rng.uniform(-100, 100, (3, 30))
    r = orc.ransac_rt(x, y, _table(30, 102), 0.01, 101)
    assert r["trialcount"] == 102                           # capped at maxTrials + 1
    assert r["Rt"] is None and len(r["inliers"]) == 0       # fewer than 3 inliers: empty result
    assert r["best_trial"] == 101                           # every trial ties at 3 inliers or fewer... the last >= wins
    assert all(c <= 3 for c in r["counts"])


def test_ransac_ties_go_to_the_later_trial():
    # two disjoint exact triples define two different transforms with 3 inliers each; everything else is far away
    rng = np.random.default_rng(3)
    R1, t1 = _rand_rigid(rng); R2, t2 = _rand_rigid(rng)
    y = rng.uniform(-20, 20, (3, 6))
    x = np.concatenate([R1 @ y[:, :3] + t1[:, None], R2 @ y[:, 3:] + t2[:, None]], 1)
    table = np.array([[0, 1, 2], [3, 4, 5]] * 20)
    r = orc.ransac_rt(x, y, table, 1e-6, 3)
    assert r["counts"][:2] == [3, 3]
    assert r["trialcount"] == 4 and r["best_trial"] == 3    # trials 0..3 tie; the last one wins
    assert list(r["inliers"]) == [3, 4, 5]


@pytest.mark.parametrize("n", [0, 1, 2, 3])
def test_ransac_tiny_sets(n):
    rng = np.random.default_rng(4)
    R, t = _rand_rigid(rng)
    y = rng.uniform(-20, 20, (3, n)); x = R @ y + t[:, None]
    r = orc.ransac_rt(x, y, _table(max(n, 3), 5), 1.0, 4)
    assert r["trialcount"] == 0 and r["best_trial"] == -1
    if n < 3:
        assert r["Rt"] is None and len(r["inliers"]) == 0
    else:
        assert list(r["inliers"]) == [0, 1, 2] and np.abs(r["Rt"][:, :3] - R).max() <= 1e-9


def test_union_order_matches_np_unique():
    rng = np.random.default_rng(5)
    nn12 = rng.integers(0, 40, (50, 5)); nn21 = rng.integers(0, 50, (40, 5))
    c = orc.correspondences(nn12, nn21)
    rows = np.concatenate([np.stack([np.repeat(np.arange(50), 5), nn12.ravel()], 1),
                           np.stack([nn21.ravel(), np.repeat(np.arange(40), 5)], 1)])
    assert np.array_equal(c, np.unique(rows, axis=0))
    # k = 1, one direction: [i, nn(i)] in anc order
    nn = rng.integers(0, 40, (50, 1))
    assert np.array_equal(orc.correspondences(nn), np.stack([np.arange(50), nn[:, 0]], 1))


def test_compare_transform_conventions():
    from usip_b200.evaluation import registration as reg
    T = kitti_gt_transforms()
    assert T.shape == (2831, 3, 4)                      # 2,831 pairs (the list has one blank line)
    rng = np.random.default_rng(6)
    Tb = T[:64]
    # perturb: small rotation about z, y, x and a translation offset
    ang = rng.uniform(-0.05, 0.05, (64, 3))
    E = np.empty_like(Tb)
    for b in range(64):
        cz, sz = np.cos(ang[b, 0]), np.sin(ang[b, 0]); cy, sy = np.cos(ang[b, 1]), np.sin(ang[b, 1])
        cx, sx = np.cos(ang[b, 2]), np.sin(ang[b, 2])
        Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]); Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        E[b, :, :3] = Tb[b, :, :3] @ (Rz @ Ry @ Rx)          # R_gt^T R = Rz Ry Rx: ZYX Euler angles = ang
        E[b, :, 3] = Tb[b, :, 3] + np.array([0.3, -0.4, 0.0])
    dt, deg = reg.compare_transform(Tb, E)
    assert np.allclose(dt, 0.5, atol=1e-12)
    assert np.allclose(deg, np.abs(ang).sum(1) * 180 / np.pi, atol=1e-9)
    for b in range(8):
        assert np.allclose(orc.compare_transform(Tb[b], E[b]), (dt[b], deg[b]), atol=1e-9)
    # an empty result scores 3 m / 6 degrees (the catch in evaluate_*.m)
    E[3] = np.nan
    dt, deg = reg.compare_transform(Tb, E)
    assert dt[3] == 3.0 and deg[3] == 6.0 and orc.compare_transform(Tb[3], None) == (3.0, 6.0)


def test_summary_uses_successful_pairs_and_sample_std():
    from usip_b200.evaluation import registration as reg
    import torch
    B = 6
    T = kitti_gt_transforms()[:B]
    E = T.copy()
    E[:, 0, 3] += np.array([0.1, 0.2, 0.4, 2.5, 0.0, 0.3])   # pair 3 fails on translation
    E[5] = np.nan                                           # pair 5 empty -> fails
    r = reg.RansacResult(torch.from_numpy(E), torch.tensor([10, 20, 30, 40, 50, 0]), torch.tensor([11, 12, 13, 14, 15, 16]),
                         None, None, torch.zeros(B, dtype=torch.int32), None)
    s = reg.summarize_registration(T, r, torch.tensor([100] * B))
    ok = np.array([0, 1, 2, 4])
    assert s["wrong_counter"] == 2 and list(np.nonzero(s["success"])[0]) == list(ok)
    dts = np.array([0.1, 0.2, 0.4, 0.0])
    assert np.isclose(s["rte_mean"], dts.mean()) and np.isclose(s["rte_std"], np.std(dts, ddof=1))
    assert np.isclose(s["inlier_ratio"], np.mean([0.1, 0.2, 0.3, 0.5])) and np.isclose(s["trial_count"], 12.75)
    ref = orc.summarize(s["delta_t"], s["delta_deg"], s["n_inliers"] / 100.0, s["trialcount"])
    for k in ("wrong_counter", "inlier_ratio", "trial_count", "rte_mean", "rte_std", "rre_mean", "rre_std"):
        assert np.isclose(s[k], ref[k]), k


def test_descriptor_bin_round_trip(tmp_path):
    from usip_b200.evaluation import registration as reg
    rng = np.random.default_rng(7)
    xyz = rng.normal(size=(37, 3)).astype(np.float32); desc = rng.normal(size=(37, 128)).astype(np.float32)
    p = str(tmp_path / "000000.bin")
    reg.write_descriptors_bin(p, xyz, desc)
    raw = np.fromfile(p, dtype=np.float32).reshape(37, 131)     # Utils.load_descriptors: rows of 3 + C floats
    assert np.array_equal(raw[:, :3], xyz) and np.array_equal(raw[:, 3:], desc)
    x2, d2 = reg.read_descriptors_bin(p, feature_dim=128)
    assert np.array_equal(x2, xyz) and np.array_equal(d2, desc)
    with pytest.raises(ValueError):
        reg.read_descriptors_bin(p, feature_dim=127)


def test_repeatability_oracle_counts():
    rng = np.random.default_rng(8)
    R, t = _rand_rigid(rng)
    pos = rng.uniform(-10, 10, (30, 3))
    anc = pos @ R.T + t
    anc[:10] += 5.0                                             # 10 of 30 moved away
    rep, d = orc.repeatability(anc, pos, np.concatenate([R, t[:, None]], 1), 0.5)
    assert np.isclose(rep, 20 / 30) and np.allclose(d[10:], 0, atol=1e-9)
