"""GPU tests of the registration evaluation (csrc/registration.cu, usip_b200/evaluation/registration.py) against the float64
oracle restatement of the original MATLAB (oracle/registration.py)."""
import numpy as np
import pytest
import torch

from oracle import registration as orc
from tests.registration_data import kitti_gt_transforms, synth_pairs

pytestmark = pytest.mark.gpu


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ragged_desc(rng, B, C, Ma, Mb, na, nb):
    a = rng.normal(size=(B, C, Ma)).astype(np.float32)
    b = rng.normal(size=(B, C, Mb)).astype(np.float32)
    b[:, :, 7] = b[:, :, 3]                                     # exact ties: duplicate database columns
    b[:, :, 20] = b[:, :, 3]
    a[:, :, 5] = b[:, :, 3]                                     # a query sitting exactly on the duplicated column
    return a, b


@pytest.mark.parametrize("k", [1, 5])
def test_desc_knn_vs_oracle(k):
    from usip_b200 import ops
    rng = np.random.default_rng(k)
    B, C, Ma, Mb = 3, 40, 100, 90
    na, nb = np.array([100, 57, 80]), np.array([90, 33, 64])
    a, b = _ragged_desc(rng, B, C, Ma, Mb, na, nb)
    idx, dist = ops.desc_knn(cu(a), cu(b), k, cu(na.astype(np.int32)), cu(nb.astype(np.int32)), want_dist=True)
    idx = idx.cpu().numpy(); dist = dist.cpu().numpy()
    for bb in range(B):
        oi, d2 = orc.knn(a[bb][:, :na[bb]], b[bb][:, :nb[bb]], k)
        g = idx[bb, :na[bb]]
        assert (idx[bb, na[bb]:] == -1).all()
        for i in range(na[bb]):
            diff = np.nonzero(g[i] != oi[i])[0]
            for r in diff:                                      # allowed only between near-equal distances
                assert g[i, r] >= 0
                assert abs(d2[i, g[i, r]] - d2[i, oi[i, r]]) <= 1e-6 * max(d2[i, oi[i, r]], 1e-30), (bb, i, r)
            assert len(set(g[i])) == k
        assert list(g[5, :min(k, 3)]) == [3, 7, 20][:min(k, 3)]   # exact ties: smaller index first
        assert np.allclose(dist[bb, :na[bb]] ** 2, np.take_along_axis(d2, g.astype(np.int64), 1), rtol=1e-5, atol=1e-5)
    # the k = 1 column is bit-identical to the loss's nearest-descriptor search
    idx1, dist1 = ops.desc_knn(cu(a), cu(b), 1, want_dist=True)
    dp, ap = ops.desc_pairmin(cu(a), cu(b))
    assert torch.equal(idx1[:, :, 0], ap) and torch.equal(dist1[:, :, 0], dp)


@pytest.mark.parametrize("both", [False, True])
def test_corr_build_vs_oracle(both):
    from usip_b200 import ops
    rng = np.random.default_rng(10 + both)
    B, Ma, Mb = 4, 300, 260
    k = 5 if both else 1
    na, nb = np.array([300, 1, 150, 299]), np.array([260, 200, 1, 77])
    nn12 = np.stack([rng.integers(0, nb[b], (Ma, k)) for b in range(B)]).astype(np.int32)
    nn21 = np.stack([rng.integers(0, na[b], (Mb, k)) for b in range(B)]).astype(np.int32)
    corr, cnt = ops.corr_build(cu(nn12), Mb, cu(nn21) if both else None, cu(na.astype(np.int32)), cu(nb.astype(np.int32)))
    corr = corr.cpu().numpy(); cnt = cnt.cpu().numpy()
    for b in range(B):
        ref = orc.correspondences(nn12[b, :na[b]], nn21[b, :nb[b]] if both else None)
        assert cnt[b] == len(ref) and np.array_equal(corr[b, :cnt[b]], ref), b
        assert (corr[b, cnt[b]:] == -1).all()
    with pytest.raises(RuntimeError, match="1024"):
        ops.corr_build(torch.zeros((1, 1025, 1), dtype=torch.int32, device="cuda"), 4)


def _draw_table(rng, B, T, n):
    """(B,T,3) distinct indices per row in [0, n_b)"""
    n = np.asarray(n).reshape(B, 1)
    i0 = (rng.random((B, T)) * n).astype(np.int64)
    i1 = (rng.random((B, T)) * (n - 1)).astype(np.int64); i1 += i1 >= i0
    i2 = (rng.random((B, T)) * (n - 2)).astype(np.int64)
    lo, hi = np.minimum(i0, i1), np.maximum(i0, i1)
    i2 += i2 >= lo; i2 += i2 >= hi
    return np.stack([i0, i1, i2], -1).astype(np.int32)


def _pairs(B, M, ratios, seed, C=32):
    T = kitti_gt_transforms()[seed * 37: seed * 37 + B]
    anc, pos, ad, pd = synth_pairs(T, M, ratios, C=C, seed=seed)
    return T, anc, pos, ad, pd


def _oracle_pair(r_gpu_corr, n, anc, pos, table, thr, max_trials):
    c = r_gpu_corr[:n].astype(np.int64)
    return orc.ransac_rt(anc[c[:, 0]].T.astype(np.float64), pos[c[:, 1]].T.astype(np.float64), table, thr, max_trials)


def _check_same(r, b, o, nmax):
    assert int(r.trialcount[b]) == o["trialcount"], b
    assert int(r.best_trial[b]) == o["best_trial"], b
    mask = np.zeros(nmax, np.uint8); mask[o["inliers"]] = 1
    assert int(r.n_inliers[b]) == len(o["inliers"]), b
    assert np.array_equal(r.inlier_mask[b].cpu().numpy(), mask), b
    if o["Rt"] is None:
        assert int(r.status[b]) in (1, 2) and torch.isnan(r.Rt[b]).all()
    else:
        assert int(r.status[b]) == 0
        assert np.abs(r.Rt[b].cpu().numpy() - o["Rt"]).max() <= 1e-9, b


def test_ransac_explicit_table_vs_oracle():
    from usip_b200.evaluation import registration as reg
    B, M, max_trials = 6, 128, 1500
    T, anc, pos, ad, pd = _pairs(B, M, np.linspace(0.1, 0.5, B), seed=1)
    corr, cnt = reg.match_descriptors(ad, pd)
    corr_h, cnt_h = corr.cpu().numpy(), cnt.cpu().numpy()
    table = _draw_table(np.random.default_rng(3), B, max_trials + 1, cnt_h)
    r = reg.ransac_fit_rt(anc, pos, corr, cnt, max_trials=max_trials, samples=table)
    for b in range(B):
        o = _oracle_pair(corr_h[b], cnt_h[b], anc[b], pos[b], table[b], 1.0, max_trials)
        assert o["margin"] >= 1e-9, (b, o["margin"])          # no residual within rounding of the threshold
        _check_same(r, b, o, corr.shape[1])


def test_ransac_device_sampling_vs_oracle_and_seed():
    from usip_b200.evaluation import registration as reg
    B, M, max_trials = 6, 128, 3000
    T, anc, pos, ad, pd = _pairs(B, M, np.linspace(0.15, 0.5, B), seed=2)
    corr, cnt = reg.match_descriptors(ad, pd)
    corr_h, cnt_h = corr.cpu().numpy(), cnt.cpu().numpy()
    r = reg.ransac_fit_rt(anc, pos, corr, cnt, max_trials=max_trials, seed=7, return_samples=True)
    table = r.samples.cpu().numpy()
    for b in range(B):
        used = table[b, :int(r.trialcount[b])]
        assert (used >= 0).all() and (used < cnt_h[b]).all()
        assert (used[:, 0] != used[:, 1]).all() and (used[:, 0] != used[:, 2]).all() and (used[:, 1] != used[:, 2]).all()
        o = _oracle_pair(corr_h[b], cnt_h[b], anc[b], pos[b], table[b], 1.0, max_trials)
        assert o["margin"] >= 1e-9, (b, o["margin"])
        _check_same(r, b, o, corr.shape[1])
    r2 = reg.ransac_fit_rt(anc, pos, corr, cnt, max_trials=max_trials, seed=7, return_samples=True)
    for f in r._fields:
        assert torch.equal(getattr(r, f), getattr(r2, f)), f
    r3 = reg.ransac_fit_rt(anc, pos, corr, cnt, max_trials=max_trials, seed=8, return_samples=True)
    assert not torch.equal(r3.samples[:, :10], r.samples[:, :10])


def test_ransac_sampling_is_uniform():
    from scipy.stats import chi2
    from usip_b200.evaluation import registration as reg
    rng = np.random.default_rng(4)
    B, n, max_trials = 4, 50, 20000
    x = rng.uniform(-100, 100, (B, n, 3)); y = rng.uniform(-100, 100, (B, n, 3))   # all outliers: every trial runs
    corr = np.broadcast_to(np.stack([np.arange(n), np.arange(n)], 1), (B, n, 2)).astype(np.int32)
    r = reg.ransac_fit_rt(x, y, corr, np.full(B, n, np.int32), threshold=1e-3, max_trials=max_trials, return_samples=True)
    assert (r.trialcount.cpu().numpy() == max_trials + 1).all() and (r.status.cpu().numpy() == 2).all()
    s = r.samples.cpu().numpy()
    assert (s >= 0).all() and (s < n).all()
    for col in range(3):                                        # each draw position, pooled over the pairs
        obs = np.bincount(s[:, :, col].ravel(), minlength=n)
        stat = ((obs - obs.mean()) ** 2 / obs.mean()).sum()
        assert chi2.sf(stat, n - 1) > 1e-4, (col, stat)


def test_ransac_degenerate_triples():
    from usip_b200.evaluation import registration as reg
    rng = np.random.default_rng(5)
    T = kitti_gt_transforms()[:3]
    n = 24
    y = np.zeros((3, n, 3))
    y[0] = np.outer(np.linspace(-5, 5, n), [1.0, 0.5, 0.2])               # all collinear
    y[1] = rng.uniform(-5, 5, (n, 3)); y[1][::2] = y[1][0]                 # many duplicates of one point
    y[2] = np.repeat(rng.uniform(-5, 5, (1, 3)), n, 0)                     # every point identical
    x = np.einsum("bij,bmj->bmi", T[:, :, :3], y) + T[:, None, :, 3]
    corr = np.broadcast_to(np.stack([np.arange(n), np.arange(n)], 1), (3, n, 2)).astype(np.int32)
    r = reg.ransac_fit_rt(x, y, corr, np.full(3, n, np.int32), max_trials=200)
    torch.cuda.synchronize()
    Rt = r.Rt.cpu().numpy(); mask = r.inlier_mask.cpu().numpy().astype(bool)
    for b in range(3):
        assert int(r.status[b]) == 0
        R = Rt[b, :, :3]
        assert np.abs(R @ R.T - np.eye(3)).max() <= 1e-9 and abs(np.linalg.det(R) - 1) <= 1e-9
        assert mask[b].sum() == int(r.n_inliers[b]) >= 3
        d = np.linalg.norm(x[b] - (y[b] @ R.T + Rt[b, :, 3]), axis=1)
        assert (d[mask[b]] < 1.0 + 1e-6).all()                # the refit still explains the inliers it was fitted to


def test_evaluate_registration_end_to_end_synthetic():
    from usip_b200.evaluation import registration as reg
    B, M = 16, 256
    ratios = np.linspace(0.1, 0.5, B)
    T, anc, pos, ad, pd = _pairs(B, M, ratios, seed=3)
    res = reg.evaluate_registration(anc, ad, pos, pd, T, protocol="kitti", seed=11)
    # the same stages by hand, with the sample table, against the oracle
    corr, cnt = reg.match_descriptors(ad, pd)
    r = reg.ransac_fit_rt(anc, pos, corr, cnt, seed=11, return_samples=True)
    assert torch.equal(r.Rt, torch.from_numpy(res["Rt"]).cuda())
    corr_h, cnt_h, table = corr.cpu().numpy(), cnt.cpu().numpy(), r.samples.cpu().numpy()
    for b in range(B):
        o = _oracle_pair(corr_h[b], cnt_h[b], anc[b], pos[b], table[b], 1.0, 10001)
        dt, deg = orc.compare_transform(T[b], o["Rt"])
        assert bool(res["success"][b]) == (not (dt > 2 or deg > 5)), b
        assert abs(res["delta_t"][b] - dt) <= 1e-6 and abs(res["delta_deg"][b] - deg) <= 1e-6
    assert res["wrong_counter"] == 0
    assert res["delta_t"].max() < 0.05 and res["delta_deg"].max() < 0.2    # within the 0.05 m keypoint noise
    assert np.all(np.abs(res["n_inliers"] / res["n_corr"] - ratios) < 0.1)
    # Oxford protocol: the 5-NN union adds ~8 wrong matches per keypoint, so the low-ratio pairs exhaust 10,001 trials
    ox = reg.evaluate_registration(anc, ad, pos, pd, T, protocol="oxford", seed=11)
    assert (ox["n_corr"] >= res["n_corr"]).all() and ox["success"][-8:].all()
    assert ox["rte_mean"] < 0.5 and ox["rre_mean"] < 1.0     # the refit also takes wrong matches that land within 1 m


def test_repeatability_vs_oracle():
    from usip_b200.evaluation import registration as reg
    rng = np.random.default_rng(6)
    T = kitti_gt_transforms()[100:104]
    anc, pos = [], []
    for b, (ma, mb) in enumerate([(128, 100), (37, 64), (256, 256), (5, 1)]):
        p = rng.uniform(-20, 20, (mb, 3)).astype(np.float32)
        a = p[rng.integers(0, mb, ma)] @ T[b, :, :3].T.astype(np.float32) + T[b, :, 3].astype(np.float32)
        a = a + rng.normal(0, 0.4, a.shape)                    # about half within 0.5 m
        anc.append(a.astype(np.float32)); pos.append(p)
    res = reg.repeatability(anc, pos, T, radius=0.5)
    for b in range(4):
        rep, d = orc.repeatability(anc[b], pos[b], T[b], 0.5)
        near = np.abs(d - 0.5) < 1e-5
        lo, hi = ((d < 0.5) & ~near).sum(), ((d < 0.5) | near).sum()
        got = res["per_pair"][b] * len(anc[b])
        assert lo - 1e-9 <= got <= hi + 1e-9, b
        if not near.any():
            assert res["per_pair"][b] == rep
    assert res["mean"] == pytest.approx(res["per_pair"].mean()) and res["min"] == res["per_pair"].min()
    assert res["keypoint_mean"] == pytest.approx(np.mean([128, 37, 256, 5]))


def test_registration_through_the_models_recovers_a_translation():
    """FPS keypoints of a synthetic cloud and a translated copy, descriptors from ModelDescriptor.run_model (balls hold
    fewer than K points, so max pooling makes the descriptor order-invariant): the registration recovers the shift."""
    from usip_b200 import ops
    from usip_b200.evaluation import registration as reg
    from usip_b200.models.keypoint_descriptor import ModelDescriptor
    from tests.util_gpu import make_opt
    torch.manual_seed(0)
    rng = np.random.default_rng(7)
    N, M, S, K = 2048, 96, 4, 64
    pc = rng.uniform(-5, 5, (1, 3, N)).astype(np.float32)
    sn = rng.normal(size=(1, S, N)).astype(np.float32)
    shift = np.array([1.5, -0.75, 0.25], np.float32)
    _, kp = ops.fps(cu(pc.transpose(0, 2, 1)), torch.zeros(1, dtype=torch.int32, device="cuda"), M)
    opt = make_opt(batch_size=1, input_pc_num=N, node_num=M, surface_normal_len=S, ball_radius=1.0, ball_nsamples=K,
                   descriptor_len=128)
    md = ModelDescriptor(opt)
    pc_a, pc_p = cu(pc), cu(pc + shift[None, :, None])
    kp_p = kp + cu(shift)[None, :, None]
    # every ball around a keypoint holds fewer than K points
    d = torch.cdist(kp.transpose(1, 2), pc_a.transpose(1, 2))
    assert int((d < opt.ball_radius).sum(2).max()) < K
    da = md.run_model(pc_a, cu(sn), kp.contiguous())
    dp = md.run_model(pc_p, cu(sn), kp_p.contiguous())
    T = np.concatenate([np.eye(3), -shift[:, None].astype(np.float64)], 1)[None]   # maps pos points into the anc frame
    res = reg.evaluate_registration(kp.transpose(1, 2), da.transpose(1, 2), kp_p.transpose(1, 2), dp.transpose(1, 2), T)
    assert res["wrong_counter"] == 0
    assert np.abs(res["Rt"][0][:, 3] + shift).max() < 1e-3 and np.abs(res["Rt"][0][:, :3] - np.eye(3)).max() < 1e-3
