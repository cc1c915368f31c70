"""-m gpu parity tests of the individual C-ABI kernels against oracle/ (bit-exact for index / integer work,
1e-4 relative for fp) and against outputs of the reference's own CUDA extensions stored in tests/golden/."""
import numpy as np
import pytest
import torch

from oracle import usip_oracle as orc
from tests.util_gpu import cu, dev, digest, golden, rel_err

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------ index_max
def test_index_max_golden_cases():
    from usip_b200 import index_max
    g = golden("index_max.npz")
    for c in "abcd":
        out = index_max.forward_cuda_shared_mem(cu(g["data_" + c]), cu(g["index_" + c]), int(g["K_" + c]))
        assert out.dtype == torch.int32
        assert np.array_equal(out.cpu().numpy(), g["out_" + c]), c
        out2 = index_max.forward_cuda(cu(g["data_" + c]), cu(g["index_" + c]), int(g["K_" + c]))
        assert np.array_equal(out2.cpu().numpy(), g["out_" + c]), c


@pytest.mark.parametrize("B,C,N,K", [(3, 64, 5000, 512), (2, 128, 16384, 512), (1, 5, 1001, 7), (2, 16, 4096, 3000),
                                     (1, 2, 2048, 20000)])
def test_index_max_vs_oracle(B, C, N, K):
    from usip_b200 import index_max
    rng = np.random.default_rng(B * 1000 + C)
    data = rng.normal(size=(B, C, N)).astype(np.float32)
    data[:, 0] = np.maximum(data[:, 0], 0)            # post-ReLU like: many exact zeros / ties
    data[0, -1, ::5] = -0.0
    index = rng.integers(0, K, size=(B, N)).astype(np.int32)
    out = index_max.forward_cuda_shared_mem(cu(data), cu(index), K).cpu().numpy()
    assert np.array_equal(out, orc.index_max(data, index, K))


def test_index_max_bucket_kernel_edge_cases():
    """The HBM-speed bucket kernel (csrc/indexmax.cu; taken when B*C >= 64, C >= 8, N % 4 == 0, N <= 16384): exact ties
    (first maximum wins whatever the bucket order), values at / below the -1000 floor, NaN, empty clusters, -0.0."""
    from usip_b200 import index_max
    rng = np.random.default_rng(77)
    B, C, N, K = 5, 16, 2000, 48
    data = (np.round(rng.normal(size=(B, C, N)) * 2) / 2).astype(np.float32)          # many exact ties
    data[:, 1, :] = -2000.0                                                            # never above the floor
    data[:, 2, ::3] = -1000.0                                                          # exactly the floor: not '>'
    data[:, 3, ::7] = np.nan
    data[:, 4, ::2] = -0.0
    data[:, 5, :] = 3.5                                                                # one value everywhere: n = first of the cluster
    index = rng.integers(0, K // 2, size=(B, N)).astype(np.int32)                      # upper half of the clusters empty
    out = index_max.forward_cuda_shared_mem(cu(data), cu(index), K).cpu().numpy()
    assert np.array_equal(out, orc.index_max(data, index, K))


def index_max_full_size_inputs():
    torch.manual_seed(0)
    data = torch.randn(16, 128, 16384, device=dev())
    index = torch.randint(0, 512, (16, 16384), device=dev(), dtype=torch.int32)
    return data, index


def test_index_max_vs_reference_cuda_full_size():
    """KITTI shape (B'=16, C=128, N=16384, K=512) against the reference's own kernel (global-mem variant, no cap); its
    output on these inputs is stored as a digest (tools/make_golden_gpu.py)."""
    from usip_b200 import index_max
    data, index = index_max_full_size_inputs()
    ours = index_max.forward_cuda_shared_mem(data, index, 512)
    assert digest(ours) == str(golden("ref_gpu_ops.npz")["index_max_full_size"])


def test_index_max_errors():
    from usip_b200 import index_max
    d = torch.randn(1, 2, 8); i = torch.zeros(1, 8, dtype=torch.int32)
    with pytest.raises(RuntimeError):
        index_max.forward_cuda_shared_mem(d, i, 2)                      # CPU tensor
    with pytest.raises(RuntimeError):
        index_max.forward_cuda_shared_mem(d.to(dev()).transpose(1, 2), i.to(dev()), 2)   # non-contiguous
    with pytest.raises(NotImplementedError):
        index_max.forward_cpu(d, i, 2)


# ------------------------------------------------------------------------------------------ ball query
@pytest.mark.parametrize("B,M,N,K,r", [(2, 33, 1000, 16, 0.9), (1, 8, 257, 64, 2.5), (2, 16, 4096, 64, 0.2)])
def test_ball_query_dist_vs_oracle(B, M, N, K, r):
    from usip_b200 import ball_query
    rng = np.random.default_rng(5)
    dist = np.abs(rng.normal(size=(B, M, N))).astype(np.float32)
    dist[0, 0] = 100.0                 # zero hits
    dist[0, 1, :3] = 0.0               # very few hits
    dist[0, 2] = 0.0                   # everything hits
    out = ball_query.forward_cuda_shared_mem(cu(dist), r, K).cpu().numpy()
    assert np.array_equal(out, orc.ball_query_dist(dist, r, K))


def ball_query_inputs():
    torch.manual_seed(1)
    pc = torch.rand(8, 3, 4096, device=dev()) * 8
    kp = pc[:, :, :256] + 0.05 * torch.randn(8, 3, 256, device=dev())
    dist = torch.norm(kp.unsqueeze(3) - pc.unsqueeze(2), dim=1).contiguous()
    return pc, kp, dist


def test_ball_query_vs_reference_cuda():
    """Against the reference's own kernel, whose output on these inputs is stored as a digest (tools/make_golden_gpu.py)."""
    from usip_b200 import ball_query
    pc, kp, dist = ball_query_inputs()
    theirs = str(golden("ref_gpu_ops.npz")["ball_query"])
    ours = ball_query.forward_cuda_shared_mem(dist, 1.0, 64)
    assert digest(ours) == theirs
    fused, _ = ball_query.forward_fused(pc.contiguous(), None, kp.contiguous(), 1.0, 64, want_group=False)
    assert digest(fused) == theirs


@pytest.mark.parametrize("S", [0, 4])
def test_ball_group_fused_vs_oracle(S):
    from usip_b200 import ball_query
    rng = np.random.default_rng(9)
    B, N, M, K = 2, 3000, 40, 32
    pc = (rng.uniform(-4, 4, (B, 3, N))).astype(np.float32)
    sn = rng.normal(size=(B, S, N)).astype(np.float32)
    kp = pc[:, :, :M] + rng.normal(0, 0.1, (B, 3, M)).astype(np.float32)
    kp[:, :, 0] = 99.0
    idx, grp = ball_query.forward_fused(cu(pc), cu(sn) if S else None, cu(kp), 1.0, K)
    ref_idx = orc.ball_query_xyz(pc, kp, 1.0, K)
    assert np.array_equal(idx.cpu().numpy(), ref_idx)
    x_aug = np.concatenate([pc, sn], 1) if S else pc
    gi = np.broadcast_to(ref_idx.astype(np.int64).reshape(B, 1, M * K), (B, 3 + S, M * K))
    ball = np.take_along_axis(x_aug, gi, axis=2).reshape(B, 3 + S, M, K).copy()
    ball[:, :3] -= kp[:, :, :, None]
    assert np.array_equal(grp.cpu().numpy(), ball)


# ------------------------------------------------------------------------------------------ grouping
def test_som_assign_sort_mean_segmax():
    from usip_b200 import ops
    B, N, M, S = 3, 5000, 96, 4
    d = orc.synth_pair(B, N, M, S, kind="lidar", seed=3)
    x, sn, node = d["src_pc"], d["src_sn"], d["src_node"].copy()
    node[:, :, 7] = 1000.0             # empty cluster
    min_idx, count = ops.som_assign(cu(x), cu(node))
    ref_idx = orc.som_assign(x, node)
    assert np.array_equal(min_idx.cpu().numpy(), ref_idx)
    cnt = np.stack([np.bincount(ref_idx[b], minlength=M) for b in range(B)])
    assert np.array_equal(count.cpu().numpy(), cnt)
    seg_off, perm, row_seg = ops.cluster_sort(min_idx, M)
    so, pm, rs = seg_off.cpu().numpy(), perm.cpu().numpy(), row_seg.cpu().numpy()
    for b in range(B):
        assert np.array_equal(so[b], np.concatenate([[0], np.cumsum(cnt[b])]))
        assert np.array_equal(pm[b], np.argsort(ref_idx[b], kind="stable"))          # stable: ascending n per node
        assert np.array_equal(rs[b], b * M + ref_idx[b][pm[b]])
    cmean, x_aug = ops.cluster_mean_decenter(cu(x), cu(sn), seg_off, perm, M, ldx=8)
    cm = cmean.cpu().numpy(); xa = x_aug.cpu().numpy().reshape(B, N, 8)
    for b in range(B):
        for m in range(M):
            pts = x[b][:, ref_idx[b] == m]
            ref_mean = pts.sum(1) / (pts.shape[1] + 1e-5) if pts.shape[1] else np.zeros(3)
            assert np.allclose(cm[b, :, m], ref_mean, rtol=1e-5, atol=1e-5)
        exp = np.concatenate([x[b][:, pm[b]] - cm[b][:, ref_idx[b][pm[b]]], sn[b][:, pm[b]]], 0).T
        assert np.allclose(xa[b, :, :7], exp, rtol=0, atol=1e-6)
        assert np.all(xa[b, :, 7] == 0)
    # segmented max of a random feature map over the sorted rows
    C = 64
    F = torch.randn(B * N, C, device=dev())
    pooled, arg = ops.segmax(F, C, seg_off, perm, B, N, M)
    Fh = F.cpu().numpy().reshape(B, N, C)
    pl, ag = pooled.cpu().numpy().reshape(B, M, C), arg.cpu().numpy().reshape(B, M, C)
    for b in range(B):
        # express in the reference's (B,C,N) layout / original point order and use the index_max oracle
        orig = np.zeros((C, N), np.float32); orig[:, pm[b]] = Fh[b].T
        idx = orc.index_max(orig[None], ref_idx[b][None], M)[0]                       # (C,M) original n
        exp = np.take_along_axis(orig, idx.astype(np.int64), 1).T * (cnt[b] > 0)[:, None]
        assert np.array_equal(pl[b], exp)
        got_n = pm[b][np.clip(ag[b] - b * N, 0, N - 1)]
        assert np.array_equal(np.where(cnt[b][:, None] > 0, got_n, 0), np.where(cnt[b][:, None] > 0, idx.T, 0))


def test_knn_nodes_vs_oracle():
    from usip_b200 import ops
    rng = np.random.default_rng(4)
    pts = rng.uniform(-10, 10, (4, 3, 200)).astype(np.float32)
    pts[0, :, 50] = pts[0, :, 20]          # duplicate point -> exact ties
    for K in (16, 32):
        out = ops.knn_nodes(cu(pts), K).cpu().numpy()
        ref, _ = orc.knn(pts, pts, K)
        assert np.array_equal(out, ref)


def test_query_topk_api():
    from usip_b200.util import som
    g = golden("query_topk.npz")
    d = orc.synth_pair(2, 2048, 64, 4, kind="lidar", seed=int(g["seed_lidar"]))
    mask, row_max, min_idx = som.query_topk(cu(g["node_lidar"]), cu(d["src_pc"]), 64, 1)
    assert np.array_equal(min_idx.cpu().numpy().astype(np.int32), g["min_idx_lidar"])
    assert np.array_equal(row_max.cpu().numpy(), g["row_max_lidar"])
    assert mask.shape == (2, 2048, 64) and int(mask.sum()) == 2 * 2048


# ------------------------------------------------------------------------------------------ shared-MLP layer
def _layer_ref(X, W, b, scale, shift, relu, addend, add_idx):
    A = X.astype(np.float64)
    if scale is not None:
        A = A * scale + shift
    if relu:
        A = np.maximum(A, 0)
    Y = A @ W.astype(np.float64).T
    if b is not None:
        Y = Y + b
    if addend is not None:
        Y = Y + addend[add_idx]
    return Y


@pytest.mark.parametrize("precision", [0, 1])             # 0: fp32 SIMT, 1: tcgen05 3xTF32
@pytest.mark.parametrize("P,Cin,Cout,group", [(1000, 7, 64, 0), (4096, 64, 64, 16), (2048, 128, 128, 32),
                                              (1536, 256, 256, 16), (1024, 512, 512, 64), (700, 640, 512, 0),
                                              (512, 256, 4, 0), (640, 131, 256, 0),
                                              # many tiles per CTA, ragged tails
                                              (16512, 256, 256, 16), (8320, 512, 512, 32), (16400, 64, 256, 0)])
def test_layer_fwd(P, Cin, Cout, group, precision):
    from usip_b200 import ops
    if precision and not (Cin % 32 == 0 and Cout % 64 == 0):
        pytest.skip("tensor-core path needs Cin%32==0 and Cout%64==0")
    rng = np.random.default_rng(P + Cin)
    ldx = Cin + (8 - Cin % 8) % 8
    X = rng.normal(size=(P, ldx)).astype(np.float32)
    W = (rng.normal(size=(Cout, Cin)) / np.sqrt(Cin)).astype(np.float32)
    b = rng.normal(size=Cout).astype(np.float32)
    scale = rng.normal(size=Cin).astype(np.float32); shift = rng.normal(size=Cin).astype(np.float32)
    G = 37
    addend = rng.normal(size=(G, Cout)).astype(np.float32)
    add_idx = rng.integers(0, G, size=P).astype(np.int32)
    Xd = cu(X)
    Y = torch.empty((P, Cout), device=dev())
    want_grp = bool(group and P % group == 0)
    nt = ops.stat_slots(P, Cout, precision, group if want_grp else 0, want_grp)
    part = torch.full((nt, 2, Cout), float("nan"), device=dev())     # every slot must be written
    kw = {}
    if group and P % group == 0:
        Q = P // group
        kw = dict(gmax=torch.empty((Q, Cout), device=dev()), gmin=torch.empty((Q, Cout), device=dev()),
                  garg_max=torch.empty((Q, Cout), dtype=torch.int32, device=dev()),
                  garg_min=torch.empty((Q, Cout), dtype=torch.int32, device=dev()), group=group)
    ops.layer_fwd(Xd, cu(W), cu(b), P, Cin, Cout, ldx=ldx, in_scale=cu(scale), in_shift=cu(shift), in_relu=True,
                  addend=cu(addend), add_index=cu(add_idx), Y=Y, stat_partial=part, precision=precision, **kw)
    torch.cuda.synchronize()
    ref = _layer_ref(X[:, :Cin], W, b, scale, shift, True, addend, add_idx)
    e = rel_err(Y.cpu().numpy(), ref)
    assert e < 2e-5, e
    st = part.cpu().numpy().astype(np.float64).sum(0)
    assert rel_err(st[0], ref.sum(0)) < 1e-4 and rel_err(st[1], (ref ** 2).sum(0)) < 1e-4
    if kw:
        Yh = Y.cpu().numpy().reshape(P // group, group, Cout)
        assert np.array_equal(kw["gmax"].cpu().numpy(), Yh.max(1)) and np.array_equal(kw["gmin"].cpu().numpy(), Yh.min(1))
        assert np.array_equal(kw["garg_max"].cpu().numpy(), Yh.argmax(1)) and np.array_equal(kw["garg_min"].cpu().numpy(), Yh.argmin(1))
    # plain variant: no prologue / addend / stats, strided output
    Ybig = torch.zeros((P, Cout + 16), device=dev())
    ops.layer_fwd(Xd, cu(W), None, P, Cin, Cout, ldx=ldx, Y=Ybig[:, 8:8 + Cout], precision=precision)
    assert rel_err(Ybig[:, 8:8 + Cout].cpu().numpy(), _layer_ref(X[:, :Cin], W, None, None, None, False, None, None)) < 2e-5
    assert float(Ybig[:, :8].abs().max()) == 0 and float(Ybig[:, 8 + Cout:].abs().max()) == 0


def test_bn_finalize_matches_batch_norm():
    from usip_b200 import ops
    P, C = 3000, 96
    torch.manual_seed(0)
    Y = torch.randn(P, C, device=dev()) * 3 + 1.5
    W = torch.eye(C, device=dev())
    tile = ops.tile_rows(); nt = (P + tile - 1) // tile
    part = torch.zeros((nt, 2, C), device=dev())
    out = torch.empty_like(Y)
    ops.layer_fwd(Y, W, None, P, C, C, Y=out, stat_partial=part)
    gamma = torch.rand(C, device=dev()) + 0.5; beta = torch.randn(C, device=dev())
    rm = torch.randn(C, device=dev()); rv = torch.rand(C, device=dev()) + 0.5
    rm2, rv2 = rm.clone(), rv.clone()
    scale = torch.empty(C, device=dev()); shift = torch.empty(C, device=dev())
    ops.bn_finalize(part, nt, P, C, gamma, beta, 1e-5, 0.1, rm2, rv2, scale, shift)
    ref = torch.nn.functional.batch_norm(Y, rm, rv, gamma, beta, True, 0.1, 1e-5)
    assert rel_err((Y * scale + shift).cpu().numpy(), ref.cpu().numpy()) < 1e-5
    assert rel_err(rm2.cpu().numpy(), rm.cpu().numpy()) < 1e-5 and rel_err(rv2.cpu().numpy(), rv.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------------------ losses
def test_losses_vs_golden_and_grads():
    from usip_b200.models import losses
    from tests.util_gpu import make_opt
    g = golden("losses.npz")
    opt = make_opt()
    crit = losses.ChamferLoss_Brute(opt)
    src = cu(g["src"]).requires_grad_(True); dst = cu(g["dst"]).requires_grad_(True)
    ss = cu(g["sig_src"]).requires_grad_(True); sd = cu(g["sig_dst"]).requires_grad_(True)
    loss, pure, weighted = crit(src, dst, ss, sd)
    assert rel_err(loss.item(), g["loss"]) < 1e-5 and rel_err(pure.item(), g["pure"]) < 1e-5
    assert rel_err(weighted.item(), g["weighted"]) < 1e-5
    loss.backward()
    for got, name in ((src.grad, "g_src"), (dst.grad, "g_dst"), (ss.grad, "g_sig_src"), (sd.grad, "g_sig_dst")):
        assert rel_err(got.cpu().numpy(), g[name]) < 1e-4, name
    kp = cu(g["kp"]).requires_grad_(True)
    d = losses.SingleSideChamferLoss_Brute(opt)(kp, cu(g["pc"]))
    assert np.array_equal(d.detach().cpu().numpy(), g["single"])          # sqrt of the same fp32 sum: bit exact
    d.mean().backward()
    assert rel_err(kp.grad.cpu().numpy(), g["g_kp"]) < 1e-5
    l2, _, _ = crit(cu(g["src"]), cu(g["dst"]))
    assert rel_err(l2.cpu().numpy(), g["nosigma"]) < 1e-6


def test_pairwise_min_full_size_properties():
    """KITTI size (16 x 512 keypoints vs 16384 points): bit-exact vs the oracle on a slice + sortedness property."""
    from usip_b200 import ops
    rng = np.random.default_rng(0)
    pc = rng.uniform(-40, 40, (16, 3, 16384)).astype(np.float32)
    kp = pc[:, :, :512] + rng.normal(0, 0.3, (16, 3, 512)).astype(np.float32)
    d, arg = ops.pairwise_min(cu(kp), cu(pc))
    dh, ah = d.cpu().numpy(), arg.cpu().numpy()
    rd, ra = orc.pairwise_min(kp[:2], pc[:2])
    assert np.array_equal(dh[:2], rd) and np.array_equal(ah[:2], ra)
    # property: the reported neighbour really is at the reported distance, and no sampled point is closer
    sel = np.take_along_axis(pc, np.broadcast_to(ah[:, None, :].astype(np.int64), (16, 3, 512)), 2)
    assert np.allclose(np.sqrt(((kp - sel) ** 2).sum(1)), dh, rtol=1e-6)
    samp = pc[:, :, ::64]
    dd = np.sqrt(((kp[:, :, :, None] - samp[:, :, None, :]) ** 2).sum(1)).min(2)
    assert np.all(dh <= dd * (1 + 1e-6))


def test_ball_group_grid_full_size_vs_reference_cuda():
    """Oxford descriptor shape (B'=16, N=16384, 1024 keypoints, r=1, K=64): cell-binned fused kernel vs the reference
    kernel on the materialised torch.norm distance matrix (bit-exact indices, stored as digests by
    tools/make_golden_gpu.py), plus a dense cloud that exercises the sort path (hits > K) and the in-order fallback
    (hits > 256)."""
    g = golden("ref_gpu_ops.npz")
    for dense, pc, sn, kp, K in ball_group_grid_cases():
        B, M = kp.shape[0], kp.shape[2]
        idx, grp, rows = ops_ball_group(pc, sn, kp, 1.0, K)
        assert digest(idx) == str(g["ball_group_grid_dense" if dense else "ball_group_grid"]), dense
        x_aug = torch.cat([pc, sn], 1)
        gi = idx.long().view(B, 1, M * K).expand(B, 7, M * K)
        ball = torch.gather(x_aug, 2, gi).view(B, 7, M, K).clone()
        ball[:, :3] -= kp.unsqueeze(3)
        assert torch.equal(grp, ball)
        assert torch.equal(rows.view(B, M, K, 8)[..., :7].permute(0, 3, 1, 2), ball)


def ball_group_grid_cases():
    torch.manual_seed(3)
    for dense in (False, True):
        B, N, M, K = (16, 16384, 1024, 64) if not dense else (2, 8192, 256, 64)
        ext = torch.tensor([40.0, 2.0, 40.0], device=dev()).view(1, 3, 1) * (0.08 if dense else 1.0)
        pc = (torch.rand(B, 3, N, device=dev()) * 2 - 1) * ext
        sn = torch.randn(B, 4, N, device=dev())
        sel = torch.randint(0, N, (B, M), device=dev())
        kp = torch.gather(pc, 2, sel.unsqueeze(1).expand(B, 3, M)) + 0.1 * torch.randn(B, 3, M, device=dev())
        yield dense, pc, sn, kp, K


def ops_ball_group(pc, sn, kp, r, K):
    from usip_b200 import ops
    return ops.ball_group(pc.contiguous(), sn.contiguous(), kp.contiguous(), r, K, want_group=True, rows_ld=8)


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("P,Cout,Cin", [(4096, 128, 64), (8192, 256, 256), (5000, 512, 512), (4100, 128, 128), (6144, 512, 640)])
def test_wgrad(P, Cout, Cin, precision):
    """gW += GY^T act(X): SIMT and tcgen05 (MN-major 3xTF32) kernels against fp64."""
    from usip_b200 import _lib
    from usip_b200.ops import _p, _stream
    rng = np.random.default_rng(P + Cout)
    GY = rng.normal(size=(P, Cout)).astype(np.float32)
    X = rng.normal(size=(P, Cin)).astype(np.float32)
    sc = rng.normal(size=Cin).astype(np.float32); sh = rng.normal(size=Cin).astype(np.float32)
    gW = torch.zeros((Cout, Cin), device=dev())
    gy, x, s_, h_ = cu(GY), cu(X), cu(sc), cu(sh)
    _lib.check(_lib.load().usip_wgrad(_p(gy), Cout, _p(x), Cin, _p(s_), _p(h_), 1, _p(gW), Cin, P, Cout, Cin, precision,
                                      _stream()), "usip_wgrad")
    torch.cuda.synchronize()
    A = np.maximum(X.astype(np.float64) * sc + sh, 0)
    ref = GY.astype(np.float64).T @ A
    e = rel_err(gW.cpu().numpy(), ref)
    assert e < 2e-5, e


def test_fps_vs_reference_golden_and_oracle():
    """GPU farthest point sampling: the reference's FarthestSampler outputs (golden), the oracle at the KITTI node shape
    (16 clouds x 5461 candidates x 512 nodes) bit for bit, and the drop-in class incl. its RNG consumption."""
    from usip_b200 import ops
    from usip_b200.data.kitti_detector_loader import FarthestSampler
    g = golden("fps.npz")
    fs = FarthestSampler(dev())
    for name in ("lidar", "dup", "few"):
        pts, k = g["pts_" + name], int(g["k_" + name])
        np.random.seed(77)
        nodes = fs.sample(pts, k)
        assert nodes.dtype == np.float64 and np.array_equal(nodes, g["nodes_" + name]), name
        np.random.seed(77); np.random.randint(len(pts))
        after = np.random.randint(1 << 30)
        np.random.seed(77); fs.sample(pts, k)
        assert np.random.randint(1 << 30) == after                       # exactly one draw consumed
    rng = np.random.default_rng(5)
    B, Ns, k = 16, 5461, 512
    pts = (rng.uniform(-40, 40, (B, Ns, 3)) * np.array([1, 0.05, 1])).astype(np.float32)
    pts[3, 100:200] = pts[3, 0:100]                                      # exact duplicates
    start = rng.integers(0, Ns, B).astype(np.int32)
    idx, nodes = ops.fps(cu(pts), cu(start), k)
    idx = idx.cpu().numpy(); nodes = nodes.cpu().numpy()
    for b in range(B):
        ref = orc.fps(pts[b], int(start[b]), k)
        assert np.array_equal(idx[b], ref), b
        assert np.array_equal(nodes[b], pts[b][ref].T)


def test_nms_vs_reference_golden_and_oracle(tmp_path):
    """GPU radius NMS: the reference's own nms() outputs (golden), the oracle on a batch at the detector's shape, the
    batched select_keypoints() and the .bin wire format."""
    from usip_b200 import ops
    from usip_b200.evaluation import save_keypoints as sk
    g = golden("nms.npz")
    for name in ("lidar", "dense", "ties", "off"):
        kp, sg, r = g["kp_" + name], g["sigma_" + name], float(g["radius_" + name])
        vk, vs = sk.nms(kp, sg, r, device=dev())
        assert np.array_equal(vk, g["valid_kp_" + name]) and np.array_equal(vs, g["valid_sigma_" + name]), name
    rng = np.random.default_rng(9)
    B, M = 16, 512
    kp = (rng.uniform(-40, 40, (B, 3, M)) * np.array([1, 0.05, 1]).reshape(1, 3, 1)).astype(np.float32)
    sg = rng.uniform(0.01, 2.0, (B, M)).astype(np.float32)
    sg[2, ::7] = sg[2, 0]                                                # equal sigmas: ties by index
    idx, cnt = ops.nms(cu(kp), cu(sg), 3.0)
    idx = idx.cpu().numpy(); cnt = cnt.cpu().numpy()
    sel = sk.select_keypoints(cu(kp), cu(sg), 3.0, desired_keypoint_num=128)
    for b in range(B):
        ref = orc.nms(kp[b].T.copy(), sg[b], 3.0)
        assert cnt[b] == len(ref) and np.array_equal(idx[b, :cnt[b]], ref) and np.all(idx[b, cnt[b]:] == -1), b
        assert np.array_equal(sel[b].cpu().numpy(), kp[b].T[ref[:128]])
    f = str(tmp_path / "kp.bin")
    sk.write_keypoints_bin(f, sel[0])
    assert np.array_equal(sk.read_keypoints_bin(f), sel[0].cpu().numpy())
    a = rng.normal(size=(100, 8)).astype(np.float64); np.save(str(tmp_path / "pc.npy"), a)
    pc, sn = sk.read_pointcloud_npy(str(tmp_path / "pc.npy"))
    assert pc.dtype == np.float32 and pc.shape == (100, 3) and np.array_equal(sn, a[:, 3:7].astype(np.float32))


def test_point_on_surface_loss_vs_reference_golden():
    """KeypointOnPCLoss(keypoint, pc, sn) = PointOnSurfaceLoss ('point_to_plane'): value (B,M,1,1) and keypoint gradient
    against the reference's autograd (golden), S=4 surface-normal channels."""
    from usip_b200.models import losses
    from tests.util_gpu import make_opt
    g = golden("losses.npz")
    kp = cu(g["kp"]).requires_grad_(True)
    out = losses.KeypointOnPCLoss(make_opt())(kp, cu(g["pc"]), cu(g["sn4"]))
    assert tuple(out.shape) == tuple(g["on_surface"].shape)
    (out.mean() * 0.37).backward()
    assert rel_err(out.detach().cpu().numpy(), g["on_surface"]) < 1e-4
    assert rel_err(kp.grad.cpu().numpy(), g["g_kp_surface"]) < 1e-4


@pytest.mark.parametrize("B,Ma,Nb", [(2, 64, 700), (2, 100, 5000), (8, 512, 5000), (3, 33, 2049)])
def test_pairwise_min_all_paths_vs_oracle(B, Ma, Nb):
    """usip_pairwise_min_f32 picks one of two kernels by database size (direct, or split database with a 64-bit atomicMin
    merge): distances and first-index arg-min equal the oracle bit for bit, exact ties included."""
    from usip_b200 import ops
    rng = np.random.default_rng(B * 1000 + Ma)
    a = rng.normal(size=(B, 3, Ma)).astype(np.float32)
    b = np.round(rng.normal(size=(B, 3, Nb)) * 4).astype(np.float32) / 4          # coarse grid: many exact distance ties
    b[:, :, Nb // 2:Nb // 2 + 50] = b[:, :, 0:50]                                  # duplicated points far apart in index
    a[:, :, 0] = b[:, :, 7]                                                        # a zero distance
    d, arg = ops.pairwise_min(cu(a), cu(b))
    rd, ra = orc.pairwise_min(a, b)
    assert np.array_equal(arg.cpu().numpy(), ra) and np.array_equal(d.cpu().numpy(), rd)


@pytest.mark.parametrize("case", ["lidar", "ties", "flat", "identical", "far_queries", "nonfinite", "small", "volume"])
def test_pairwise_min_grid_equals_brute_force(case):
    """usip_pairwise_min_grid_f32 (cell grid + shell search) against the brute-force kernels on the same inputs: distances
    and first-index arg-min bit for bit -- exact ties, duplicated points, degenerate extents, queries far outside the cloud
    (ring fallback), non-finite points and queries."""
    from usip_b200 import ops
    rng = np.random.default_rng(["lidar", "ties", "flat", "identical", "far_queries", "nonfinite", "small", "volume"].index(case))
    B, Ma, Nb = 4, 512, 16384
    if case == "lidar":
        r = np.abs(rng.normal(0, 15, (B, Nb))) + 1; th = rng.uniform(0, 2 * np.pi, (B, Nb))
        b = np.stack([r * np.cos(th), rng.normal(-1.5, 0.3, (B, Nb)), r * np.sin(th)], 1).astype(np.float32)
        a = b[:, :, rng.integers(0, Nb, Ma)] + rng.normal(0, 0.5, (B, 3, Ma)).astype(np.float32)
    elif case == "ties":
        b = np.round(rng.normal(size=(B, 3, Nb)) * 3).astype(np.float32)             # integer lattice: masses of exact ties
        a = np.round(rng.normal(size=(B, 3, Ma)) * 3).astype(np.float32) + 0.5
    elif case == "flat":
        b = rng.uniform(-30, 30, (B, 3, Nb)).astype(np.float32); b[:, 1] = 2.0        # zero extent along y
        a = rng.uniform(-35, 35, (B, 3, Ma)).astype(np.float32)
    elif case == "identical":
        b = np.full((B, 3, Nb), 1.25, np.float32)
        a = rng.normal(size=(B, 3, Ma)).astype(np.float32)
    elif case == "far_queries":
        b = rng.uniform(-1, 1, (B, 3, Nb)).astype(np.float32)
        a = (rng.normal(size=(B, 3, Ma)) * 50).astype(np.float32)
        a[:, :, :64] = rng.uniform(-1, 1, (B, 3, 64)).astype(np.float32)
    elif case == "nonfinite":
        b = rng.uniform(-10, 10, (B, 3, Nb)).astype(np.float32)
        b[0, 0, ::7] = np.nan; b[1, 2, ::5] = np.inf; b[2, :, :] = np.nan; b[3, 1, 3] = -np.inf
        a = rng.uniform(-10, 10, (B, 3, Ma)).astype(np.float32)
        a[:, 0, 5] = np.nan; a[:, 1, 9] = np.inf
    elif case == "small":
        B, Ma, Nb = 3, 37, 301
        b = rng.normal(size=(B, 3, Nb)).astype(np.float32); a = rng.normal(size=(B, 3, Ma)).astype(np.float32)
    else:                                                                             # uniform volume, many cells per axis
        b = rng.uniform(-1, 1, (B, 3, Nb)).astype(np.float32)
        a = rng.uniform(-1.2, 1.2, (B, 3, Ma)).astype(np.float32)
    dg, ag = ops.pairwise_min(cu(a), cu(b), method="grid")
    db, ab = ops.pairwise_min(cu(a), cu(b), method="brute")
    assert torch.equal(ag, ab), int((ag != ab).sum())
    assert torch.equal(dg.view(torch.int32), db.view(torch.int32))


@pytest.mark.parametrize("case", ["kitti", "modelnet", "ties", "flat", "outliers", "nonfinite", "tiny"])
def test_som_assign_grid_equals_brute_force(case):
    """usip_som_assign_grid_f32 against the brute-force scan: nearest-node index (smallest m on ties) and per-node counts
    identical -- node sets from FPS-like subsets, lattice ties, degenerate extents, points far from every node, non-finite
    points and nodes."""
    from usip_b200 import ops
    rng = np.random.default_rng(["kitti", "modelnet", "ties", "flat", "outliers", "nonfinite", "tiny"].index(case) + 10)
    B, N, M = 4, 16384, 512
    if case == "kitti":
        r = np.abs(rng.normal(0, 15, (B, N))) + 1; th = rng.uniform(0, 2 * np.pi, (B, N))
        x = np.stack([r * np.cos(th), rng.normal(-1.5, 0.3, (B, N)), r * np.sin(th)], 1).astype(np.float32)
        node = x[:, :, rng.choice(N, M, replace=False)] + rng.normal(0, 0.05, (B, 3, M)).astype(np.float32)
    elif case == "modelnet":
        B, N, M = 6, 5000, 64
        x = rng.normal(size=(B, 3, N)).astype(np.float32); x /= np.linalg.norm(x, axis=1, keepdims=True)
        node = x[:, :, rng.choice(N, M, replace=False)].copy()
    elif case == "ties":
        x = np.round(rng.normal(size=(B, 3, N)) * 3).astype(np.float32) + 0.5
        node = np.round(rng.normal(size=(B, 3, M)) * 3).astype(np.float32)
        node[:, :, M // 2:M // 2 + 40] = node[:, :, :40]                              # duplicated nodes
    elif case == "flat":
        x = rng.uniform(-30, 30, (B, 3, N)).astype(np.float32); x[:, 1] = 0.0
        node = rng.uniform(-30, 30, (B, 3, M)).astype(np.float32); node[:, 1] = 0.0
    elif case == "outliers":
        x = (rng.normal(size=(B, 3, N)) * 40).astype(np.float32)
        node = rng.uniform(-1, 1, (B, 3, M)).astype(np.float32)
    elif case == "nonfinite":
        x = rng.uniform(-10, 10, (B, 3, N)).astype(np.float32); x[0, 0, ::9] = np.nan; x[1, 2, ::11] = np.inf
        node = rng.uniform(-10, 10, (B, 3, M)).astype(np.float32); node[2, 1, ::3] = np.nan; node[3] = np.inf
    else:
        B, N, M = 2, 1500, 70
        x = rng.normal(size=(B, 3, N)).astype(np.float32); node = rng.normal(size=(B, 3, M)).astype(np.float32)
    ig, cg = ops.som_assign(cu(x), cu(node), method="grid")
    ib, cb = ops.som_assign(cu(x), cu(node), method="brute")
    assert torch.equal(ig, ib), int((ig != ib).sum())
    assert torch.equal(cg, cb)


def test_knn_gather_matches_reference_semantics():
    """operations.knn_gather_by_indexing / knn_gather_wrapper (operations.py:243-287): out[b,c,n,k] = src[b,c,I[b,n,k]],
    i.e. the expand + torch.gather of the reference, bit for bit (pure data movement)."""
    from usip_b200.models import operations
    torch.manual_seed(3)
    B, C, N, K = 3, 5, 700, 9
    src = torch.randn(B, C, N, device=dev())
    idx = torch.randint(0, N, (B, N, K), device=dev())
    out = operations.knn_gather_by_indexing(src, idx)
    ref = torch.gather(src.unsqueeze(3).expand(B, C, N, K), 2, idx.unsqueeze(1).expand(B, C, N, K))
    assert torch.equal(out, ref)
    out3 = operations.knn_gather_wrapper(src[:, :3].contiguous(), idx)
    assert torch.equal(out3, ref[:, :3])
