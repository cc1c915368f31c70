"""-m gpu parity at the FULL BASELINE.json shapes against THE REFERENCE ITSELF, run on a B200.

The unmodified reference (`models/keypoint_detector.py`, `networks.py`, `losses.py`, ... with its own two CUDA extensions)
was run with TF32 switched off on the identical seeded tensors and parameters by tools/make_golden_gpu.py, in float32 and
in float64; what these tests compare against is stored in tests/golden/ref_gpu_*.npz.  A full-size output or gradient is
too large to keep whole, so the goldens hold every element of the small tensors, a fixed, evenly spread sample of the
elements of each large one, statistics the generator computed over the whole tensor, and digests where the comparison is
bit-exact.  Compared:

  * keypoints, sigmas, recomputed nodes (sampled) and all six loss terms, eval- and train-mode BatchNorm: 1e-4 relative
    to the reference's full-tensor max (the bar `north_star` states for fp features and the chamfer loss);
  * the parameter gradients of one optimize() step: per tensor max|g - g_ref| <= GRAD_EL * max|g_ref| on the stored
    elements, the L2 error extrapolated from them, and | ||g|| - ||g_ref|| | <= GRAD_NORM * ||g_ref|| over the whole
    tensor;
  * BatchNorm running statistics after the step (all elements), parameters after the Adam step (stored elements);
  * descriptor: ball-query indices (via x_features) bit-exact, descriptors 1e-4.

Also the boundary test SURVEY section 7 step 1 asks for: the reference's own `models/networks.py` (unmodified) running
on top of THIS repo's `index_max` / `ball_query` operator modules must reproduce the run on its own extensions
bit-for-bit (networks.py:118,131,359).  Those two tests execute the reference's Python sources, which this repository
does not contain: they run where oracle/build_ref.py staged them under oracle/_ref and are skipped elsewhere."""
import random
import zlib

import numpy as np
import pytest
import torch

from oracle import usip_oracle as orc
from tests.util_gpu import digest, golden, load_params, make_opt

pytestmark = pytest.mark.gpu
REL = 1e-4
# Gradient tolerances.  The arbiter is the reference itself run in FLOAT64 on the same GPU.  Its own float32 run (TF32 off)
# already differs from that by 0.2-1.4 % of max|g| per element and ~0.5 % in L2 (measured on B200, DESIGN.md section 2):
# every max() (cluster max-pool, max over the K neighbours) routes its whole gradient through ONE arg-max row and the
# weight gradient of those layers is a sum of only B'*M = 8192 such rows per channel, so a handful of arg-max / ReLU
# decisions that flip under a 1e-7 perturbation of the forward move single elements by ~1e-2.  This repo is held to the
# same band: absolute caps a little above the reference's own float32 error AND at most GRAD_SLACK times that error.
GRAD_EL = 3e-2        # max|g - g64| / scale, any single element
GRAD_L2 = 1.5e-2      # ||g - g64|| / ||g64|| per tensor
GRAD_NORM = 3e-3      # | ||g|| - ||g64|| | / ||g64||
GRAD_SLACK = 8.0      # ... and never more than this factor above the reference's own float32-vs-float64 error

KEYS = ("src_pc", "src_sn", "src_node", "dst_pc", "dst_sn", "dst_node", "R", "scale", "shift")
CONFIGS = {
    # BASELINE.json configs[2] / configs[1] (SURVEY.md 8d)
    "kitti": dict(B=8, N=16384, M=512, S=4, Kn=16, kind="lidar", lb=1e-3, alpha=0.01, seed=1236),
    "modelnet": dict(B=24, N=5000, M=512, S=3, Kn=32, kind="object", lb=1e-4, alpha=1.0, seed=1235),
}
OUTS = ("node", "kp", "sig")
SAMPLE = 256           # stored elements of each parameter / gradient tensor (smaller tensors whole)
OUT_SAMPLE = 512       # stored elements of each detector output (keypoints, sigmas, nodes)
DESC_SAMPLE = 2048     # stored descriptor elements


def sample_idx(n, k, name):
    """Positions of the stored elements of a flattened tensor of n elements: all of them when n <= k, else k distinct,
    evenly spread ones (a multiple of a prime larger than n is never 0 mod n), fixed by `name`."""
    if n <= k:
        return np.arange(n)
    return np.sort((np.arange(k, dtype=np.int64) * 2654435761 + zlib.crc32(name.encode())) % n)


@pytest.fixture(scope="module")
def ref():
    from oracle import build_ref, ref_shim
    if not (ref_shim.reference_available() and build_ref.have("index_max") and build_ref.have("ball_query")):
        pytest.skip("oracle/_ref (reference extensions + staged reference tree) not built")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return ref_shim.modules(mode="cuda")


def _params(cfg):
    P = orc.init_detector_params(S=cfg["S"], seed=cfg["seed"], randomize_bn=True)
    P["mlp3.conv.weight"] = (P["mlp3.conv.weight"] * 1000).astype(np.float32)   # non-trivial keypoint offsets / sigmas
    return P


def _mk(cls, cfg, use_tc=True):
    opt = make_opt(batch_size=cfg["B"], input_pc_num=cfg["N"], node_num=cfg["M"], surface_normal_len=cfg["S"],
                   node_knn_k_1=cfg["Kn"], loss_sigma_lower_bound=cfg["lb"], keypoint_on_pc_alpha=cfg["alpha"],
                   scene="outdoor" if cfg["kind"] == "lidar" else "object", use_tensor_cores=use_tc)
    md = cls(opt)
    load_params(md.detector, _params(cfg))
    return md


def _randomized_state(net, seed):
    """state_dict for a (reference or own) network from a seeded generator alone: convolution weights with PyTorch's
    default init bound 1/sqrt(fan_in), non-trivial BatchNorm affine / running statistics.  Keys are visited in sorted
    order, so both implementations of a network receive the same values."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in sorted(net.state_dict().items()):
        v = v.detach().cpu().clone()
        if k.endswith("norm.weight") or k.endswith("running_var"):
            v = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith("norm.bias") or k.endswith("running_mean"):
            v = torch.randn(v.shape, generator=g) * 0.1
        elif k.endswith("conv.bias"):
            v = torch.randn(v.shape, generator=g) * 0.05
        elif k.endswith("conv.weight"):
            v = (torch.rand(v.shape, generator=g) * 2 - 1) / float(np.sqrt(v[0].numel()))
        sd[k] = v
    return sd


def _loss_vec(md):
    return np.array([md.loss.item(), md.loss_chamfer.item(), md.chamfer_pure.item(), md.chamfer_weighted.item(),
                     md.loss_keypoint_on_pc_src.item(), md.loss_keypoint_on_pc_dst.item()], np.float64)


def _outs(md):
    return dict(kp=torch.cat([md.src_keypoints, md.dst_keypoints]).detach().cpu().numpy(),
                sig=torch.cat([md.src_sigmas, md.dst_sigmas]).detach().cpu().numpy(),
                node=torch.cat([md.src_node_recomputed, md.dst_node_recomputed]).detach().cpu().numpy(),
                loss=_loss_vec(md))


def _cmp_outs(a, G, mode, tag, fails):
    """Our outputs against the reference's `mode` run (eval / train / train64) at the stored positions, relative to the
    reference's max over the whole tensor."""
    e = {}
    for t in OUTS:
        got = a[t].reshape(-1)[sample_idx(a[t].size, OUT_SAMPLE, t)].astype(np.float64)
        e[t] = float(np.abs(got - G["%s_%s" % (mode, t)]).max() / max(float(G["%s_%s_absmax" % (mode, t)]), 1e-12))
    b_loss = G[mode + "_loss"]
    e_loss = float(np.max(np.abs(a["loss"] - b_loss) / np.maximum(np.abs(b_loss), 1e-6)))
    print("[%s] rel err: nodes %.2e keypoints %.2e sigmas %.2e losses %.2e" % (tag, e["node"], e["kp"], e["sig"], e_loss))
    if not (e["node"] < 1e-5 and e["kp"] < REL and e["sig"] < REL and e_loss < REL):
        fails.append((tag, e["node"], e["kp"], e["sig"], e_loss))


def _sample(k, a):
    """The elements of tensor k (flattened) that the golden stores."""
    return a.reshape(-1)[sample_idx(a.size, SAMPLE, k)]


@pytest.mark.parametrize("name", ["kitti", "modelnet"])
def test_detector_full_size_vs_reference_gpu(name):
    from usip_b200.models.keypoint_detector import ModelDetector
    cfg = CONFIGS[name]
    G = golden("ref_gpu_detector_%s.npz" % name)
    d = orc.synth_pair(cfg["B"], cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=cfg["seed"])
    ins = [torch.from_numpy(d[k]) for k in KEYS]

    md = _mk(ModelDetector, cfg)
    md.set_input(*ins)
    md.test_model()
    fails = []
    _cmp_outs(_outs(md), G, "eval", name + " eval-BN", fails)
    random.seed(0); np.random.seed(0)
    md.optimize(epoch=0)
    torch.cuda.synchronize()
    _cmp_outs(_outs(md), G, "train", name + " train-BN", fails)
    _cmp_outs(_outs(md), G, "train64", name + " train-BN vs float64 reference", fails)

    # ---- gradients.  Scale of a tensor = max|g| of the float64 reference; a conv BIAS is measured on the scale of its
    # layer's weight gradient: biases in front of a train-mode BatchNorm -- and the two BN-free PointNet output biases,
    # whose constant shift the next layer's BatchNorm removes -- have an analytically (near-)zero gradient, so both
    # implementations hold only rounding noise there (this repo: exact zeros for the BN-preceded ones).
    # gstat|k, over the whole tensor: max|g64|, ||g64||, max|g32 - g64|, ||g32 - g64||.  The single-element error is taken
    # over the stored elements; the L2 error is extrapolated from them (exact where the tensor is stored whole); the
    # norm error uses our whole tensor.
    worst = dict(ours=0.0, ref32=0.0, norm=0.0, cos=1.0)
    for k, p in md.detector.named_parameters():
        g_full = p.grad.detach().cpu().numpy().astype(np.float64)
        g, g64 = _sample(k, g_full), G["g64|" + k].astype(np.float64)
        amax64, n64, dmax32, dl2_32 = G["gstat|" + k]
        wk = k.replace("bias", "weight")
        w_amax64, w_n64 = G["gstat|" + wk][:2]
        scale = amax64
        if k.endswith("conv.bias"):
            scale = max(scale, w_amax64)
        e_ours, e_ref = _grad_err(g, g64, scale), dmax32 / max(scale, 1e-300)
        l2_scale = max(n64, w_n64 * 1e-3 if k.endswith("conv.bias") else n64, 1e-300)
        l2_ours = np.sqrt(g_full.size / g.size * ((g - g64) ** 2).sum()) / l2_scale
        l2_ref = dl2_32 / l2_scale
        analytic_zero = n64 < 1e-6 * w_n64 if k.endswith("conv.bias") else False
        e_norm = 0.0 if analytic_zero else abs(np.linalg.norm(g_full) - n64) / max(n64, 1e-300)
        cos = 1.0 if analytic_zero else float((g * g64).sum() / max(np.linalg.norm(g) * np.linalg.norm(g64), 1e-300))
        worst = dict(ours=max(worst["ours"], e_ours), ref32=max(worst["ref32"], e_ref), norm=max(worst["norm"], e_norm),
                     cos=min(worst["cos"], cos), l2=max(worst.get("l2", 0.0), l2_ours), l2ref=max(worst.get("l2ref", 0.0), l2_ref))
        print("   grad %-44s max-el ours %.2e ref32 %.2e | L2 ours %.2e ref32 %.2e | norm err %.2e" % (k, e_ours, e_ref, l2_ours, l2_ref, e_norm))
        ok = (e_ours <= GRAD_EL and l2_ours <= GRAD_L2 and e_norm <= GRAD_NORM and
              e_ours <= max(2e-3, GRAD_SLACK * e_ref) and l2_ours <= max(1e-3, GRAD_SLACK * l2_ref))
        if not ok:
            fails.append((k, e_ours, e_ref, l2_ours, l2_ref, e_norm))
    print("[%s] gradients vs the float64 reference: worst max|dg|/scale ours %.2e (reference float32 %.2e); "
          "worst L2 ours %.2e (reference float32 %.2e); worst norm err %.2e"
          % (name, worst["ours"], worst["ref32"], worst["l2"], worst["l2ref"], worst["norm"]))
    assert not fails, fails

    # ---- state after the step.  step|k = (parameter before - parameter after) / lr of the reference, big|k marks the
    # elements whose float32 reference gradient is well above the comparison tolerance (> 0.2 max|g32|, and none where
    # the gradient is analytically zero: there the reference steps on rounding noise).
    sd = md.detector.state_dict()
    lr = md.opt.lr
    P0 = _params(cfg)
    for k, v in sd.items():
        a = v.detach().cpu().numpy().astype(np.float64)
        if k.endswith("num_batches_tracked"):
            assert np.array_equal(a, G["buf|" + k]), k
        elif k.endswith("running_mean") or k.endswith("running_var"):
            b_ = G["buf|" + k].astype(np.float64)
            assert np.abs(a - b_).max() <= 2e-4 * max(np.abs(b_).max(), 1e-6), k
        else:
            # first Adam step = lr*g/(|g|+1e-8): same landing point wherever the gradient is well above the comparison
            # tolerance, at most 2*lr apart where it is noise (dead channels, |g| ~ 1e-8)
            a = _sample(k, a)
            b_ = _sample(k, np.asarray(P0[k], np.float32)).astype(np.float64) - lr * G["step|" + k].astype(np.float64)
            big = np.unpackbits(G["big|" + k], count=a.size).astype(bool)
            assert np.abs(a - b_).max() <= 2.0 * lr * 1.0001 + 1e-7, k
            if big.any():
                assert np.abs(a - b_)[big].max() <= 0.02 * lr + 1e-7, (k, np.abs(a - b_)[big].max())


def _grad_err(g, ref, scale):
    return float(np.abs(g - ref).max() / max(scale, 1e-300))


def descriptor_inputs():
    """BASELINE configs[3]: Oxford descriptor path B'=16, N=16384, 1024 keypoints, r=1.0, K=64."""
    B, N, M, S, K = 16, 16384, 1024, 4, 64
    d = orc.synth_pair(B // 2, N, 128, S, kind="lidar", seed=1237)
    pc = np.concatenate([d["src_pc"], d["dst_pc"]]); sn = np.concatenate([d["src_sn"], d["dst_sn"]])
    rng = np.random.default_rng(5)
    pick = rng.integers(0, N, size=(B, M))
    kp = np.take_along_axis(pc, pick[:, None, :], axis=2) + rng.normal(0, 0.1, size=(B, 3, M)).astype(np.float32)
    kp = kp.astype(np.float32)
    opt = make_opt(batch_size=B // 2, input_pc_num=N, node_num=M, surface_normal_len=S, ball_radius=1.0, ball_nsamples=K,
                   descriptor_len=128)
    x, s, k = (torch.from_numpy(a).cuda() for a in (pc, sn, kp))
    return opt, x, s, k


def descriptor_run(cls, opt, x, s, k):
    """{mode: (descriptors, x_features)} of a freshly built DescriptorLiteOld with the seeded state, eval and train BN."""
    net = cls(opt).cuda()
    net.load_state_dict(_randomized_state(net, seed=3))
    out = {}
    for mode in ("eval", "train"):
        net.train(mode == "train")
        np.random.seed(11)                                   # networks.py:345 draws the point permutation from numpy
        with torch.no_grad(), torch.cuda.device(0):
            desc, feats = net(x, s, k, mode == "train", 0)
        out[mode] = (desc.cpu().numpy(), feats)
    del net
    torch.cuda.empty_cache()
    return out


def test_descriptor_full_size_vs_reference_gpu():
    from usip_b200.models import networks as our_networks
    G = golden("ref_gpu_descriptor.npz")
    out = descriptor_run(our_networks.DescriptorLiteOld, *descriptor_inputs())
    for mode in ("eval", "train"):
        do, fo = out[mode]
        assert digest(fo) == str(G[mode + "_feats"]), "x_features (gathered, decentred ball groups) must be bit-identical"
        got = do.reshape(-1)[sample_idx(do.size, DESC_SAMPLE, "descriptor")].astype(np.float64)
        e = float(np.abs(got - G[mode + "_desc"]).max() / float(G[mode + "_desc_absmax"]))
        print("[descriptor %s-BN] rel err %.2e" % (mode, e))
        assert e < REL, (mode, e)


def test_reference_networks_on_our_operators(ref):
    """The unmodified reference networks.py with its `index_max` / `ball_query` modules replaced by this repo's drop-in
    operator modules: outputs must be bit-identical to the run on the reference's own extensions."""
    import ball_query as ref_bq
    import index_max as ref_im
    from usip_b200 import ball_query as our_bq
    from usip_b200 import index_max as our_im
    nets = ref.networks
    assert nets.index_max is ref_im and nets.ball_query is ref_bq
    cfg = dict(B=2, N=8192, M=256, S=4, Kn=16, kind="lidar", lb=1e-3, alpha=0.01, seed=21)
    d = orc.synth_pair(cfg["B"], cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=cfg["seed"])
    ins = [torch.from_numpy(d[k]) for k in KEYS]
    rmd = _mk(ref.keypoint_detector.ModelDetector, cfg)
    rmd.set_input(*ins)
    res = {}
    calls = {"im": 0, "bq": 0}

    def counted(fn, key):
        def f(*a):
            calls[key] += 1
            return fn(*a)
        return f

    class _OurIM:
        forward_cuda_shared_mem = staticmethod(counted(our_im.forward_cuda_shared_mem, "im"))
        forward_cuda = staticmethod(counted(our_im.forward_cuda, "im"))

    class _OurBQ:
        forward_cuda_shared_mem = staticmethod(counted(our_bq.forward_cuda_shared_mem, "bq"))

    # descriptor inputs
    Bd, Md = 4, 256
    pcd = torch.from_numpy(np.concatenate([d["src_pc"], d["dst_pc"]])).cuda()
    snd = torch.from_numpy(np.concatenate([d["src_sn"], d["dst_sn"]])).cuda()
    kpd = pcd[:, :, :Md].contiguous() + 0.05
    dopt = make_opt(batch_size=2, input_pc_num=cfg["N"], node_num=Md, surface_normal_len=4, ball_radius=1.0, ball_nsamples=64)
    dnet = nets.DescriptorLiteOld(dopt).cuda()
    dnet.load_state_dict(_randomized_state(dnet, seed=3))
    dnet.eval()
    try:
        for tag, im, bq in (("ref", ref_im, ref_bq), ("ours", _OurIM, _OurBQ)):
            nets.index_max, nets.ball_query = im, bq
            with torch.no_grad():
                rmd.test_model()
                np.random.seed(4)
                with torch.cuda.device(0):
                    desc, feats = dnet(pcd, snd, kpd, False, 0)
            res[tag] = [t.detach().cpu().numpy() for t in (rmd.src_keypoints, rmd.dst_keypoints, rmd.src_sigmas,
                                                            rmd.dst_sigmas, rmd.loss.reshape(1), desc, feats)]
    finally:
        nets.index_max, nets.ball_query = ref_im, ref_bq
    assert calls["im"] == 2 and calls["bq"] == 1          # networks.py:118,131 and :359 really went through our modules
    for a, b in zip(res["ours"], res["ref"]):
        assert np.array_equal(a, b)


def test_dropin_directory_serves_the_reference_networks(ref, tmp_path):
    """INTEGRATION.md section 2, literally: a fresh interpreter puts <repo>/usip_b200/dropin in front of the (staged)
    reference tree, imports the reference's own `models.networks` -- whose `import index_max` / `import ball_query`
    (networks.py:17-18) now resolve to this repo -- and must reproduce, bit for bit, what the reference computes on its own
    extensions in this process."""
    import os, subprocess, sys
    cfg = dict(B=2, N=4096, M=128, S=4, Kn=16, kind="lidar", lb=1e-3, alpha=0.01, seed=31)
    d = orc.synth_pair(cfg["B"], cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=cfg["seed"])
    rmd = _mk(ref.keypoint_detector.ModelDetector, cfg)
    rmd.set_input(*[torch.from_numpy(d[k]) for k in KEYS])
    with torch.no_grad():
        rmd.test_model()
    want = os.path.join(tmp_path, "want.npz")
    np.savez(want, kp=torch.cat([rmd.src_keypoints, rmd.dst_keypoints]).cpu().numpy(),
             sig=torch.cat([rmd.src_sigmas, rmd.dst_sigmas]).cpu().numpy(), loss=np.float32(rmd.loss.item()))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, os; sys.path.insert(0, %r)\n"
        "import numpy as np, torch\n"
        "torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False\n"
        "from oracle import ref_shim, usip_oracle as orc\n"
        "ref = ref_shim.modules(mode='cuda', operators='dropin')\n"
        "import index_max, ball_query\n"
        "drop = os.path.join(%r, 'usip_b200', 'dropin')\n"
        "assert index_max.__file__.startswith(drop) and ball_query.__file__.startswith(drop), index_max.__file__\n"
        "assert ref.networks.index_max is index_max and 'oracle' in ref.networks.__file__\n"
        "from tests import test_gpu_vs_reference as T\n"
        "cfg = %r\n"
        "d = orc.synth_pair(cfg['B'], cfg['N'], cfg['M'], cfg['S'], kind=cfg['kind'], seed=cfg['seed'])\n"
        "rmd = T._mk(ref.keypoint_detector.ModelDetector, cfg)\n"
        "rmd.set_input(*[torch.from_numpy(d[k]) for k in T.KEYS])\n"
        "with torch.no_grad(): rmd.test_model()\n"
        "w = np.load(%r)\n"
        "assert np.array_equal(torch.cat([rmd.src_keypoints, rmd.dst_keypoints]).cpu().numpy(), w['kp'])\n"
        "assert np.array_equal(torch.cat([rmd.src_sigmas, rmd.dst_sigmas]).cpu().numpy(), w['sig'])\n"
        "assert np.float32(rmd.loss.item()) == w['loss']\n"
        "print('dropin ok')\n" % (root, root, cfg, want))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "dropin ok" in r.stdout, (r.stdout[-1000:], r.stderr[-3000:])
