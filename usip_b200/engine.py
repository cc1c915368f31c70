"""Fused B200 execution plan of the USIP detector / descriptor networks.

This is NOT a layer-by-layer translation of models/networks.py: the (B,C,N) activations of the reference
are replaced by point-major [rows, C] buffers over points SORTED BY NODE, so that
  * index_max + gather + mask (networks.py:117-120,130-133) is a contiguous segmented max,
  * the un-pool gather (networks.py:123-126) and the concat that follows become a per-node GEMM whose
    result is added in the consuming layer's epilogue (W [a;b] = Wa a + Wb b),
  * the kNN group tensor (B,3+C,M,K) of layers.py:422-429 is never built: W_feat @ feat is computed once
    per node and gathered; the broadcast-max half of layers.py:435 likewise,
  * train-mode BatchNorm (layers.py:69-71) is "epilogue emits statistics -> finalize -> next layer's
    prologue normalises": every pre-BN activation is written once and read once,
  * max_k relu(bn(y_k)) (layers.py:433,438) comes from per-group max/min of the raw GEMM output.
All arithmetic happens in libusip_b200.so; torch only owns memory / streams / autograd plumbing.
"""
import torch

from . import _lib, ops

f32 = torch.float32
i32 = torch.int32
EPS = 1e-5

# Optional per-op device timing (bench.py): set PROFILE = {} to record CUDA-event pairs around every op of the
# plan on the launching stream; collect_profile() turns them into mean milliseconds per op name.
PROFILE = None


class _Prof:
    def __init__(self, name, flops=None, nbytes=None, precision=None):
        self.on = PROFILE is not None
        if self.on:
            self.name, self.flops, self.nbytes, self.precision = name, flops, nbytes, precision

    def __enter__(self):
        if self.on:
            self.e0 = torch.cuda.Event(enable_timing=True); self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *a):
        if self.on:
            self.e1.record()
            rec = PROFILE.setdefault(self.name, dict(ev=[], flops=self.flops, bytes=self.nbytes, precision=self.precision))
            rec["ev"].append((self.e0, self.e1))
        return False


def collect_profile():
    out = {}
    if not PROFILE:
        return out
    torch.cuda.synchronize()
    for k, rec in PROFILE.items():
        ms = [a.elapsed_time(b) for a, b in rec["ev"]]
        out[k] = dict(ms=sum(ms) / len(ms), n=len(ms), flops=rec["flops"], bytes=rec["bytes"], precision=rec["precision"])
    return out


def _w2d(w):
    """(Cout, Cin[,1[,1]]) conv weight -> [Cout, Cin] view that remembers its owning Parameter (packed-weight cache)."""
    t = w.detach().reshape(w.shape[0], -1)
    t._owner = w
    return t


def _cols(t, a, b=None):
    """Column slice of a _w2d view (concat halves of a conv weight), keeping the owner."""
    v = t[:, a:b]
    v._owner = getattr(t, "_owner", None)
    return v


class BNState:
    """Folded affine of one BatchNorm for the current step (+ what backward needs)."""
    __slots__ = ("scale", "shift", "mean", "invstd", "count")


# Packed (hi/lo TF32, pre-swizzled) weight tiles are cached per weight view and re-used while the parameter's
# autograd version counter is unchanged (inference / fwd-only loops); an optimizer step bumps the version and the
# next launch re-packs into the same workspace.
class _PackEntry:
    """One packed-weight workspace: the version it was packed at, and -- once the layer has run -- a copy of its descriptor,
    so that prepack_weights() can re-pack it together with all the others in one launch."""
    __slots__ = ("ver", "ws", "ptr", "desc", "keep", "used_step")

    def __init__(self, ver, ws, ptr):
        self.ver, self.ws, self.ptr, self.desc, self.keep, self.used_step = ver, ws, ptr, None, None, -1


_PACK_STEP = [0]


def _tc_workspace(W, P, Cin, Cout, group, transposed, prec=1):
    """-> (workspace, already_packed, entry or None)"""
    owner = getattr(W, "_owner", None)
    if owner is None:                                  # unknown provenance: never reuse packed tiles
        return torch.empty((2 * Cin * Cout,), dtype=f32, device=W.device), False, None
    cache = owner.__dict__.setdefault("_usip_tc", {})  # lives and dies with the Parameter object
    key = (W.data_ptr() - owner.data_ptr(), W.stride(0), P, Cin, Cout, bool(transposed), group > 32, prec)
    ver = (owner._version, _lib.WEIGHT_GEN[0])
    ent = cache.get(key)
    if ent is not None and ent.ver == ver and ent.ptr == owner.data_ptr():
        ent.used_step = _PACK_STEP[0]
        return ent.ws, True, ent
    if ent is None or ent.ptr != owner.data_ptr():
        ent = _PackEntry(ver, ent.ws if ent is not None else torch.empty((2 * Cin * Cout,), dtype=f32, device=W.device),
                         owner.data_ptr())
        cache[key] = ent
    ent.ver = ver
    ent.used_step = _PACK_STEP[0]
    return ent.ws, False, ent


def prepack_weights(module):
    """Re-pack, in ONE launch (usip_layer_tc_pack_many), every tensor-core weight matrix of `module` that went stale since it
    was last packed (an optimizer step moved the weights) and was used by the previous step.  The train step calls this first:
    its 26 per-layer pack launches become one.  Layers that have not run yet are packed by their own first launch."""
    jobs = []
    step = _PACK_STEP[0]
    for p in module.parameters():
        cache = p.__dict__.get("_usip_tc")
        if not cache:
            continue
        ver = (p._version, _lib.WEIGHT_GEN[0])
        for ent in cache.values():
            if ent.desc is not None and ent.used_step == step and ent.ver != ver and ent.ptr == p.data_ptr():
                jobs.append((ent, ver))
    _PACK_STEP[0] = step + 1
    if not jobs:
        return 0
    ops.layer_tc_pack_many([ent.desc for ent, _ in jobs])
    for ent, ver in jobs:
        ent.ver = ver
    return len(jobs)


def invalidate_packed_weights(module):
    """Drop every cached packed (hi/lo TF32) weight tile of `module`'s parameters.  The cache key follows the autograd
    version counter, which in-place writes through `.data` (legacy checkpoint loaders, EMA, weight clipping) do NOT bump:
    call this after such a write.  load_state_dict(), train()/eval() switches and the optimizer step invalidate by
    themselves (models/networks.py hooks; Adam bumps the version)."""
    for p in module.parameters():
        p.__dict__.pop("_usip_tc", None)


_TC_PREC = 1          # usip_layer_desc.precision of the tcgen05 3xTF32 kernel


def _precision_for(P, Cin, Cout, use_tc, group=0):
    """Tensor-core kernel only for shapes it implements; everything else takes the fp32 SIMT kernel.  The tcgen05 group
    epilogue handles groups of 16/32/64/128 rows (the SIMT kernel any multiple of 4 dividing 128)."""
    if group and group not in (16, 32, 64, 128):
        return 0
    return _TC_PREC if (use_tc and Cin % 32 == 0 and Cout % 64 == 0 and P >= 1024) else 0


class LayerRunner:
    """Runs conv1x1(+BN) layers of one nn.Module tree through usip_layer_fwd / usip_bn_finalize."""

    def __init__(self, training, use_tc, dev):
        self.training = training
        self.use_tc = use_tc
        self.dev = dev

    def bn_state(self, norm, part, ntiles, count, momentum):
        C = norm.weight.numel()
        st = BNState()
        st.scale = torch.empty(C, dtype=f32, device=self.dev)
        st.shift = torch.empty(C, dtype=f32, device=self.dev)
        st.count = count
        if self.training:
            st.mean = torch.empty(C, dtype=f32, device=self.dev)
            st.invstd = torch.empty(C, dtype=f32, device=self.dev)
            ops.bn_finalize(part, ntiles, count, C, norm.weight.detach(), norm.bias.detach(), EPS, momentum,
                            norm.running_mean, norm.running_var, st.scale, st.shift, st.mean, st.invstd)
        else:
            st.mean = st.invstd = None
            ops.bn_eval_affine(norm.weight.detach(), norm.bias.detach(), norm.running_mean, norm.running_var, EPS,
                               st.scale, st.shift)
        return st

    def partials(self, P, Cout, prec=0, group=0, want_group=False):
        ntiles = ops.stat_slots(P, Cout, prec, group, want_group)
        if not self.training:
            return None, ntiles
        return torch.empty((ntiles, 2, Cout), dtype=f32, device=self.dev), ntiles

    def run(self, X, P, W, bias, norm=None, momentum=0.1, prev=None, relu_in=None, Y=None, write_y=True,
            addend=None, add_index=None, add_group=0, group=0, want_group=False, want_arg=False, count=None, name="layer"):
        """Y = act(X) W^T + bias (+addend); returns (Y, BNState or None, group dict or None)."""
        Cout, Cin = W.shape
        if Y is None and write_y:
            Y = torch.empty((P, Cout), dtype=f32, device=self.dev)
        prec = _precision_for(P, Cin, Cout, self.use_tc, group if want_group else 0)
        part, ntiles = self.partials(P, Cout, prec, group, want_group) if norm is not None else (None, 0)
        grp = None
        if want_group:
            Q = P // group
            grp = dict(gmax=torch.empty((Q, Cout), dtype=f32, device=self.dev),
                       gmin=torch.empty((Q, Cout), dtype=f32, device=self.dev))
            if want_arg:
                grp["amax"] = torch.empty((Q, Cout), dtype=i32, device=self.dev)
                grp["amin"] = torch.empty((Q, Cout), dtype=i32, device=self.dev)
        ws, packed, pack_ent = _tc_workspace(W, P, Cin, Cout, group if want_group else 0, False, prec) if prec else (None, False, None)
        with _Prof("%s[%dx%d->%d]" % (name, P, Cin, Cout), flops=2.0 * P * Cin * Cout,
                   precision="3xTF32 tcgen05" if prec else "fp32 SIMT"):
            ops.layer_fwd(X, W, bias, P, Cin, Cout,
                          in_scale=None if prev is None else prev.scale, in_shift=None if prev is None else prev.shift,
                          in_relu=(prev is not None) if relu_in is None else relu_in,
                          addend=addend, add_index=add_index, add_group=add_group, Y=Y if write_y else None,
                          stat_partial=part,
                          gmax=None if grp is None else grp["gmax"], gmin=None if grp is None else grp["gmin"],
                          garg_max=None if grp is None else grp.get("amax"),
                          garg_min=None if grp is None else grp.get("amin"),
                          group=group, precision=prec, tc_ws=ws, tc_packed=packed, pack_entry=pack_ent)
        st = None
        if norm is not None:
            with _Prof("bn_finalize"):
                st = self.bn_state(norm, part, ntiles, P if count is None else count, momentum)
        return Y, st, grp

    def run_module(self, m, X, P, epoch=None, **kw):
        """run() for the conv1x1(+BN) module m: weight, bias and BatchNorm (if m has one) come from m.  Passing the epoch
        decays the BN momentum (layers.py:62-66); the reference calls some layers without it, and then it never decays."""
        norm = getattr(m, "norm", None)
        mom = 0.1 if norm is None else _bn_mom(norm, epoch)
        return self.run(X, P, _w2d(m.conv.weight), m.conv.bias.detach(), norm, mom, **kw)


def _bn_mom(norm, epoch):
    """layers.py:62-66 -- side effect on norm.momentum kept, like the reference."""
    if (epoch is not None) and (epoch >= 1) and (norm.momentum_decay_step is not None) and (norm.momentum_decay_step > 0):
        norm.momentum = norm.momentum_original * (norm.momentum_decay ** (epoch // norm.momentum_decay_step))
        if norm.momentum < 0.01:
            norm.momentum = 0.01
    return norm.momentum


def _knn_head_forward(R, net, AGG, C1, coords, Bp, M, Kn, epoch, keep):
    """GeneralKNNFusionModule on the nodes (layers.py:401-440) + head mlp1/2/3 + softplus (networks.py:143-154).
    AGG [Q, C1+C2]: columns [0,C1) hold the per-node feature (pool 2) on entry, columns [C1,C1+C2) receive the fused kNN
    feature.  coords (B,3,M) are the nodes the kNN runs on and the keypoint offsets are added to.  Shared by RPN_Detector /
    RPN_DetectorLite (coords = cluster means) and the ablation networks RPN_Detector_KNN / _Ball (coords = the given nodes)."""
    opt = net.opt
    dev = AGG.device
    Q = Bp * M
    G = Q * Kn
    kb = net.knnlayer_1.layers_before
    ka = net.knnlayer_1.layers_after
    C2 = ka[-1].conv.weight.shape[0]
    pool2 = AGG[:, :C1]
    cmean = coords
    # ---- GeneralKNNFusionModule (layers.py:401-440)
    with _Prof("knn_nodes"):
        knn_i = ops.knn_nodes(cmean, Kn)
    W5 = _w2d(kb[0].conv.weight)
    Cb = W5.shape[0]
    Z, _, _ = R.run(pool2, Q, _cols(W5, 3), None, relu_in=False, name="knn_b0_node")
    Y5 = torch.empty((G, Cb), dtype=f32, device=dev)
    part5, nt5 = R.partials(G, Cb)
    with _Prof("knn_combine", nbytes=8.0 * G * Cb):
        ops.knn_combine(Z, cmean, knn_i, W5, W5.stride(0), kb[0].conv.bias.detach(), Y5, part5, Bp, M, Kn, Cb)
    bn5 = R.bn_state(kb[0].norm, part5, nt5, G, _bn_mom(kb[0].norm, epoch))
    before = [(kb[0], Y5, bn5)]                      # (module, pre-BN output, BNState) of every layer
    for li in range(1, len(kb)):                     # only the last layer returns its group max/min
        last = li == len(kb) - 1
        Yn, bnn, grp_b = R.run_module(kb[li], before[-1][1], G, epoch, prev=before[-1][2], group=Kn, want_group=last,
                                      want_arg=last and keep, name="knn_b%d" % li)
        before.append((kb[li], Yn, bnn))
    # max over K of the activated features (layers.py:433): from group max/min of the raw output
    _, Yb, bnb = before[-1]
    amax = torch.empty((Q, Cb), dtype=f32, device=dev)
    with _Prof("group_select"):
        ops.group_select(grp_b["gmax"], grp_b["gmin"], bnb.scale, bnb.shift, amax, Q, Cb)
    W8 = _w2d(ka[0].conv.weight)
    U, _, _ = R.run(amax, Q, _cols(W8, 0, Cb), None, relu_in=False, name="knn_a0_node")                                    # max half (layers.py:435)
    Y8, bn8, _ = R.run(Yb, G, _cols(W8, Cb), ka[0].conv.bias.detach(), ka[0].norm, _bn_mom(ka[0].norm, epoch),
                       prev=bnb, addend=U, add_group=Kn, name="knn_a0")
    after = [(ka[0], Y8, bn8)]
    for li in range(1, len(ka)):
        last = li == len(ka) - 1
        Yn, bnn, grp_a = R.run_module(ka[li], after[-1][1], G, epoch, prev=after[-1][2], group=Kn, want_group=last,
                                      want_arg=last and keep, write_y=(not last) or keep, name="knn_a%d" % li)
        after.append((ka[li], Yn, bnn))
    bna = after[-1][2]
    ops.group_select(grp_a["gmax"], grp_a["gmin"], bna.scale, bna.shift, AGG[:, C1:], Q, C2)   # layers.py:438

    # ---- head (networks.py:143-154); mlp1/mlp2 are called WITHOUT epoch in the reference
    Y10, bn10, _ = R.run_module(net.mlp1, AGG, Q, relu_in=False, name="mlp1")
    Y11, bn11, _ = R.run_module(net.mlp2, Y10, Q, prev=bn10, name="mlp2")
    OUT, _, _ = R.run_module(net.mlp3, Y11, Q, prev=bn11, name="mlp3")
    with _Prof("head_finalize"):
        keypoints, sigmas = ops.head_finalize(OUT, cmean, opt.loss_sigma_lower_bound, Bp, M)

    kctx = dict(knn_i=knn_i)
    if keep:
        # head: AGG as the raw input of mlp1, then (module, pre-BN output, BNState) of mlp1..mlp3
        kctx.update(Kn=Kn, C1=C1, C2=C2, Cb=Cb, AGG=AGG, Z=Z, before=before, grp_b=grp_b, amax=amax, U=U,
                    after=after, grp_a=grp_a, coords=coords,
                    head=[(None, AGG, None), (net.mlp1, Y10, bn10), (net.mlp2, Y11, bn11), (net.mlp3, OUT, None)])
    return keypoints, sigmas, kctx


def detector_forward(net, x, sn, node, epoch=None, use_tc=True, keep=False):
    """RPN_Detector.forward (models/networks.py:75-162) on the fused plan.

    x (B,3,N), sn (B,S,N), node (B,3,M) CUDA f32 contiguous.  Returns
    (cluster_mean (B,3,M), keypoints (B,3,M), sigmas (B,M), ctx) -- ctx holds everything backward needs when
    keep=True."""
    opt = net.opt
    assert opt.k == 1, "only k=1 is supported (every shipped config; networks.py:91-92)"
    if keep and not net.training:
        raise NotImplementedError("gradients through eval-mode BatchNorm are not part of the hot path "
                                  "(the reference only back-propagates in train mode, keypoint_detector.py:170)")
    assert len(net.knnlayer_1.layers_before) >= 2 and len(net.knnlayer_1.layers_after) >= 2
    dev = x.device
    Bp, _, N = x.shape
    M = node.shape[2]
    S = opt.surface_normal_len if opt.surface_normal_len >= 1 else 0
    Kn = opt.node_knn_k_1
    P, Q = Bp * N, Bp * M
    R = LayerRunner(net.training, use_tc, dev)
    x = x.detach().contiguous(); node = node.detach().contiguous()
    snc = sn.detach().contiguous() if S else None

    # ---- grouping (som.query_topk + networks.py:87-108)
    with _Prof("som_assign", nbytes=4.0 * Bp * (4 * N + 3 * M)):
        min_idx, count = ops.som_assign(x, node)
    with _Prof("cluster_sort"):
        seg_off, perm, row_seg = ops.cluster_sort(min_idx, M)
    with _Prof("cluster_mean_decenter", nbytes=4.0 * Bp * N * (3 + S + 8 + 1)):
        cmean, X0 = ops.cluster_mean_decenter(x, snc, seg_off, perm, M, ldx=8)

    # ---- first PointNet (3+S -> C1/2 -> C1/2 -> C1/2), networks.py:111-114
    fp = net.first_pointnet.layers
    H = fp[0].conv.weight.shape[0]
    Y0, bn0, _ = R.run_module(fp[0], X0, P, epoch, name="pn1.0")
    Y1, bn1, _ = R.run_module(fp[1], Y0, P, epoch, prev=bn0, name="pn1.1")
    F1, _, _ = R.run_module(fp[2], Y1, P, prev=bn1, name="pn1.2")
    # ---- pool 1 (index_max + gather * mask, networks.py:117-120)
    with _Prof("segmax1", nbytes=4.0 * P * H):
        pool1, arg1 = ops.segmax(F1, H, seg_off, perm, Bp, N, M, want_arg=keep)
    # ---- second PointNet on cat(first, scattered max) (networks.py:123-127): W [f; s] = Wa f + Wb s
    sp = net.second_pointnet.layers
    C1 = sp[0].conv.weight.shape[0]
    W3 = _w2d(sp[0].conv.weight)
    V, _, _ = R.run(pool1, Q, _cols(W3, H), None, relu_in=False, name="pn2.0_node")
    Y3, bn3, _ = R.run(F1, P, _cols(W3, 0, H), sp[0].conv.bias.detach(), sp[0].norm, _bn_mom(sp[0].norm, epoch),
                       relu_in=False, addend=V, add_index=row_seg, name="pn2.0")
    F2, _, _ = R.run_module(sp[1], Y3, P, prev=bn3, name="pn2.1")
    # ---- pool 2 -> first C1 columns of the head input (networks.py:130-133,143)
    C2 = net.knnlayer_1.layers_after[-1].conv.weight.shape[0]
    AGG = torch.empty((Q, C1 + C2), dtype=f32, device=dev)
    pool2 = AGG[:, :C1]
    with _Prof("segmax2", nbytes=4.0 * P * C1):
        _, arg2 = ops.segmax(F2, C1, seg_off, perm, Bp, N, M, out=pool2, want_arg=keep)

    keypoints, sigmas, kctx = _knn_head_forward(R, net, AGG, C1, cmean, Bp, M, Kn, epoch, keep)
    knn_i = kctx["knn_i"]

    ctx = None
    if keep:
        ctx = dict(kctx)
        ctx.update(Bp=Bp, N=N, M=M, S=S, H=H,
                   seg_off=seg_off, perm=perm, row_seg=row_seg, min_idx=min_idx, count=count, cmean=cmean,
                   X0=X0, pn1=[(fp[0], Y0, bn0), (fp[1], Y1, bn1), (fp[2], F1, None)], pool1=pool1, arg1=arg1, V=V,
                   Y3=Y3, bn3=bn3, F2=F2, arg2=arg2, use_tc=use_tc)
    aux = dict(min_idx=min_idx, count=count, perm=perm, seg_off=seg_off, knn_i=knn_i)
    return cmean, keypoints, sigmas, ctx, aux


class _Bwd:
    """Gradient bookkeeping of the backward plans and the per-layer steps they are written in."""

    def __init__(self, net, dev, use_tc):
        self.dev = dev
        self.use_tc = use_tc
        # opt.backward_precision: "3xtf32" (default, fp32-equivalent like the forward) or "tf32" -- the dgrad / wgrad GEMMs as
        # ONE TF32 MMA per MAC, the arithmetic PyTorch's default cuDNN path gives the reference's backward
        self.tf32_bwd = str(getattr(getattr(net, "opt", None), "backward_precision", "3xtf32")).lower() == "tf32"
        params = list(net.parameters())
        # usip_b200.optim.FlatAdam publishes a view of its flat gradient buffer on every parameter: accumulate straight
        # into it (autograd's own semantics for an existing .grad) and hand autograd nothing to add.  Without it (a
        # caller's own optimizer) the gradients are fresh tensors returned through autograd.
        self.direct = all(getattr(p, "_usip_flat_grad", None) is not None for p in params)
        if self.direct:
            for p in params:
                if p.grad is None or p.grad.data_ptr() != p._usip_flat_grad.data_ptr():   # module.zero_grad(set_to_none=True)
                    p._usip_flat_grad.zero_()
                    p.grad = p._usip_flat_grad
            self.grads = {p: p._usip_flat_grad for p in params}
        else:
            self.grads = {p: torch.zeros_like(p, memory_format=torch.contiguous_format) for p in params}

    def result(self, net):
        """What the autograd Function returns for the parameters."""
        if self.direct:
            return [None for _ in net.parameters()]
        return [self.grads[q] for q in net.parameters()]

    def g2d(self, w):
        g = self.grads[w]
        return g.view(g.shape[0], -1)

    def bn_bwd(self, G, Y, st, norm, name="bn_bwd"):
        """g_y [P,C] (new buffer) of a train-mode BN+ReLU layer from the gradient G of its output; writes g_gamma / g_beta."""
        P, C = G.shape
        with _Prof(name, nbytes=4.0 * P * C * 5):
            part = ops.bn_bwd_reduce(G, Y, st.scale, st.shift, st.mean, st.invstd, True)
            c1, c2 = ops.bn_bwd_finalize(part, P, self.grads[norm.weight], self.grads[norm.bias])
            return ops.bn_bwd_apply(G, Y, st.scale, st.shift, st.mean, st.invstd, c1, c2, True)

    def groupmax_select(self, Gout, grp, st, with_stats):
        """ops.groupmax_bwd_select of out = max_k relu(bn(y_k)) for the group outputs `grp` of LayerRunner.run."""
        return ops.groupmax_bwd_select(Gout, grp["gmax"], grp["gmin"], grp["amax"], grp["amin"], st.scale, st.shift, st.mean,
                                       st.invstd, with_stats)

    def groupmax_bn_bwd(self, Gout, Y, grp, st, norm, K):
        """g_y [Q*K, C] of a layer whose ONLY consumer is max_k relu(bn(y)) (layers.py:433,438; networks.py:572,700)."""
        G, C = Gout.shape[0] * K, Gout.shape[1]
        gz, arg, part = self.groupmax_select(Gout, grp, st, True)
        c1, c2 = ops.bn_bwd_finalize(part, G, self.grads[norm.weight], self.grads[norm.bias])
        with _Prof("groupmax_bwd_apply", nbytes=8.0 * G * C):
            return ops.groupmax_bwd_apply(Y, gz, arg, st.scale, st.mean, st.invstd, c1, c2, K)

    def wgrad(self, GY, X, gW, prev=None, name="wgrad"):
        """gW += GY^T act(X), act = the BN+ReLU of `prev` (BNState) or the identity."""
        P, (Cout, Cin) = GY.shape[0], gW.shape
        tc = self.use_tc and Cout % 4 == 0 and Cout >= 64 and Cin % 64 == 0 and P >= 4096
        with _Prof("%s[%dx%d->%d]" % (name, P, Cin, Cout), flops=2.0 * P * Cin * Cout,
                   precision="3xTF32 tcgen05" if tc else "fp32 SIMT"):
            ops.wgrad(GY, X, gW, None if prev is None else prev.scale, None if prev is None else prev.shift, prev is not None,
                      (4 if self.tf32_bwd else 1) if self.use_tc else 0)

    def dgrad(self, GY, W2d, name="dgrad"):
        """G_in[P,Cin] = GY[P,Cout] @ W2d[Cout,Cin] (the forward weight, used transposed by the layer kernel)."""
        P, (Cout, Cin) = GY.shape[0], W2d.shape
        out = torch.empty((P, Cin), dtype=f32, device=self.dev)
        prec = _precision_for(P, Cout, Cin, self.use_tc)
        ws, packed, pack_ent = _tc_workspace(W2d, P, Cout, Cin, 0, True, prec) if prec else (None, False, None)
        with _Prof("%s[%dx%d->%d]" % (name, P, Cout, Cin), flops=2.0 * P * Cin * Cout,
                   precision="3xTF32 tcgen05" if prec else "fp32 SIMT"):
            ops.layer_fwd(GY, W2d, None, P, Cout, Cin, Y=out, precision=prec, w_transposed=True, tc_ws=ws, tc_packed=packed,
                          debug_flags=8 if (self.tf32_bwd and prec) else 0, pack_entry=pack_ent)
        return out

    def layer_bwd(self, GY, m, src, name, bn_name):
        """Backward of the conv1x1 layer m from GY, the gradient of its pre-BN output rows.  Accumulates m's weight gradient
        (and its bias gradient when no BN follows m: a bias in front of a train-mode BN has exactly zero gradient) and
        returns the gradient of what m read.  src = (module, Y, BNState) of the layer m reads through BN+ReLU: the result is
        the gradient of that layer's pre-BN output Y.  src = (None, X, None): X is m's raw input and the result its gradient."""
        pm, X, st = src
        W = _w2d(m.conv.weight)
        self.wgrad(GY, X, self.g2d(m.conv.weight), prev=st, name="wgrad_" + name)
        if getattr(m, "norm", None) is None:
            ops.colsum(GY, self.grads[m.conv.bias])
        G_in = self.dgrad(GY, W, name="dgrad_" + name)
        if st is None:
            return G_in
        return self.bn_bwd(G_in, X, st, pm.norm, name=bn_name)


def _knn_head_backward(bw, net, ctx, g_kp, g_sig):
    """Backward of _knn_head_forward: parameter gradients of mlp1/2/3 and knnlayer_1 are accumulated into bw.grads; returns
    the gradient [Q, C1] of the per-node feature that entered AGG[:, :C1] (head path + kNN path)."""
    dev = bw.dev
    Bp, M = ctx["Bp"], ctx["M"]
    Kn, C1, Cb = ctx["Kn"], ctx["C1"], ctx["Cb"]
    Q = Bp * M
    before, after, head = ctx["before"], ctx["after"], ctx["head"]
    g_kp = None if g_kp is None else g_kp.contiguous()
    g_sig = None if g_sig is None else g_sig.contiguous()
    # ---- head (networks.py:143-154): mlp3 -> mlp2 -> mlp1
    GY = ops.head_bwd(g_kp, g_sig, head[-1][1], Bp, M)
    for li in range(len(head) - 1, 0, -1):
        GY = bw.layer_bwd(GY, head[li][0], head[li - 1], "mlp%d" % li, "bn_bwd")
    G_pool2, G_feat = GY[:, :C1], GY[:, C1:]                               # GY: gradient of AGG [Q, C1+C2]

    # ---- kNN fusion, layers_after (layers.py:435-438), last -> 1
    ka_last, Ya_last, bna_last = after[-1]
    GYa = bw.groupmax_bn_bwd(G_feat, Ya_last, ctx["grp_a"], bna_last, ka_last.norm, Kn)
    for li in range(len(after) - 1, 0, -1):
        GYa = bw.layer_bwd(GYa, after[li][0], after[li - 1], "knn_a%d" % li, "bn_bwd_knn_a%d" % (li - 1))
    # ka[0]: Y8 = a7 Wnb^T + U[row/K] + b, U = amax Wmax^T
    ka0, kb0 = after[0][0], before[0][0]
    W8, gW8 = _w2d(ka0.conv.weight), bw.g2d(ka0.conv.weight)
    kb_last, Yb_last, bnb_last = before[-1]
    bw.wgrad(GYa, Yb_last, gW8[:, Cb:], prev=bnb_last, name="wgrad_knn_a0")
    G_a7 = bw.dgrad(GYa, _cols(W8, Cb), name="dgrad_knn_a0")                 # [G, Cb]
    G_U = ops.group_sum(GYa, Kn)                                            # [Q, C2]
    del GYa
    bw.wgrad(G_U, ctx["amax"], gW8[:, :Cb], name="wgrad_knn_a0_node")
    G_amax = bw.dgrad(G_U, _cols(W8, 0, Cb), name="dgrad_knn_a0_node")        # [Q, Cb]
    # max path joins the dense gradient of a7 at the arg rows (ReLU mask is applied by bn_bwd below)
    _, arg7, _ = bw.groupmax_select(G_amax, ctx["grp_b"], bnb_last, False)
    ops.groupmax_scatter_add(G_a7, G_amax, arg7, Kn)
    # ---- layers_before, last -> 1
    GYb = bw.bn_bwd(G_a7, Yb_last, bnb_last, kb_last.norm, name="bn_bwd_knn_b%d" % (len(before) - 1))
    del G_a7
    for li in range(len(before) - 1, 0, -1):
        GYb = bw.layer_bwd(GYb, before[li][0], before[li - 1], "knn_b%d" % li, "bn_bwd_knn_b%d" % (li - 1))
    # kb[0] = knn_combine: Y5 = Z[nbr] + Wxyz*delta + b, Z = pool2 Wf^T
    W5, gW5 = _w2d(kb0.conv.weight), bw.g2d(kb0.conv.weight)
    G_Z = torch.zeros((Q, Cb), dtype=f32, device=dev)
    with _Prof("knn_combine_bwd"):
        ops.knn_combine_bwd(GYb, ctx["coords"], ctx["knn_i"], G_Z, gW5, Bp, M, Kn)
    del GYb
    bw.wgrad(G_Z, ctx["AGG"][:, :C1], gW5[:, 3:], name="wgrad_knn_b0_node")
    G_pool2_tot = bw.dgrad(G_Z, _cols(W5, 3), name="dgrad_knn_b0_node")       # [Q, C1]
    G_pool2_tot += G_pool2                                                 # tiny [Q,C1] plumbing add
    return G_pool2_tot


def detector_backward(net, ctx, g_kp, g_sig):
    """Backward of detector_forward.  Returns the gradients of net.parameters() in order."""
    dev = ctx["cmean"].device
    Bp, N, M = ctx["Bp"], ctx["N"], ctx["M"]
    H, C1 = ctx["H"], ctx["C1"]
    P = Bp * N
    bw = _Bwd(net, dev, ctx["use_tc"])
    sp, pn1 = net.second_pointnet.layers, ctx["pn1"]

    G_pool2_tot = _knn_head_backward(bw, net, ctx, g_kp, g_sig)

    # ---- pool 2 un-pool (index_max gather backward), second PointNet
    G_F2 = torch.zeros((P, C1), dtype=f32, device=dev)
    ops.unpool_scatter(G_F2, G_pool2_tot, ctx["arg2"], accumulate=False)
    GY3 = bw.layer_bwd(G_F2, sp[1], (sp[0], ctx["Y3"], ctx["bn3"]), "pn2.1", "bn_bwd_pn2.0")
    del G_F2
    W3 = _w2d(sp[0].conv.weight)
    gW3 = bw.g2d(sp[0].conv.weight)
    bw.wgrad(GY3, pn1[-1][1], gW3[:, :H], name="wgrad_pn2.0")
    G_F1 = bw.dgrad(GY3, _cols(W3, 0, H), name="dgrad_pn2.0")                  # [P, H]
    G_V = ops.seg_sum(GY3, ctx["seg_off"], Bp, N, M)                         # [Q, C1]
    del GY3
    bw.wgrad(G_V, ctx["pool1"], gW3[:, H:], name="wgrad_pn2.0_node")
    G_pool1 = bw.dgrad(G_V, _cols(W3, H), name="dgrad_pn2.0_node")             # [Q, H]
    ops.unpool_scatter(G_F1, G_pool1, ctx["arg1"], accumulate=True)
    # ---- first PointNet, last -> 1, then the weight gradient of layer 0 (the points carry none)
    GY = G_F1
    del G_F1
    for li in range(len(pn1) - 1, 0, -1):
        GY = bw.layer_bwd(GY, pn1[li][0], pn1[li - 1], "pn1.%d" % li, "bn_bwd_pn1.%d" % (li - 1))
    bw.wgrad(GY, ctx["X0"], bw.g2d(pn1[0][0].conv.weight), name="wgrad_pn1.0")
    # conv biases in front of a train-mode BatchNorm receive exactly zero gradient (BN removes the mean); they
    # stay zero-initialised in bw.grads.
    return bw.result(net)


def _group_net_forward(R, net, rows, Bp, M, K, keep, out=None):
    """The grouped PointNet shared by DescriptorLiteOld (networks.py:375-381) and the ablation detectors
    RPN_Detector_KNN / RPN_Detector_Ball (networks.py:567-572, 695-700):
        conv1 -> conv2 -> conv3 -> max_k -> conv4 on cat(y, broadcast max) -> conv5 -> max_k
    on point-major rows [Bp*M*K, ld] of the gathered, decentred groups.  conv1..conv4 carry BN+ReLU; conv5 is linear in the
    descriptor (the raw group max is returned) and BN+ReLU in the detectors (max_k relu(bn(.)) is written to `out`).
    The reference calls these convolutions WITHOUT epoch: their BN momentum never decays."""
    dev = rows.device
    G, Q = Bp * M * K, Bp * M
    c1, c2, c3, c4, c5 = net.conv1, net.conv2, net.conv3, net.conv4, net.conv5
    D = c3.conv.weight.shape[0]
    Y1, bn1, _ = R.run_module(c1, rows, G, name="grp.conv1")
    Y2, bn2, _ = R.run_module(c2, Y1, G, prev=bn1, name="grp.conv2")
    Y3, bn3, grp3 = R.run_module(c3, Y2, G, prev=bn2, group=K, want_group=True, want_arg=keep, name="grp.conv3")
    amax = torch.empty((Q, D), dtype=f32, device=dev)
    ops.group_select(grp3["gmax"], grp3["gmin"], bn3.scale, bn3.shift, amax, Q, D)          # y_first_max (networks.py:377)
    W4 = _w2d(c4.conv.weight)
    U, _, _ = R.run(amax, Q, _cols(W4, D), None, relu_in=False, name="grp.conv4_node")        # cat(y_first, max): max is LAST
    Y4, bn4, _ = R.run(Y3, G, _cols(W4, 0, D), c4.conv.bias.detach(), c4.norm, c4.norm.momentum, prev=bn3, addend=U,
                       add_group=K, name="grp.conv4")
    last_bn = getattr(c5, "norm", None) is not None
    Y5, bn5, grp5 = R.run_module(c5, Y4, G, prev=bn4, group=K, want_group=True, want_arg=keep, write_y=last_bn and keep,
                                 name="grp.conv5")
    result = grp5["gmax"]
    if last_bn:
        C5 = c5.conv.weight.shape[0]
        if out is None:
            out = torch.empty((Q, C5), dtype=f32, device=dev)
        ops.group_select(grp5["gmax"], grp5["gmin"], bn5.scale, bn5.shift, out, Q, C5)
        result = out
    gctx = dict(D=D)
    if keep:
        gctx.update(Bp=Bp, M=M, K=K, rows=rows, layers=[(c1, Y1, bn1), (c2, Y2, bn2), (c3, Y3, bn3), (c4, Y4, bn4)],
                    grp3=grp3, amax=amax, Y5=Y5, bn5=bn5, grp5=grp5)
    return result, gctx


ABLATION_K = 64             # networks.py:554, 680: `k = 64` is hard-coded in both ablation detectors
ABLATION_RADIUS = 2.0       # networks.py:681


def ablation_forward(net, x, sn, node, epoch=None, use_tc=True, keep=False, mode="knn"):
    """RPN_Detector_KNN.forward (models/networks.py:545-608, mode="knn") / RPN_Detector_Ball.forward (:671-738, mode="ball")
    on the fused plan: group the points around the GIVEN nodes (64 nearest points / first 64 points within radius 2, both
    without the (B,M,N) distance matrix), the grouped PointNet conv1..conv5 with two max-pools over the group, then the same
    node-level kNN fusion module and head as RPN_Detector -- on the nodes themselves, which are also returned in place of the
    recomputed cluster means.  Returns (node, keypoints, sigmas, ctx)."""
    opt = net.opt
    if keep and not net.training:
        raise NotImplementedError("gradients through eval-mode BatchNorm are not part of the hot path")
    dev = x.device
    Bp, _, N = x.shape
    M = node.shape[2]
    S = opt.surface_normal_len if opt.surface_normal_len >= 1 else 0
    Kn = opt.node_knn_k_1
    K = ABLATION_K
    Q = Bp * M
    R = LayerRunner(net.training, use_tc, dev)
    x = x.detach().contiguous(); node = node.detach().contiguous()
    snc = sn.detach().contiguous() if S else None
    with _Prof("group_%s" % mode):
        if mode == "knn":
            _, _, rows = ops.knn_group(x, snc, node, K, want_group=False, rows_ld=8)
        else:
            _, _, rows = ops.ball_group(x, snc, node, ABLATION_RADIUS, K, want_group=False, rows_ld=8)
    C1 = net.conv5.conv.weight.shape[0]
    C2 = net.knnlayer_1.layers_after[-1].conv.weight.shape[0]
    AGG = torch.empty((Q, C1 + C2), dtype=f32, device=dev)
    _, gctx = _group_net_forward(R, net, rows, Bp, M, K, keep, out=AGG[:, :C1])      # second_pn_out_max (networks.py:572)
    keypoints, sigmas, kctx = _knn_head_forward(R, net, AGG, C1, node, Bp, M, Kn, epoch, keep)
    ctx = None
    if keep:
        ctx = dict(kctx)                                        # (both plans keep an "amax": the grouped PointNet's state is nested)
        ctx.update(Bp=Bp, M=M, use_tc=use_tc, group_net=gctx)
    return node, keypoints, sigmas, ctx


def ablation_backward(net, ctx, g_kp, g_sig):
    """Backward of ablation_forward: gradients of net.parameters() in order (points and nodes carry none)."""
    dev = ctx["AGG"].device
    gctx = ctx["group_net"]
    bw = _Bwd(net, dev, ctx["use_tc"])
    G_pool = _knn_head_backward(bw, net, ctx, g_kp, g_sig)                  # gradient of max_k relu(bn5(conv5)) [Q, C1]
    GY5 = bw.groupmax_bn_bwd(G_pool, gctx["Y5"], gctx["grp5"], gctx["bn5"], net.conv5.norm, gctx["K"])
    _group_net_backward(bw, net, gctx, GY5)
    return bw.result(net)


def descriptor_forward(net, x, sn, keypoints, epoch, permute_idx, use_tc=True, keep=False):
    """DescriptorLiteOld.forward (models/networks.py:333-385) on the fused plan.
    Returns (descriptor (B,C,M), x_features (B,3+S,M,K), ctx) -- ctx holds what descriptor_backward needs (keep=True)."""
    opt = net.opt
    dev = x.device
    if keep and not net.training:
        raise NotImplementedError("gradients through eval-mode BatchNorm are not part of the hot path "
                                  "(the reference only back-propagates in train mode, keypoint_descriptor.py:138)")
    Bp, _, N = x.shape
    M = keypoints.shape[2]
    K = opt.ball_nsamples
    S = opt.surface_normal_len if opt.surface_normal_len > 0 else 0
    R = LayerRunner(net.training, use_tc, dev)
    # permute the points on the host-drawn permutation: the ball query keeps the FIRST K hits in index order
    x = x.detach()[:, :, permute_idx].contiguous()
    snp = sn.detach()[:, :, permute_idx].contiguous() if S else None
    kp = keypoints.detach().contiguous()
    with _Prof("ball_group", nbytes=4.0 * Bp * (N * (3 + S) + 3 * M + M * K + (3 + S) * M * K)):
        idx, feats, rows = ops.ball_group(x, snp, kp, float(opt.ball_radius), K, want_group=True, rows_ld=8)
    gmax5, gctx = _group_net_forward(R, net, rows, Bp, M, K, keep, out=None)
    desc = ops.l2norm_to_bcm(gmax5, Bp, M)
    ctx = None
    if keep:
        ctx = dict(gctx)
        ctx.update(use_tc=use_tc)
    return desc, feats, ctx


def _group_net_backward(bw, net, ctx, GY5):
    """Backward of _group_net_forward from GY5 [G, C5], the gradient of conv5's raw output rows (parameter gradients are
    accumulated into bw.grads; points / centres carry no gradient)."""
    K, D = ctx["K"], ctx["D"]
    L = ctx["layers"]                                                      # (conv_i, Y_i, bn_i), i = 1..4
    c3, c4, bn3 = net.conv3, net.conv4, L[2][2]
    GY4 = bw.layer_bwd(GY5, net.conv5, L[3], "grp.conv5", "bn_bwd_grp.conv4")
    # ---- conv4 on cat(y_first, broadcast max): Y4 = a3 WA^T + U[row/K] + b,  U = amax WB^T
    W4 = _w2d(c4.conv.weight)
    gW4 = bw.g2d(c4.conv.weight)
    bw.wgrad(GY4, L[2][1], gW4[:, :D], prev=bn3, name="wgrad_grp.conv4")
    G_a3 = bw.dgrad(GY4, _cols(W4, 0, D), name="dgrad_grp.conv4")                   # [G, D]
    G_U = ops.group_sum(GY4, K)                                                     # [Q, C4]
    del GY4
    bw.wgrad(G_U, ctx["amax"], gW4[:, D:], name="wgrad_grp.conv4_node")
    G_amax = bw.dgrad(G_U, _cols(W4, D), name="dgrad_grp.conv4_node")               # [Q, D]
    # the max path joins the dense gradient of a3 at the arg rows (the ReLU mask is applied by bn_bwd below)
    _, arg3, _ = bw.groupmax_select(G_amax, ctx["grp3"], bn3, False)
    ops.groupmax_scatter_add(G_a3, G_amax, arg3, K)
    # ---- conv3, conv2, then the weight gradient of conv1
    GY = bw.bn_bwd(G_a3, L[2][1], bn3, c3.norm, name="bn_bwd_grp.conv3")
    del G_a3
    for li in (2, 1):
        GY = bw.layer_bwd(GY, L[li][0], L[li - 1], "grp.conv%d" % (li + 1), "bn_bwd_grp.conv%d" % li)
    bw.wgrad(GY, ctx["rows"], bw.g2d(net.conv1.conv.weight), name="wgrad_grp.conv1")


def descriptor_backward(net, ctx, g_desc):
    """Backward of descriptor_forward (points / keypoints carry no gradient): gradients of net.parameters() in order.

    desc = l2norm(max_k conv5(a4)),  a4 = relu(bn4(a3 WA^T + (amax WB^T)[row/K])),  amax = max_k a3,
    a3 = relu(bn3(conv3(a2))), a2 = relu(bn2(conv2(a1))), a1 = relu(bn1(conv1(rows)))      (networks.py:375-383)."""
    dev = g_desc.device
    Bp, M, K, D = ctx["Bp"], ctx["M"], ctx["K"], ctx["D"]
    bw = _Bwd(net, dev, ctx["use_tc"])
    grp5 = ctx["grp5"]
    # ---- l2 normalisation and the max over the ball (conv5 is linear: the max of the raw output routes to its arg row)
    G_y = ops.l2norm_bwd(g_desc, grp5["gmax"], Bp, M)                       # [Q, D]
    GY5 = torch.zeros((Bp * M * K, D), dtype=f32, device=dev)
    ops.groupmax_scatter_add(GY5, G_y, grp5["amax"], K)
    _group_net_backward(bw, net, ctx, GY5)
    # conv1..conv4 biases sit in front of a train-mode BatchNorm: exactly zero gradient (left zero-initialised)
    return bw.result(net)
