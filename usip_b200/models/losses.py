"""Host-side mirror of the hot-path losses of models/losses.py (same class names / signatures / returns):

  ChamferLoss_Brute            losses.py:44-99    probabilistic chamfer (sigma branch) + plain branch
  KeypointOnPCLoss             losses.py:102-116  (point_to_point -> SingleSideChamferLoss_Brute)
  SingleSideChamferLoss_Brute  losses.py:119-143

The (B,3,M,N) / (B,M,N) temporaries of the reference are never built: one tiled pairwise-L2 arg-min kernel
(usip_pairwise_min_f32) serves all three, the reductions and the backward passes are small fused kernels.
"""
import torch
import torch.nn as nn

from usip_b200 import ops


# ---- functional cores: used by the autograd Functions below and by the autograd-free train step of ModelDetector ----
def chamfer_prob_fwd(src, dst, sig_src, sig_dst):
    """ChamferLoss_Brute sigma branch (losses.py:79-97): -> (out3 = [loss, pure, weighted], saved), where saved are the
    leading arguments of ops.chamfer_prob_bwd."""
    d_sd, i_sd = ops.pairwise_min(src, dst)
    d_ds, i_ds = ops.pairwise_min(dst, src)
    out3 = ops.chamfer_prob_reduce(d_sd, i_sd, d_ds, i_ds, sig_src, sig_dst)
    return out3, (src, dst, sig_src, sig_dst, d_sd, i_sd, d_ds, i_ds)


def point_on_surface_fwd(kp, pc, sn):
    _, arg = ops.pairwise_min(kp, pc)                       # nearest cloud point of every keypoint (not differentiated)
    return ops.point_on_surface(kp, pc, sn, arg), arg


class _PairMinFn(torch.autograd.Function):
    """min_j ||a_i - b_j|| (B,Ma); differentiable w.r.t. both point sets (sub-gradient 0 at d == 0)."""

    @staticmethod
    def forward(ctx, a, b):
        a = a.contiguous(); b = b.contiguous()
        from usip_b200 import engine
        with engine._Prof("pairwise_min[%dx%dx%d]" % (a.shape[0], a.shape[2], b.shape[2])):
            d, arg = ops.pairwise_min(a, b)
        ctx.save_for_backward(a, b, d, arg)
        return d

    @staticmethod
    def backward(ctx, g):
        a, b, d, arg = ctx.saved_tensors
        ga, gb = ops.pairwise_min_bwd(a, b, d, arg, g, want_b=ctx.needs_input_grad[1])
        return (ga if ctx.needs_input_grad[0] else None), gb


class _ChamferProbFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, dst, sig_src, sig_dst):
        src = src.contiguous(); dst = dst.contiguous()
        sig_src = sig_src.contiguous(); sig_dst = sig_dst.contiguous()
        from usip_b200 import engine
        with engine._Prof("chamfer_prob"):
            out3, saved = chamfer_prob_fwd(src, dst, sig_src, sig_dst)
        ctx.save_for_backward(*saved)
        loss, pure, weighted = out3[0], out3[1], out3[2]
        ctx.mark_non_differentiable(pure, weighted)
        return loss, pure, weighted

    @staticmethod
    def backward(ctx, g_loss, g_pure, g_weighted):
        return ops.chamfer_prob_bwd(*ctx.saved_tensors, g_loss.reshape(1).to(torch.float32).contiguous())


class _TransformFn(torch.autograd.Function):
    """R @ kp * scale + shift (keypoint_detector.py:182-184); gradient only w.r.t. kp."""

    @staticmethod
    def forward(ctx, kp, R, scale, shift):
        kp = kp.contiguous(); R = R.contiguous()
        scale = scale.reshape(-1).contiguous(); shift = shift.reshape(shift.shape[0], 3).contiguous()
        ctx.save_for_backward(R, scale)
        return ops.transform_points(kp, R, scale, shift)

    @staticmethod
    def backward(ctx, g):
        R, scale = ctx.saved_tensors
        return ops.transform_points_bwd(g, R, scale), None, None, None


class _MeanScaleFn(torch.autograd.Function):
    """mean(d) * alpha (keypoint_detector.py:193-197)."""

    @staticmethod
    def forward(ctx, d, alpha):
        ctx.alpha = alpha; ctx.n = d.numel(); ctx.shape = d.shape
        return ops.mean_scale(d.contiguous(), alpha)[0]

    @staticmethod
    def backward(ctx, g):
        return (g * (ctx.alpha / ctx.n)).expand(ctx.shape), None


def transform_keypoints(kp, R, scale, shift):
    return _TransformFn.apply(kp, R, scale, shift)


def mean_scale(d, alpha):
    return _MeanScaleFn.apply(d, float(alpha))


class ChamferLoss_Brute(nn.Module):
    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        self.dimension = 3

    def forward(self, pc_src_input, pc_dst_input, sigma_src=None, sigma_dst=None):
        """pc_src (B,3,M), pc_dst (B,3,N), sigma (B,M)/(B,N) -> (loss, chamfer_pure, chamfer_weighted);
        without sigmas: un-reduced (B,M) tensors (losses.py:68-78)."""
        if sigma_src is None or sigma_dst is None:
            forward_loss = _PairMinFn.apply(pc_src_input, pc_dst_input)
            backward_loss = _PairMinFn.apply(pc_dst_input, pc_src_input)
            chamfer_pure = forward_loss + backward_loss
            return forward_loss + backward_loss, chamfer_pure, chamfer_pure
        return _ChamferProbFn.apply(pc_src_input, pc_dst_input, sigma_src, sigma_dst)


class SingleSideChamferLoss_Brute(nn.Module):
    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        self.dimension = 3

    def forward(self, pc_src_input, pc_dst_input):
        """(B,3,M), (B,3,N) -> (B,M) min distances (losses.py:125-143)."""
        return _PairMinFn.apply(pc_src_input, pc_dst_input)


class _PointOnSurfaceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, keypoint, pc, sn):
        kp = keypoint.contiguous(); pc = pc.contiguous(); sn = sn.contiguous()
        B, _, M = kp.shape
        loss, arg = point_on_surface_fwd(kp, pc, sn)
        ctx.save_for_backward(kp, pc, sn, arg)
        return loss.view(B, M, 1, 1)                            # the reference returns the (B,M,1,1) matmul result

    @staticmethod
    def backward(ctx, g):
        kp, pc, sn, arg = ctx.saved_tensors
        return ops.point_on_surface(kp, pc, sn, arg, g.reshape(arg.shape).contiguous().float()), None, None


class PointOnSurfaceLoss(nn.Module):
    """models/losses.py:146-183 ('point_to_plane'): squared cosine between the surface normal of the nearest cloud point
    and the direction from that point to the keypoint; gradient w.r.t. the keypoint only."""

    def __init__(self, opt):
        super().__init__()
        self.opt = opt

    def forward(self, keypoint, pc, sn):
        return _PointOnSurfaceFn.apply(keypoint, pc.detach(), sn.detach())


class KeypointOnPCLoss(nn.Module):
    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        self.single_side_chamfer = SingleSideChamferLoss_Brute(opt)
        self.keypoint_on_surface = PointOnSurfaceLoss(opt)

    def forward(self, keypoint, pc, sn=None):
        if sn is None:
            return self.single_side_chamfer(keypoint, pc)
        return self.keypoint_on_surface(keypoint, pc, sn)


class _DescTripletFn(torch.autograd.Function):
    """loss (B,M), active (B) of DescPairScanLoss; backward through the two descriptor-space nearest neighbours."""

    @staticmethod
    def forward(ctx, anc, pos, neg, sigmas, gamma, sigma_max):
        a = anc.contiguous(); p_ = pos.contiguous(); n_ = neg.contiguous(); sg = sigmas.contiguous().float()
        dpos, ipos = ops.desc_pairmin(a, p_)
        dneg, ineg = ops.desc_pairmin(a, n_)
        loss, active = ops.desc_triplet(dpos, dneg, sg, gamma, sigma_max)
        ctx.save_for_backward(a, p_, n_, sg, dpos, ipos, dneg, ineg)
        ctx.gamma, ctx.sigma_max = float(gamma), float(sigma_max)
        ctx.mark_non_differentiable(active)
        return loss, active

    @staticmethod
    def backward(ctx, g_loss, g_active):
        a, p_, n_, sg, dpos, ipos, dneg, ineg = ctx.saved_tensors
        g_a, g_p, g_n = ops.desc_triplet_bwd(a, p_, n_, dpos, ipos, dneg, ineg, sg, ctx.gamma, ctx.sigma_max,
                                             g_loss.contiguous().float())
        return g_a, g_p, g_n, None, None, None


class DescPairScanLoss(nn.Module):
    """Triplet loss over scan pairs (models/losses.py:190-237): for every anchor keypoint the closest descriptor in
    the positive and in the negative scan (two fused C-dimensional pairwise-min kernels instead of two (B,C,M,M)
    difference tensors), sigma-derived (detached) weights; backward through the matched pairs (SURVEY 8 f-1)."""

    def __init__(self, opt):
        super().__init__()
        self.opt = opt

    def forward(self, anc_descriptors, pos_descriptors, neg_descriptors, anc_sigmas):
        return _DescTripletFn.apply(anc_descriptors, pos_descriptors, neg_descriptors, anc_sigmas.detach(),
                                    self.opt.triple_loss_gamma, self.opt.sigma_max)
