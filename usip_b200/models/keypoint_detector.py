"""`ModelDetector` -- same API surface as models/keypoint_detector.py:15-365 (constructor on `opt`,
set_input / forward / forward_siamese / optimize / test_model / freeze_model / run_model /
run_model_siamese / get_current_errors / save_network / update_learning_rate and the public attributes
callers read), on top of the fused B200 plan.

Multi-GPU: the reference wraps the detector in nn.DataParallel (keypoint_detector.py:35-37).  Here the unit is
one process per GPU (torch.distributed, NCCL): every rank runs the same step on its own pairs, BatchNorm
statistics stay per rank (the per-replica semantics DataParallel already has) and the only exchange is one
all-reduce of a flat fp32 gradient buffer (`enable_data_parallel()`), launched by `optimize()`.
"""
import os
from collections import OrderedDict

import torch

from usip_b200 import _lib, engine, ops
from usip_b200.optim import FlatAdam

from . import losses, networks
from ._common import random_point_dropout


class ModelDetector():
    def __init__(self, opt):
        self.opt = opt
        if opt.scene == 'indoor':
            self.detector = networks.RPN_DetectorLite(opt)      # keypoint_detector.py:19-22
        else:
            self.detector = networks.RPN_Detector(opt)
        self.chamfer_criteria = losses.ChamferLoss_Brute(opt)
        self.keypoint_on_pc_criteria = losses.KeypointOnPCLoss(opt)

        if opt.gpu_ids[0] < 0:
            raise RuntimeError("usip_b200.ModelDetector needs a CUDA device (opt.gpu_ids[0] >= 0): there is no CPU path")
        self.detector = self.detector.to(self.opt.device)

        self.old_lr_detector = self.opt.lr
        # Adam(lr, betas=(0.9, 0.999), weight_decay=0) as in keypoint_detector.py:42-45, as ONE kernel over flat buffers
        self.optimizer_detector = FlatAdam(self.detector.parameters(), lr=self.old_lr_detector, betas=(0.9, 0.999),
                                           weight_decay=0)
        self._dp = None
        self.use_cuda_graph = bool(getattr(opt, "use_cuda_graph", True)) and not os.environ.get("USIP_NO_TRAIN_GRAPH")
        self._train_graph_key = None

        dev = self.opt.device
        B, N, M = self.opt.batch_size, self.opt.input_pc_num, self.opt.node_num
        # place holders, same names as the reference (keypoint_detector.py:51-97)
        self.src_pc = torch.empty(B, 3, N, device=dev).uniform_()
        self.src_sn = torch.empty(B, 3, N, device=dev).uniform_()
        self.src_label = torch.ones(B, dtype=torch.long, device=dev)
        self.src_node = torch.empty(B, 3, M, device=dev)
        self.dst_pc = torch.empty(B, 3, N, device=dev).uniform_()
        self.dst_sn = torch.empty(B, 3, N, device=dev).uniform_()
        self.dst_label = torch.ones(B, dtype=torch.long, device=dev)
        self.dst_node = torch.empty(B, 3, M, device=dev)
        self.src_R_dst = torch.zeros((B, 3, 3), dtype=torch.float32, device=dev)
        self.src_scale_dst = torch.zeros((B, 1), dtype=torch.float32, device=dev)
        self.src_shift_dst = torch.zeros((B, 3, 1), dtype=torch.float32, device=dev)
        z = lambda: torch.tensor([0], dtype=torch.float32, requires_grad=False, device=dev)
        self.test_chamfer_average = z(); self.test_loss_average = z(); self.test_keypoint_on_pc_average = z()
        self.chamfer_pure = z(); self.test_chamfer_pure_average = z()
        self.chamfer_weighted = z(); self.test_chamfer_weighted_average = z()

    # ------------------------------------------------------------------ data parallel (one process / GPU)
    def enable_data_parallel(self, process_group=None):
        """Switch on the gradient all-reduce.  Call after torch.distributed.init_process_group."""
        from usip_b200.dp import FlatGradAllReduce
        self._dp = FlatGradAllReduce(self.optimizer_detector, process_group, buffers=list(self.detector.buffers()))
        self._train_graph_key = None

    def _allreduce_grads(self):
        if self._dp is not None:
            self._dp.allreduce_mean()

    def release_cuda_graphs(self):
        """Drop the captured step graphs (they are re-captured on demand).  A graph that holds an NCCL all-reduce must be
        destroyed BEFORE its communicator: call this (or usip_b200.dp.shutdown) ahead of destroy_process_group()."""
        for k in ("_tgraph", "_tgraph_in", "_tgraph_out", "_graph", "_graph_in", "_graph_out"):
            self.__dict__.pop(k, None)
        if self._train_graph_key != "failed":
            self._train_graph_key = None
        if hasattr(self, "_graph_key"):
            self._graph_key = None

    # ------------------------------------------------------------------ reference API
    _INPUT_FIELDS = ("src_pc", "src_sn", "src_node", "dst_pc", "dst_sn", "dst_node", "src_R_dst", "src_scale_dst", "src_shift_dst")

    def set_input(self, src_pc, src_sn, src_node, dst_pc, dst_sn, dst_node, src_R_dst, src_scale_dst, src_shift_dst):
        """keypoint_detector.py:120-134.  If the same host tensors were staged by prefetch_input(), the staged device
        copies are adopted with a stream-side wait instead of nine copies and a host synchronisation."""
        args = (src_pc, src_sn, src_node, dst_pc, dst_sn, dst_node, src_R_dst, src_scale_dst, src_shift_dst)
        st = getattr(self, "_staged", None)
        if st is not None and len(st[0]) == len(args) and all(a is b for a, b in zip(st[0], args)):
            cur = torch.cuda.current_stream()
            cur.wait_event(st[2])
            for k, v in zip(self._INPUT_FIELDS, st[1]):
                v.record_stream(cur)                                  # allocated on the copy stream, consumed here
                setattr(self, k, v)
            self._staged = None
            return
        dev = self.opt.device
        for k, a in zip(self._INPUT_FIELDS, args):
            setattr(self, k, a.float().to(dev, non_blocking=True).detach())
        torch.cuda.synchronize()                                  # keypoint_detector.py:134

    def prefetch_input(self, *args):
        """Not in the reference: stage the NEXT batch (same nine tensors as set_input, ideally pinned) with asynchronous
        host-to-device copies on a dedicated stream, so that the transfer overlaps the step that is running.  The
        following set_input() with the same tensor objects adopts the staged copies."""
        dev = self.opt.device
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(self._copy_stream):
            staged = [a.float().to(dev, non_blocking=True).detach() for a in args]
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        self._staged = (tuple(args), staged, ev)

    def forward(self, pc, sn, node, is_train=False, epoch=None):
        with torch.cuda.device(pc.get_device()):
            return self.detector(pc, sn, node, is_train, epoch)

    def forward_siamese(self, pc_tuple, sn_tuple, node_tuple, is_train=False, epoch=None):
        size_of_single_chunk = pc_tuple[0].size()[0]
        pc_cat = torch.cat(pc_tuple, dim=0)
        node_recomputed, keypoints, sigmas, descriptors = self.detector(pc_cat,
                                                                        torch.cat(sn_tuple, dim=0),
                                                                        torch.cat(node_tuple, dim=0), is_train, epoch)
        node_recomputed_tuple = torch.split(node_recomputed, split_size_or_sections=size_of_single_chunk, dim=0)
        keypoints_tuple = torch.split(keypoints, split_size_or_sections=size_of_single_chunk, dim=0)
        # both clouds / both keypoint sets as one tensor each: _losses() searches them in ONE nearest-neighbour call
        self._siamese_cat = (pc_tuple[0], pc_tuple[1], pc_cat, keypoints, keypoints_tuple[0], keypoints_tuple[1]) \
            if len(pc_tuple) == 2 else None
        sigmas_tuple = torch.split(sigmas, split_size_or_sections=size_of_single_chunk, dim=0)
        descriptors_tuple = (None, None)
        return node_recomputed_tuple, keypoints_tuple, sigmas_tuple, descriptors_tuple

    def _losses(self):
        # keypoint_detector.py:182-204 (and :219-241)
        self.src_keypoints_transformed = losses.transform_keypoints(self.src_keypoints, self.src_R_dst,
                                                                    self.src_scale_dst, self.src_shift_dst)
        self.loss_chamfer, self.chamfer_pure, self.chamfer_weighted = self.chamfer_criteria(
            self.src_keypoints_transformed, self.dst_keypoints, self.src_sigmas, self.dst_sigmas)
        cat = getattr(self, "_siamese_cat", None)
        if (self.opt.keypoint_on_pc_type == 'point_to_point' and not torch.is_grad_enabled() and cat is not None
                and cat[0] is self.src_pc and cat[1] is self.dst_pc and cat[4] is self.src_keypoints
                and cat[5] is self.dst_keypoints):
            # no autograd graph wanted (test_model / forward_loss): one search over the 2B clouds instead of two over B
            B = self.src_pc.shape[0]
            d, _ = ops.pairwise_min(cat[3].contiguous(), cat[2])
            self.loss_keypoint_on_pc_src = losses.mean_scale(d[:B], self.opt.keypoint_on_pc_alpha)
            self.loss_keypoint_on_pc_dst = losses.mean_scale(d[B:], self.opt.keypoint_on_pc_alpha)
        elif self.opt.keypoint_on_pc_type == 'point_to_point':
            self.loss_keypoint_on_pc_src = losses.mean_scale(
                self.keypoint_on_pc_criteria(self.src_keypoints, self.src_pc, None), self.opt.keypoint_on_pc_alpha)
            self.loss_keypoint_on_pc_dst = losses.mean_scale(
                self.keypoint_on_pc_criteria(self.dst_keypoints, self.dst_pc, None), self.opt.keypoint_on_pc_alpha)
        elif self.opt.keypoint_on_pc_type == 'point_to_plane':          # keypoint_detector.py:198-202
            self.loss_keypoint_on_pc_src = losses.mean_scale(
                self.keypoint_on_pc_criteria(self.src_keypoints, self.src_pc, self.src_sn), self.opt.keypoint_on_pc_alpha)
            self.loss_keypoint_on_pc_dst = losses.mean_scale(
                self.keypoint_on_pc_criteria(self.dst_keypoints, self.dst_pc, self.dst_sn), self.opt.keypoint_on_pc_alpha)
        else:
            raise NotImplementedError("keypoint_on_pc_type=%r" % self.opt.keypoint_on_pc_type)
        self.loss = self.loss_chamfer + self.loss_keypoint_on_pc_src + self.loss_keypoint_on_pc_dst

    def _run_siamese(self, is_train, epoch):
        (self.src_node_recomputed, self.dst_node_recomputed), \
        (self.src_keypoints, self.dst_keypoints), \
        (self.src_sigmas, self.dst_sigmas), \
        (self.src_descriptors, self.dst_descriptors) = self.forward_siamese((self.src_pc, self.dst_pc),
                                                                            (self.src_sn, self.dst_sn),
                                                                            (self.src_node, self.dst_node),
                                                                            is_train=is_train, epoch=epoch)

    def optimize(self, epoch=None):
        """keypoint_detector.py:158-207: (optional point dropout,) train-mode siamese forward, the three losses, backward,
        (gradient all-reduce when data parallel,) Adam.  With `opt.use_cuda_graph` (default) and no point dropout the
        whole step -- ~200 kernel launches, the NCCL all-reduce included -- is captured once per input shape and replayed
        as ONE CUDA graph; results land in the same public attributes."""
        with torch.cuda.device(self.src_pc.device):
            self.src_pc, self.src_sn, self.dst_pc, self.dst_sn = random_point_dropout(
                self.opt, self.src_pc, self.src_sn, self.dst_pc, self.dst_sn)
            self.detector.train()
            if self.use_cuda_graph and self.opt.random_pc_dropout_lower_limit >= 0.99 and self._train_graph_key != "failed":
                self._optimize_graph(epoch)
            else:
                self._optimize_eager(epoch)

    def _optimize_eager(self, epoch):
        """One train step.  The default is the autograd-free plan (`_train_step_direct`): this class owns the whole chain
        loss -> keypoints/sigmas -> network, so forward, the three losses, their gradients and engine.detector_backward are
        launched back to back on the current stream -- no autograd graph, no engine thread hand-off, capturable as one
        CUDA graph.  `opt.use_autograd_step = True` runs the reference's literal sequence (forward_siamese, criteria,
        loss.backward()) through the autograd Functions instead; both give the same gradients (tests)."""
        if getattr(self.opt, "use_autograd_step", False) or not isinstance(self.detector, networks._RPNBase):
            self._run_siamese(is_train=True, epoch=epoch)
            self.optimizer_detector.zero_grad()
            self._losses()
            self.loss.backward()
        else:
            self._train_step_direct(epoch)
        self._allreduce_grads()
        self.optimizer_detector.step()

    @torch.no_grad()
    def _train_step_direct(self, epoch):
        """keypoint_detector.py:170-205 without autograd: same kernels as the autograd Functions in losses.py / networks.py."""
        net, opt = self.detector, self.opt
        B = self.src_pc.shape[0]
        engine.prepack_weights(net)                     # all weight matrices the last Adam step made stale: one launch
        x = torch.cat((self.src_pc, self.dst_pc), dim=0)
        sn = torch.cat((self.src_sn, self.dst_sn), dim=0)
        node = torch.cat((self.src_node, self.dst_node), dim=0)
        cmean, kp, sig, ctx, aux = engine.detector_forward(net, x, sn, node, epoch, use_tc=net.use_tc, keep=True)
        net._last_aux = aux
        self.src_node_recomputed, self.dst_node_recomputed = cmean[:B], cmean[B:]
        self.src_keypoints, self.dst_keypoints = kp[:B], kp[B:]
        self.src_sigmas, self.dst_sigmas = sig[:B], sig[B:]
        self.src_descriptors = self.dst_descriptors = None
        self.optimizer_detector.zero_grad()                                   # keypoint_detector.py:186
        # ---- losses, forward (keypoint_detector.py:182-204)
        R = self.src_R_dst.contiguous()
        scale = self.src_scale_dst.reshape(-1).contiguous()
        shift = self.src_shift_dst.reshape(B, 3).contiguous()
        kp_t = ops.transform_points(self.src_keypoints, R, scale, shift)
        self.src_keypoints_transformed = kp_t
        out3, saved = losses.chamfer_prob_fwd(kp_t, self.dst_keypoints, self.src_sigmas, self.dst_sigmas)
        self.loss_chamfer, self.chamfer_pure, self.chamfer_weighted = out3[0], out3[1], out3[2]
        alpha = float(opt.keypoint_on_pc_alpha)
        plane = opt.keypoint_on_pc_type == 'point_to_plane'
        if not plane and opt.keypoint_on_pc_type != 'point_to_point':
            raise NotImplementedError("keypoint_on_pc_type=%r" % opt.keypoint_on_pc_type)
        sides = []
        d_all = arg_all = None
        if not plane:                                    # both sides in ONE nearest-neighbour call over the 2B clouds
            d_all, arg_all = ops.pairwise_min(kp, x)
        for side, (kps, pc, snn) in enumerate(((self.src_keypoints, self.src_pc, self.src_sn),
                                               (self.dst_keypoints, self.dst_pc, self.dst_sn))):
            pc = pc.contiguous()
            if plane:
                snn = snn.contiguous()
                d, arg = losses.point_on_surface_fwd(kps, pc, snn)
            else:
                d, arg = d_all[side * B:(side + 1) * B], arg_all[side * B:(side + 1) * B]
            sides.append((kps, pc, snn, d, arg, ops.mean_scale(d, alpha)[0]))
        self.loss_keypoint_on_pc_src, self.loss_keypoint_on_pc_dst = sides[0][5], sides[1][5]
        self.loss = self.loss_chamfer + self.loss_keypoint_on_pc_src + self.loss_keypoint_on_pc_dst
        # ---- losses, backward: d loss / d keypoints, sigmas
        if getattr(self, "_one", None) is None or self._one.device != kp.device:
            self._one = torch.ones(1, dtype=torch.float32, device=kp.device)
        g_kpt, g_dst, g_ss, g_sd = ops.chamfer_prob_bwd(*saved, self._one)
        g_kp = torch.empty_like(kp)
        g_kp[:B] = ops.transform_points_bwd(g_kpt, R, scale)
        g_kp[B:] = g_dst
        for half, (kps, pc, snn, d, arg, _) in zip((g_kp[:B], g_kp[B:]), sides):
            n = d.numel()
            g = self._one.expand(d.shape[0], d.shape[1]).contiguous() if not plane else None
            if plane:
                gk = ops.point_on_surface(kps, pc, snn, arg, torch.full_like(d, alpha / n))
            else:
                gk, _ = ops.pairwise_min_bwd(kps, pc, d, arg, g, want_b=False, scale=alpha / n)
            half += gk
        g_sig = torch.cat((g_ss, g_sd), dim=0)
        engine.detector_backward(net, ctx, g_kp, g_sig)

    def _optimize_graph(self, epoch):
        ins = [getattr(self, k) for k in self._GRAPH_INPUTS]
        decays = any(getattr(m, "momentum_decay_step", None) for m in self.detector.modules())
        key = (tuple(tuple(t.shape) for t in ins), (None if epoch is None else int(epoch)) if decays else None,
               self._dp is not None, tuple(p.requires_grad for p in self.detector.parameters()))
        if self._train_graph_key != key:
            try:
                self._capture_train_step(key, ins, epoch)
            except Exception as e:                       # e.g. a collective that cannot be captured: keep training eagerly
                import warnings
                warnings.warn("usip_b200: CUDA-graph capture of the train step failed (%s: %s); running eagerly"
                              % (type(e).__name__, e))
                self._train_graph_key = "failed"
                torch.cuda.synchronize()
                for k, v in zip(self._GRAPH_INPUTS, ins):
                    setattr(self, k, v)
                return self._optimize_eager(epoch)
        self.optimizer_detector.sync_hyperparams()        # lr lives in device memory; mirror it outside the graph
        for dst, src in zip(self._tgraph_in, ins):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self._tgraph.replay()
        _lib.LAUNCHES[0] += self._tgraph_launches
        _lib.WEIGHT_GEN[0] += 1                           # the replay moved the weights: packed tiles cached by eager paths are stale
        for k, v in zip(self._GRAPH_INPUTS, self._tgraph_in):
            setattr(self, k, v)
        for k, v in self._tgraph_out.items():
            setattr(self, k, v)

    def _capture_train_step(self, key, ins, epoch):
        opt_ = self.optimizer_detector
        self._tgraph_in = [t.clone() for t in ins]
        for k, v in zip(self._GRAPH_INPUTS, self._tgraph_in):
            setattr(self, k, v)
        # warm-up steps (allocator, kernel attributes) must not count as training: parameters, Adam state, the step
        # counter and the BatchNorm buffers are restored afterwards
        saved = [(t, t.detach().clone()) for t in [opt_.flat_p, opt_.exp_avg, opt_.exp_avg_sq, opt_.step_dev]
                 + list(self.detector.buffers())]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._optimize_eager(epoch)
            with torch.no_grad():
                for t, v in saved:
                    t.copy_(v)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        _lib.WEIGHT_GEN[0] += 1                           # the capture must contain the weight (re-)packing kernels
        g = torch.cuda.CUDAGraph()
        n0 = _lib.LAUNCHES[0]
        with torch.cuda.graph(g):
            self._optimize_eager(epoch)
        self._tgraph_launches = _lib.LAUNCHES[0] - n0
        self._tgraph = g
        self._tgraph_out = {k: getattr(self, k) for k in self._GRAPH_OUTPUTS}
        self._train_graph_key = key

    def test_model(self):
        self.detector.eval()
        with torch.cuda.device(self.src_pc.device), torch.no_grad():    # kernels launch on the inputs' device, whatever is current
            self._run_siamese(is_train=False, epoch=None)
            self._losses()

    _GRAPH_INPUTS = ("src_pc", "src_sn", "src_node", "dst_pc", "dst_sn", "dst_node",
                     "src_R_dst", "src_scale_dst", "src_shift_dst")
    _GRAPH_OUTPUTS = ("src_node_recomputed", "dst_node_recomputed", "src_keypoints", "dst_keypoints", "src_sigmas",
                      "dst_sigmas", "src_keypoints_transformed", "loss_chamfer", "chamfer_pure", "chamfer_weighted",
                      "loss_keypoint_on_pc_src", "loss_keypoint_on_pc_dst", "loss")

    def forward_loss(self, epoch=None, train_bn=True, graph=False):
        """fwd+loss only (the BASELINE metric): train-mode BatchNorm statistics, no backward.

        graph=True replays the whole step (≈70 kernel launches) as ONE CUDA graph: the launch sequence is captured the
        first time a given input shape / BN momentum / parameter version is seen, inputs are copied into the graph's
        static buffers, outputs (loss, keypoints, sigmas, ...) are the graph's static output tensors."""
        self.detector.train(train_bn)
        with torch.cuda.device(self.src_pc.device):
            return self._forward_loss(epoch, train_bn, graph)

    def _forward_loss(self, epoch, train_bn, graph):
        if not graph:
            with torch.no_grad():
                self._run_siamese(is_train=train_bn, epoch=epoch)
                self._losses()
            return self.loss
        ins = [getattr(self, k) for k in self._GRAPH_INPUTS]
        key = (tuple(tuple(t.shape) for t in ins), bool(train_bn), epoch if epoch is None else int(epoch),
               tuple(p._version for p in self.detector.parameters()), _lib.WEIGHT_GEN[0])
        if getattr(self, "_graph_key", None) != key:
            self._capture_forward_loss(key, ins, epoch, train_bn)
        for dst, src in zip(self._graph_in, ins):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self._graph.replay()
        _lib.LAUNCHES[0] += self._graph_launches
        for k, v in zip(self._GRAPH_INPUTS, self._graph_in):
            setattr(self, k, v)
        for k, v in self._graph_out.items():
            setattr(self, k, v)
        return self.loss

    def _capture_forward_loss(self, key, ins, epoch, train_bn):
        self._graph_in = [t.clone() for t in ins]
        for k, v in zip(self._GRAPH_INPUTS, self._graph_in):
            setattr(self, k, v)
        # the warm-up passes must not count as training steps: BatchNorm running statistics (and num_batches_tracked)
        # are restored afterwards, so a captured run leaves the same buffers behind as an eager one
        bn_buffers = [(b, b.detach().clone()) for b in self.detector.buffers()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():          # warm-up on a side stream (allocator, smem attributes,
            for _ in range(2):                                   # packed-weight cache) before capture
                self._run_siamese(is_train=train_bn, epoch=epoch)
                self._losses()
            for b, saved in bn_buffers:
                b.copy_(saved)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        n0 = _lib.LAUNCHES[0]
        with torch.cuda.graph(g), torch.no_grad():
            self._run_siamese(is_train=train_bn, epoch=epoch)
            self._losses()
        self._graph_launches = _lib.LAUNCHES[0] - n0
        self._graph = g
        self._graph_out = {k: getattr(self, k) for k in self._GRAPH_OUTPUTS}
        # the parameter versions may have been bumped by nothing here; recompute the key with the live versions
        self._graph_key = (key[0], key[1], key[2], tuple(p._version for p in self.detector.parameters()), _lib.WEIGHT_GEN[0])

    def freeze_model(self):
        for p in self.detector.parameters():
            p.requires_grad = False

    def run_model(self, pc, sn, node):
        self.detector.eval()
        with torch.no_grad():
            _, keypoints, sigmas, _ = self.forward(pc, sn, node, is_train=False, epoch=None)
        return keypoints, sigmas

    def run_model_siamese(self, pc_tuple, sn_tuple, node_tuple):
        self.detector.eval()
        with torch.no_grad():
            _, keypoints_tuple, sigmas_tuple, _ = self.forward_siamese(pc_tuple, sn_tuple, node_tuple,
                                                                       is_train=False, epoch=None)
        return keypoints_tuple, sigmas_tuple

    def get_current_visuals(self):
        raise NotImplementedError("visdom payloads (keypoint_detector.py:259-334) are outside the hot path")

    def get_current_errors(self):
        return OrderedDict([
            ('O_loss', self.loss.item()),
            ('O_chamfer', self.loss_chamfer.item()),
            ('O_key_on_pc', self.loss_keypoint_on_pc_src.item() + self.loss_keypoint_on_pc_dst.item()),
            ('E_loss', self.test_loss_average.item()),
            ('E_chamfer', self.test_chamfer_average.item()),
            ('E_key_on_pc', self.test_keypoint_on_pc_average.item()),
            ('E_cham_pure', self.test_chamfer_pure_average.item()),
            ('E_cham_weig', self.test_chamfer_weighted_average.item())
        ])

    def save_network(self, network, network_label, epoch_label, gpu_id):
        save_filename = '%s_net_%s.pth' % (epoch_label, network_label)
        save_path = os.path.join(self.opt.checkpoints_dir, save_filename)
        torch.save(network.state_dict(), save_path)

    def update_learning_rate(self, ratio):
        lr_clip = 0.00001
        lr_detector = self.old_lr_detector * ratio
        if lr_detector < lr_clip:
            lr_detector = lr_clip
        for param_group in self.optimizer_detector.param_groups:
            param_group['lr'] = lr_detector
        print('update detector learning rate: %f -> %f' % (self.old_lr_detector, lr_detector))
        self.old_lr_detector = lr_detector
