"""Parameter update of the train step: Adam over ONE flat buffer (usip_adam_step, csrc/optim.cu).

The reference builds `torch.optim.Adam(detector.parameters(), lr, betas=(0.9, 0.999), weight_decay=0)`
(models/keypoint_detector.py:42-45, keypoint_descriptor.py:32-35) and calls `.step()` once per `optimize()`.  Here the
same update is one kernel launch:

  * all parameters are re-pointed into one contiguous fp32 buffer `flat_p` (each tensor 16-byte aligned), all `.grad`s are
    views into `flat_g`; the moments `exp_avg` / `exp_avg_sq` are flat as well (per-parameter views are published in
    `state[p]`, the keys torch's Adam uses);
  * the backward plan (engine.detector_backward / descriptor_backward) ACCUMULATES straight into the `.grad` views --
    autograd's own accumulate semantics, without 42 zero-fills and 42 tiny adds per step -- and `zero_grad()` is one memset;
  * the data-parallel exchange is one all-reduce of `flat_g` (usip_b200/dp.py);
  * the step counter and the learning rate live in device memory, so `step()` can be captured in a CUDA graph
    (ModelDetector.optimize replays the whole train step as one graph); `param_groups[i]['lr']` stays the knob callers turn
    (ModelDetector.update_learning_rate), it is mirrored to the device when it changes.
"""
import torch

from . import _lib, ops


class FlatAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0):
        params = [p for p in params]
        if weight_decay != 0:
            raise NotImplementedError("FlatAdam: weight_decay != 0 is not used by the reference (keypoint_detector.py:45)")
        if not params:
            raise ValueError("FlatAdam: no parameters")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=0))
        p0 = params[0]
        if not p0.is_cuda:
            raise RuntimeError("FlatAdam: parameters must live on a CUDA device (move the module first)")
        dev = p0.device
        offs, n = [], 0
        for p in params:
            if p.dtype != torch.float32 or p.device != dev:
                raise RuntimeError("FlatAdam: fp32 parameters on one device only")
            offs.append(n)
            n += (p.numel() + 3) // 4 * 4                        # every tensor starts 16-byte aligned
        self.n = n
        self.flat_p = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.lr_dev = torch.full((1,), float(lr), dtype=torch.float32, device=dev)
        self._lr_host = float(lr)
        self._arrive = torch.zeros(1, dtype=torch.int32, device=dev)
        self.grad_scale = 1.0                                    # 1/world when the exchanged gradient is a SUM
        self._params = params
        for p, o in zip(params, offs):
            k = p.numel()
            with torch.no_grad():
                self.flat_p[o:o + k].copy_(p.detach().reshape(-1))
            p.data = self.flat_p[o:o + k].view(p.shape)
            g = self.flat_g[o:o + k].view(p.shape)
            p.grad = g
            p._usip_flat_grad = g                                # the backward plan accumulates here (engine._Bwd)
            self.state[p] = {"step": self.step_dev, "exp_avg": self.exp_avg[o:o + k].view(p.shape),
                             "exp_avg_sq": self.exp_avg_sq[o:o + k].view(p.shape)}

    # ------------------------------------------------------------------ gradients
    def zero_grad(self, set_to_none=False):
        """One memset; the `.grad` views are kept (set_to_none would detach them from the flat buffer)."""
        self.flat_g.zero_()
        for p in self._params:
            if p.grad is None or p.grad.data_ptr() != p._usip_flat_grad.data_ptr():
                p.grad = p._usip_flat_grad

    def views_intact(self):
        return all(p.grad is not None and p.grad.data_ptr() == p._usip_flat_grad.data_ptr() for p in self._params)

    # ------------------------------------------------------------------ update
    def sync_hyperparams(self):
        """Mirror param_groups' lr to the device scalar the kernel reads (call outside a graph capture / replay)."""
        lr = float(self.param_groups[0]["lr"])
        for g in self.param_groups[1:]:
            if float(g["lr"]) != lr:
                raise NotImplementedError("FlatAdam: one learning rate for all parameter groups")
        if lr != self._lr_host:
            self.lr_dev.fill_(lr)
            self._lr_host = lr

    @torch.no_grad()
    def step(self, closure=None):
        if closure is not None:
            raise NotImplementedError("FlatAdam.step: closures are not used by the reference")
        if not torch.cuda.is_current_stream_capturing():
            self.sync_hyperparams()
            if not self.views_intact():
                # someone replaced a .grad (e.g. module.zero_grad(set_to_none=True) followed by autograd): fold it back
                for p in self._params:
                    if p.grad is None:
                        p._usip_flat_grad.zero_()
                    elif p.grad.data_ptr() != p._usip_flat_grad.data_ptr():
                        p._usip_flat_grad.copy_(p.grad)
                    p.grad = p._usip_flat_grad
        g = self.param_groups[0]
        b1, b2 = g["betas"]
        ops.adam_step(self.flat_p, self.flat_g, self.exp_avg, self.exp_avg_sq, self.lr_dev, self.step_dev, self._arrive,
                      b1, b2, g["eps"], self.grad_scale)
        _lib.WEIGHT_GEN[0] += 1                                 # the raw-pointer update does not bump autograd versions
        return None
