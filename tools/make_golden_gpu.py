"""Generate tests/golden/ref_gpu_*.npz by RUNNING THE REFERENCE (unmodified, with its own two CUDA extensions) on a GPU at
the full BASELINE.json shapes of tests/test_gpu_vs_reference.py and the full-size operator cases of tests/test_gpu_ops.py.

    python tools/make_golden_gpu.py [OUTDIR]        (default tests/golden; needs oracle/_ref from oracle/build_ref.py)

The inputs come from the tests' own input functions, so what is stored is exactly what the tests compare against.
Full-size outputs do not fit in the repository: small tensors are stored whole, large ones as a fixed, evenly spread sample
of elements plus statistics over the whole tensor, bit-exact outputs as digests (tests/util_gpu.py: digest)."""
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import usip_oracle as orc  # noqa: E402
from tests import test_gpu_ops as O, test_gpu_vs_reference as T  # noqa: E402
from tests.util_gpu import digest  # noqa: E402


def _ref_run(ref, cfg, ins, double=False):
    """The unmodified reference on cuda: test_model() (eval BN) then optimize(epoch=0).  double=True runs the same modules
    in float64 -- the arbiter for the gradient comparison (only index_max, a float32-only extension, gets a float32 copy of
    its input; it returns indices)."""
    import index_max as ref_im
    big = 2 * cfg["B"] * cfg["M"] > 12288
    saved_fn = ref_im.forward_cuda_shared_mem
    # index_max_cuda.cu:92-96: the shared-memory variant needs B*K*4 <= 48 KB and silently returns zeros beyond it (no
    # cudaFuncSetAttribute); the reference's global-memory entry point is the same algorithm
    base_fn = ref_im.forward_cuda if big else saved_fn
    ref_im.forward_cuda_shared_mem = (lambda d, i, k: base_fn(d.float().contiguous(), i, k)) if double else base_fn
    try:
        rmd = T._mk(ref.keypoint_detector.ModelDetector, cfg)
        if double:
            rmd.detector.double()
            rmd.optimizer_detector = torch.optim.Adam(rmd.detector.parameters(), lr=rmd.opt.lr, betas=(0.9, 0.999), weight_decay=0)
            names = ("src_pc", "src_sn", "src_node", "dst_pc", "dst_sn", "dst_node", "src_R_dst", "src_scale_dst", "src_shift_dst")
            for k, v in zip(names, ins):                         # set_input() casts to float32 (keypoint_detector.py:125-133)
                setattr(rmd, k, v.double().to(rmd.opt.device))
        else:
            rmd.set_input(*ins)
        with torch.no_grad():
            rmd.test_model()
        r_eval = T._outs(rmd)
        random.seed(0); np.random.seed(0)
        rmd.optimize(epoch=0)
        torch.cuda.synchronize()
        r_train = T._outs(rmd)
        r_grad = {k: p.grad.detach().cpu().numpy().astype(np.float64) for k, p in rmd.detector.named_parameters()}
        r_sd = {k: v.detach().cpu().numpy() for k, v in rmd.detector.state_dict().items()}
    finally:
        ref_im.forward_cuda_shared_mem = saved_fn
    del rmd
    torch.cuda.empty_cache()
    return r_eval, r_train, r_grad, r_sd


def detector(ref, name, out_dir):
    cfg = T.CONFIGS[name]
    d = orc.synth_pair(cfg["B"], cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=cfg["seed"])
    ins = [torch.from_numpy(d[k]) for k in T.KEYS]
    r_eval, r_train, r_grad, r_sd = _ref_run(ref, cfg, ins)
    _, r64_train, r64_grad, _ = _ref_run(ref, cfg, ins, double=True)
    out = {}
    for t in T.OUTS:
        idx = T.sample_idx(r_eval[t].size, T.OUT_SAMPLE, t)
        for mode, r in (("eval", r_eval), ("train", r_train), ("train64", r64_train)):
            out["%s_%s" % (mode, t)] = r[t].reshape(-1)[idx].astype(np.float32)
            out["%s_%s_absmax" % (mode, t)] = np.float64(np.abs(r[t]).max())
    for mode, r in (("eval", r_eval), ("train", r_train), ("train64", r64_train)):
        out[mode + "_loss"] = r["loss"]
    P0 = T._params(cfg)
    lr = T.make_opt().lr
    for k, g32 in r_grad.items():
        g64 = r64_grad[k]
        sel = T.sample_idx(g64.size, T.SAMPLE, k)
        out["g64|" + k] = g64.reshape(-1)[sel].astype(np.float32)
        out["gstat|" + k] = np.array([np.abs(g64).max(), np.linalg.norm(g64), np.abs(g32 - g64).max(), np.linalg.norm(g32 - g64)])
        step = (np.asarray(P0[k], np.float64).reshape(-1) - r_sd[k].astype(np.float64).reshape(-1)) / lr
        out["step|" + k] = step[sel].astype(np.float16)
        gr = np.abs(g32).reshape(-1)
        big = gr > 0.2 * gr.max()
        if k.endswith("conv.bias") and np.linalg.norm(g64) < 1e-6 * np.linalg.norm(r64_grad[k.replace("bias", "weight")]):
            big[:] = False
        out["big|" + k] = np.packbits(big[sel])
    for k, v in r_sd.items():
        if k.endswith("running_mean") or k.endswith("running_var") or k.endswith("num_batches_tracked"):
            out["buf|" + k] = v
    np.savez_compressed(os.path.join(out_dir, "ref_gpu_detector_%s.npz" % name), **out)


def descriptor(ref, out_dir):
    res = T.descriptor_run(ref.networks.DescriptorLiteOld, *T.descriptor_inputs())
    out = {}
    for mode, (desc, feats) in res.items():
        out[mode + "_desc"] = desc.reshape(-1)[T.sample_idx(desc.size, T.DESC_SAMPLE, "descriptor")]
        out[mode + "_desc_absmax"] = np.float64(np.abs(desc).max())
        out[mode + "_feats"] = np.array(digest(feats))
    np.savez_compressed(os.path.join(out_dir, "ref_gpu_descriptor.npz"), **out)


def ops(out_dir):
    from oracle import build_ref
    ref_im, ref_bq = build_ref._load_so("index_max"), build_ref._load_so("ball_query")
    out = {}
    data, index = O.index_max_full_size_inputs()
    out["index_max_full_size"] = digest(ref_im.forward_cuda(data, index, 512).int())
    _, _, dist = O.ball_query_inputs()
    out["ball_query"] = digest(ref_bq.forward_cuda_shared_mem(dist, 1.0, 64).int())
    for dense, pc, sn, kp, K in O.ball_group_grid_cases():
        dist = torch.norm(kp.unsqueeze(3) - pc.unsqueeze(2), dim=1).contiguous()
        out["ball_group_grid_dense" if dense else "ball_group_grid"] = digest(ref_bq.forward_cuda_shared_mem(dist, 1.0, K).int())
        del dist
    np.savez_compressed(os.path.join(out_dir, "ref_gpu_ops.npz"), **{k: np.array(v) for k, v in out.items()})


def main():
    from oracle import ref_shim
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = ref_shim.modules(mode="cuda")
    ops(out_dir)
    descriptor(ref, out_dir)
    for name in T.CONFIGS:
        detector(ref, name, out_dir)
    for f in sorted(os.listdir(out_dir)):
        print(f, os.path.getsize(os.path.join(out_dir, f)) // 1024, "KB")


if __name__ == "__main__":
    main()
