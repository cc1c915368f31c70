"""Shared helpers for the -m gpu parity tests (the CUDA path is called through the C ABI via usip_b200.ops /
usip_b200.models; the checker is oracle/ and the reference goldens)."""
import hashlib
import os
import types

import numpy as np
import torch


def dev():
    return torch.device("cuda:0")


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(dev())


def rel_err(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-12))


def make_opt(**over):
    o = types.SimpleNamespace(
        gpu_ids=[0], device=dev(), scene="outdoor",
        batch_size=2, input_pc_num=1024, surface_normal_len=4, node_num=64, k=1, node_knn_k_1=16,
        activation="relu", normalization="batch", bn_momentum=0.1, bn_momentum_decay_step=None,
        bn_momentum_decay=0.6, lr=0.001, loss_sigma_lower_bound=0.001,
        random_pc_dropout_lower_limit=1.0, keypoint_on_pc_type="point_to_point",
        keypoint_on_pc_alpha=0.01, rot_3d=False, rot_horizontal=True, checkpoints_dir="/tmp",
        ball_radius=1.0, ball_nsamples=64, descriptor_len=128, sigma_max=3.0, triple_loss_gamma=0.5,
        use_tensor_cores=True,
    )
    o.__dict__.update(over)
    return o


def load_params(module, P):
    sd = module.state_dict()
    for k in sd:
        assert k in P, k
        sd[k] = torch.from_numpy(np.asarray(P[k])).reshape(sd[k].shape).to(sd[k].dtype)
    module.load_state_dict(sd)


def golden(name):
    here = os.path.dirname(os.path.abspath(__file__))
    return np.load(os.path.join(here, "golden", name), allow_pickle=False)


def digest(t):
    """SHA-256 over shape, dtype and bytes of a tensor / array: bit-for-bit comparison against a stored output that is
    too large to keep in tests/golden/."""
    a = np.ascontiguousarray(t.detach().cpu().numpy() if torch.is_tensor(t) else t)
    h = hashlib.sha256(repr((a.shape, a.dtype.str)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def ref_ext(name):
    """The reference's own CUDA extension compiled from its sources into oracle/_ref (None if absent)."""
    try:
        from oracle import build_ref
        if not build_ref.have(name):
            return None
        return build_ref._load_so(name)
    except Exception as e:  # pragma: no cover
        print("reference ext %s unavailable: %s" % (name, e))
        return None
