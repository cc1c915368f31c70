"""Time the registration evaluation (usip_b200.evaluation.registration) on the 2,831 ground-truth transforms of the KITTI
test list, with synthetic keypoints and descriptors (inlier ratios uniform in [0.1, 0.5], 0.05 m noise, 128-dim
descriptors).  Workloads: KITTI protocol (1-NN) at 256 and 512 keypoints per frame, Oxford protocol (5-NN both ways,
union) at 256.  CUDA events after a warm-up; prints one JSON line (and writes it to --out when given).

  python tools/bench_registration.py [--reps 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.registration_data import kitti_gt_transforms  # noqa: E402
from usip_b200.evaluation import registration as reg  # noqa: E402

CHUNK_ENDS = (64, 320, 1344, 5440)                 # csrc/registration.cu RANSAC_CHUNK_ENDS
FLOP_PER_RESIDUAL = 26                             # 9 mul + 9 add (R y + t), 3 sub, 3 mul + 2 add (d^2); plus one sqrt
FP64_PEAK_TFLOPS = 37.0                            # B200 data sheet, dense FP64, one GPU


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:  # the numbers below still stand; the card is then named by torch only
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def make_pairs(T, M, C, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = T.shape[0]
    Tt = torch.from_numpy(T).cuda().float()
    ratio = torch.rand(B, generator=g, device="cuda") * 0.4 + 0.1
    scale = torch.tensor([30.0, 30.0, 3.0], device="cuda")
    pos = (torch.rand(B, M, 3, generator=g, device="cuda") * 2 - 1) * scale
    anc = pos @ Tt[:, :, :3].transpose(1, 2) + Tt[:, None, :, 3] + 0.05 * torch.randn(B, M, 3, generator=g, device="cuda")
    pd = torch.randn(B, M, C, generator=g, device="cuda")
    ad = pd + 0.05 * torch.randn(B, M, C, generator=g, device="cuda")
    outl = torch.arange(M, device="cuda")[None, :] >= (ratio[:, None] * M).round()
    anc = torch.where(outl[:, :, None], (torch.rand(B, M, 3, generator=g, device="cuda") * 2 - 1) * scale, anc)
    ad = torch.where(outl[:, :, None], torch.randn(B, M, C, generator=g, device="cuda"), ad)
    perm = torch.argsort(torch.rand(B, M, generator=g, device="cuda"), 1)
    pos = torch.gather(pos, 1, perm[:, :, None].expand(B, M, 3))
    pd = torch.gather(pd, 1, perm[:, :, None].expand(B, M, C))
    return anc.contiguous(), pos.contiguous(), ad.contiguous(), pd.contiguous()


def scored_trials(tc, T):
    ends = np.array([e for e in CHUNK_ENDS if e < T] + [T])
    return np.array([T if t >= T else ends[np.searchsorted(ends, t + 1)] if t > 0 else 0 for t in tc])


def run(name, T, M, k, both, C, reps):
    anc, pos, ad, pd = make_pairs(T, M, C, seed=M + k)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    times = {"match": [], "corr_build": [], "ransac": [], "total": []}
    for it in range(reps + 1):                     # iteration 0 warms every shape up
        e = [ev() for _ in range(5)]
        torch.cuda.synchronize()
        e[0].record()
        a = ad.transpose(1, 2).contiguous(); b = pd.transpose(1, 2).contiguous()
        from usip_b200 import ops
        nn12 = ops.desc_knn(a, b, k)
        nn21 = ops.desc_knn(b, a, k) if both else None
        e[1].record()
        corr, cnt = ops.corr_build(nn12, M, nn21)
        e[2].record()
        r = reg.ransac_fit_rt(anc, pos, corr, cnt, seed=it)
        e[3].record()
        res = reg.summarize_registration(T, r, cnt)
        e[4].record()
        torch.cuda.synchronize()
        if it:
            times["match"].append(e[0].elapsed_time(e[1])); times["corr_build"].append(e[1].elapsed_time(e[2]))
            times["ransac"].append(e[2].elapsed_time(e[3])); times["total"].append(e[0].elapsed_time(e[4]))
    tc = res["trialcount"]
    ncorr = res["n_corr"]
    work = float((scored_trials(tc, 10002) * ncorr).sum())
    t_ransac = float(np.median(times["ransac"])) * 1e-3
    rec = {"workload": name, "pairs": int(T.shape[0]), "keypoints": M, "k": k, "both_directions": both,
           "ms": {key: round(float(np.median(v)), 3) for key, v in times.items()},
           "pairs_per_s": round(T.shape[0] / (float(np.median(times["total"])) * 1e-3), 1),
           "mean_trialcount": round(float(tc.mean()), 1), "mean_correspondences": round(float(ncorr.mean()), 1),
           "wrong_counter": res["wrong_counter"], "rte_mean": round(res["rte_mean"], 4), "rre_mean": round(res["rre_mean"], 4),
           "fp64_residuals": work, "fp64_tflops": round(work * FLOP_PER_RESIDUAL / t_ransac * 1e-12, 2),
           "fp64_peak_share_ransac": round(work * FLOP_PER_RESIDUAL / t_ransac * 1e-12 / FP64_PEAK_TFLOPS, 3)}
    return rec, (anc, pos, corr, cnt, r)


def cpu_baseline(data, n_pairs=16):
    """float64 numpy oracle (oracle/registration.py) on the first n_pairs, with the GPU's own sample table"""
    from oracle import registration as orc
    anc, pos, corr, cnt, _ = data
    sub = slice(0, n_pairs)
    r = reg.ransac_fit_rt(anc[sub], pos[sub], corr[sub], cnt[sub], seed=0, return_samples=True)
    a, p, c, n, s = (t.cpu().numpy() for t in (anc[sub], pos[sub], corr[sub], cnt[sub], r.samples))
    t0 = time.perf_counter()
    for b in range(n_pairs):
        cc = c[b, :n[b]].astype(np.int64)
        orc.ransac_rt(a[b][cc[:, 0]].T.astype(np.float64), p[b][cc[:, 1]].T.astype(np.float64), s[b], 1.0, 10001)
    return {"cpu_oracle_pairs": n_pairs, "cpu_oracle_s": round(time.perf_counter() - t0, 2),
            "note": "numpy float64 oracle, one host core, RANSAC only"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_registration needs a CUDA device")
    T = kitti_gt_transforms()
    out = {"bench": "registration", **gpu_info(), "fp64_peak_tflops_datasheet": FP64_PEAK_TFLOPS,
           "flop_per_residual": FLOP_PER_RESIDUAL, "bound": "fp64 issue (residual scoring); see fp64_peak_share_ransac",
           "workloads": []}
    for name, M, k, both in (("kitti_256", 256, 1, False), ("kitti_512", 512, 1, False), ("oxford_256", 256, 5, True)):
        rec, data = run(name, T, M, k, both, 128, args.reps)
        out["workloads"].append(rec)
        if name == "kitti_256":
            out["cpu_baseline"] = cpu_baseline(data)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
