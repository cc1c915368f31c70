#!/usr/bin/env python
"""bench.py -- clouds/sec of the USIP detector fwd+loss hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's own CPU path (unmodified reference staged
                                                           # under oracle/_ref/py + its C++ index_max; else the port)
  python bench.py ... --dump-outputs DIR                   # also write the outputs of the last timed step to DIR/*.npy

Workload (config.workload): BASELINE.json configs[2] "KITTI detector" -- per rank B=8 pairs = 16 clouds,
N=16384 points, M=512 nodes, S=4, node kNN K=16, train-mode BatchNorm, probabilistic chamfer + 2x
keypoint-on-pc loss.  A step = one fwd+loss pass over one synthetic batch.  Weak scaling: every rank processes its
own batch; the fwd+loss path has no collective; the gradient all-reduce belongs to the train step, which is timed in
every run and reported in `train_step` (fwd+loss+backward+Adam, + the NCCL all-reduce when N>1).  At N=1 the line also
carries `reference_gpu` (the UNMODIFIED reference's 1-GPU PyTorch path on the same tensors, same GPU: the ">=10x"
denominator of BASELINE.json's north_star) and `descriptor` (Oxford descriptor path: fused ball-query+group roofline,
descriptor forward).  `value` = clouds of all ranks / max-over-ranks device time, inputs resident in HBM (a rotating set of
distinct batches larger than L2); `e2e` = same metric through ModelDetector.set_input() from pinned host tensors +
loss.item() every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KITTI = dict(B=8, N=16384, M=512, S=4, Kn=16, kind="lidar", lb=1e-3, alpha=0.01)
METRIC = "clouds/sec detector fwd+loss (N=16384,M=512)"
# algorithmic dense flops of one cloud's forward (SURVEY.md 8d: 13.1 GF incl. the 131->256 and the concat layers as
# the reference computes them); the flops we actually issue are lower (per-node GEMMs for the concat halves)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], bf16_tflops=j["bf16_tflops"], bf16_tflops_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  `nvidia-smi -lms` needs ~0.1 s before its
    first line and the timed region of a 1.3 ms step is a few tens of ms, so the sampler is started before the warm-up,
    every line is time-stamped, and the caller keeps the SAME steps running (untimed) after the timed region until at
    least three samples lie inside the load window; `window_ms` says how long that window was."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def count_between(self, t0, t1):
        return sum(1 for (t, _) in list(self.lines) if t0 <= t <= t1)

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for (t, ln) in self.lines:
            if t0 is not None and not (t0 <= t <= t1):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if t0 is not None:
            out["window_ms"] = round((t1 - t0) * 1e3, 1)
        return out


def make_batches(nb, cfg, seed0):
    from oracle import usip_oracle as orc       # synthetic-data generator only (SURVEY.md 8d); not a compute path
    return [orc.synth_pair(cfg["B"], cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=seed0 + i) for i in range(nb)]


KEYS = ("src_pc", "src_sn", "src_node", "dst_pc", "dst_sn", "dst_node", "R", "scale", "shift")


def _workload_config(cfg, world):
    return {"workload": "KITTI detector fwd+loss (BASELINE configs[2]): per rank B=8 pairs (16 clouds), "
                        "N=16384, M=512, S=4, node_knn_k=16, train-mode BN, chamfer + 2x keypoint-on-pc",
            "global_pairs": cfg["B"] * world}


def _ref_opt(ref_shim, cfg, B, **over):
    return ref_shim.make_opt(batch_size=B, input_pc_num=cfg["N"], node_num=cfg["M"], surface_normal_len=cfg["S"],
                             node_knn_k_1=cfg["Kn"], loss_sigma_lower_bound=cfg["lb"], keypoint_on_pc_alpha=cfg["alpha"], **over)


def _ref_fwd_loss_train_bn(rmd):
    """The reference's own fwd+loss code (ModelDetector.test_model, keypoint_detector.py:209-241) with train-mode
    BatchNorm statistics -- the metric's definition (SURVEY.md 8d) -- under no_grad: test_model() begins with
    self.detector.eval(); the instance attribute below turns that one call into a no-op so the detector stays in train()."""
    import torch
    rmd.detector.train()
    rmd.detector.eval = lambda: rmd.detector
    try:
        with torch.no_grad():
            rmd.test_model()
    finally:
        del rmd.detector.eval
    return rmd.loss


def _calibrate_cpu_threads(cfg, step_fn):
    """Thread count for the reference's CPU run.  ~90 % of its time is `torch.norm(diff, dim=1)` over the (B,3,N,M) tensors of
    som.query_topk / the chamfer losses (util/som.py:30-34, losses.py:62-66) -- a reduction over a dimension of size 3 that
    torch parallelises badly: with all 128 threads of the GPU box one pair took 19.5 s, with 8 threads of another host 2.7 s.
    The arm therefore times ONE quarter-size step (N/4 points, same M) of the reference itself at a few thread counts and
    keeps the fastest; it reports the count it used."""
    import torch
    n = os.cpu_count() or 1
    cands = sorted({c for c in (n, n // 2, n // 4, n // 8, 16, 8) if 1 <= c <= n}, reverse=True)
    best_t, best_c, log = float("inf"), n, []
    for c in cands:
        torch.set_num_threads(c)
        step_fn()
        t0 = time.perf_counter()
        step_fn()
        dt = time.perf_counter() - t0
        log.append("%d: %.2f s" % (c, dt))
        if dt < best_t:
            best_t, best_c = dt, c
    return best_c, ", ".join(log)


def cpu_reference_run(cfg, steps, warmup, threads=None):
    """The reference's CPU path on a bounded sample: ONE pair (2 clouds) of the same workload per step.
    kind="reference": the unmodified reference (oracle/_ref/py, its own C++ index_max.forward_cpu) through oracle/ref_shim;
    kind="port": the numpy/C oracle restatement, only when the reference is not staged."""
    from oracle import usip_oracle as orc
    import torch
    tried = None
    calibrate = threads is None
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    d = orc.synth_pair(1, cfg["N"], cfg["M"], cfg["S"], kind=cfg["kind"], seed=999)
    P = orc.init_detector_params(S=cfg["S"], seed=0)
    kind = "port"
    try:
        from oracle import ref_shim
        if ref_shim.reference_available():
            ref = ref_shim.modules(mode="cpu")
            from tests.util_gpu import load_params
            rmd = ref.keypoint_detector.ModelDetector(_ref_opt(ref_shim, cfg, 1))
            load_params(rmd.detector, P)
            rmd.set_input(*[torch.from_numpy(d[k]) for k in KEYS])
            kind = "reference"
            if calibrate:
                cal = dict(cfg); cal["N"] = max(1024, cfg["N"] // 4)
                dc = orc.synth_pair(1, cal["N"], cal["M"], cal["S"], kind=cal["kind"], seed=998)
                cmd = ref.keypoint_detector.ModelDetector(_ref_opt(ref_shim, cal, 1))
                load_params(cmd.detector, P)
                cmd.set_input(*[torch.from_numpy(dc[k]) for k in KEYS])
                threads, tried = _calibrate_cpu_threads(cfg, lambda: float(_ref_fwd_loss_train_bn(cmd)))
                torch.set_num_threads(threads)
                del cmd
    except Exception as e:  # pragma: no cover
        print("[bench] reference CPU path unavailable (%s); timing the oracle port" % e, file=sys.stderr)
        kind = "port"
    limiter = None
    if kind == "port":
        try:
            from threadpoolctl import threadpool_limits
            limiter = threadpool_limits(limits=threads)
        except Exception:
            pass
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        if kind == "reference":
            float(_ref_fwd_loss_train_bn(rmd))
        else:
            orc.detector_fwd_loss(P, d["src_pc"], d["src_sn"], d["src_node"], d["dst_pc"], d["dst_sn"], d["dst_node"],
                                  d["R"], d["scale"], d["shift"], node_knn_k=cfg["Kn"], sigma_lower_bound=cfg["lb"],
                                  alpha=cfg["alpha"], training=True)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    del limiter
    t = float(np.mean(times))
    what = ("unmodified reference ModelDetector (models/keypoint_detector.py:209-241, train-mode BN, no_grad) on CPU, "
            "torch %d of %d threads%s, its own C++ index_max.forward_cpu"
            % (threads, os.cpu_count() or 1, (" (fastest of a quarter-size step at %s)" % tried) if tried else "")) \
        if kind == "reference" else "numpy/BLAS + C oracle port"
    return dict(value=2.0 / t, unit="clouds/s", cores=int(threads), kind=kind,
                sample="%d x (1 pair = 2 clouds, N=%d, M=%d) fwd+loss, %s; %.2f s per pair"
                       % (len(times), cfg["N"], cfg["M"], what, t)), t


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = dict(KITTI)
    steps = max(1, args.steps); warmup = max(0, args.warmup)
    cb, t = cpu_reference_run(cfg, steps, warmup)
    conf = _workload_config(cfg, 1)
    conf["reference_sample"] = "bounded sample of that workload: 1 pair (2 clouds) per step on the host cores"
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "clouds/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": conf,
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def reference_gpu_record(cfg, resident, P, dev, ours_ms, ours_train_ms, iters=20, warm=5):
    """The UNMODIFIED reference's 1-GPU PyTorch path (oracle/_ref/py + its two CUDA extensions) on the same resident
    tensors and parameters, CUDA-event timed on this GPU: `fwd_loss` = its own test_model() code with train-mode BN under
    no_grad (the metric), `train_step` = its optimize().  Two precision settings: TF32 off (the fp32 arithmetic our
    3xTF32 path is equivalent to) and PyTorch's defaults (cuDNN convolutions may use TF32)."""
    import torch
    from oracle import build_ref, ref_shim
    if not (ref_shim.reference_available() and build_ref.have("index_max") and build_ref.have("ball_query")):
        return {"unavailable": "oracle/_ref (staged reference tree + its two extensions) not built"}
    from tests.util_gpu import load_params
    ref = ref_shim.modules(mode="cuda")
    rmd = ref.keypoint_detector.ModelDetector(_ref_opt(ref_shim, cfg, cfg["B"], device=dev, gpu_ids=[dev.index or 0]))
    load_params(rmd.detector, P)
    nb = len(resident)

    def assign(i):
        b = resident[i % nb]
        rmd.src_pc, rmd.src_sn, rmd.src_node = b["src_pc"], b["src_sn"], b["src_node"]
        rmd.dst_pc, rmd.dst_sn, rmd.dst_node = b["dst_pc"], b["dst_sn"], b["dst_node"]
        rmd.src_R_dst, rmd.src_scale_dst, rmd.src_shift_dst = b["R"], b["scale"], b["shift"]

    def timed(fn):
        for i in range(warm):
            assign(i); fn()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            assign(i); fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    clouds = 2 * cfg["B"]
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    out = {"what": "unmodified lijx10/USIP ModelDetector on cuda:%d, same tensors/parameters, %d warm-up + %d timed "
                   "iterations, CUDA events" % (dev.index or 0, warm, iters), "clouds_per_step": clouds}
    try:
        for tag, tf32 in (("tf32_off", False), ("torch_default", None)):
            if tf32 is None:
                torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
            else:
                torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
            ms_f = timed(lambda: _ref_fwd_loss_train_bn(rmd))
            ms_t = timed(lambda: rmd.optimize(epoch=0))
            out[tag] = {"fwd_loss_ms": ms_f, "fwd_loss_clouds_per_s": clouds / (ms_f * 1e-3),
                        "train_step_ms": ms_t, "train_step_clouds_per_s": clouds / (ms_t * 1e-3),
                        "ours_speedup_fwd_loss": ms_f / ours_ms,
                        "ours_speedup_train_step": None if ours_train_ms is None else ms_t / ours_train_ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    out["peak_mem_GB"] = torch.cuda.max_memory_allocated(dev) / 1e9
    del rmd
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tc", action="store_true", help="fp32 SIMT layers only")
    ap.add_argument("--train", action="store_true", help="(kept for compatibility: the train step is always timed)")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step record")
    ap.add_argument("--no-tf32-backward", action="store_true", help="skip the extra train-step record with TF32 backward GEMMs")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip timing the reference's own GPU path (N=1 only)")
    ap.add_argument("--no-descriptor", action="store_true", help="skip the descriptor-path sub-record (N=1 only)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay of the step")
    ap.add_argument("--nbatches", type=int, default=18, help="distinct resident input batches (18 x 7.3 MB > 126 MB L2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed fwd+loss step returned (keypoints, sigmas, nodes, losses; rank 0) as "
                         "DIR/<name>.npy in float32, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from usip_b200 import _lib, engine
    from usip_b200.models.keypoint_detector import ModelDetector
    from tests.util_gpu import make_opt, load_params
    from oracle import usip_oracle as orc       # parameter init + synthetic data generators only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    cfg = dict(KITTI)

    opt = make_opt(batch_size=cfg["B"], input_pc_num=cfg["N"], node_num=cfg["M"], surface_normal_len=cfg["S"],
                   node_knn_k_1=cfg["Kn"], loss_sigma_lower_bound=cfg["lb"], keypoint_on_pc_alpha=cfg["alpha"],
                   use_tensor_cores=not args.no_tc, device=dev, gpu_ids=[local])
    md = ModelDetector(opt)
    P0 = orc.init_detector_params(S=cfg["S"], seed=0)
    load_params(md.detector, P0)                                              # same weights on every rank
    nb = args.nbatches
    host = make_batches(nb, cfg, seed0=1234 + 2 + 1000 * rank)
    pinned = [{k: torch.from_numpy(b[k]).pin_memory() for k in KEYS} for b in host]
    resident = [{k: v.to(dev) for k, v in b.items()} for b in pinned]
    h2d_bytes = sum(v.numel() * 4 for v in pinned[0].values())

    def assign(b):
        md.src_pc, md.src_sn, md.src_node = b["src_pc"], b["src_sn"], b["src_node"]
        md.dst_pc, md.dst_sn, md.dst_node = b["dst_pc"], b["dst_sn"], b["dst_node"]
        md.src_R_dst, md.src_scale_dst, md.src_shift_dst = b["R"], b["scale"], b["shift"]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(step_fn, nsteps):
        """EXACTLY nsteps steps bracketed by barrier+synchronize, device time via CUDA events, max over ranks."""
        sync_all()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        _lib.LAUNCHES[0] = 0
        e0.record()
        for i in range(nsteps):
            step_fn(i)
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        launches = _lib.LAUNCHES[0]
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    # ---- per-op device times (CUDA events on the launching stream) for the roofline of the dominant kernel
    for i in range(3):
        assign(resident[i % nb]); md.forward_loss(epoch=0, train_bn=True, graph=False)
    torch.cuda.synchronize()
    engine.PROFILE = {}
    for i in range(min(K, 10)):
        assign(resident[i % nb])
        md.forward_loss(epoch=0, train_bn=True, graph=False)    # eager: events around every op
    torch.cuda.synchronize()
    prof = engine.collect_profile()
    engine.PROFILE = None
    # ---- kernel-path number: inputs resident in HBM
    def step_resident(i):
        assign(resident[i % nb])
        md.forward_loss(epoch=0, train_bn=True, graph=use_graph)

    use_graph = not args.no_graph
    sampler = ClockSampler(local); sampler.start()     # before the warm-up: nvidia-smi -lms takes ~0.1 s to its first line
    for i in range(W):
        step_resident(i)
    t_load0 = time.time()
    ms, launches = timed(step_resident, K)
    # copied now: the steps below overwrite the graph's static output tensors
    outputs = {k: getattr(md, k).detach().float().cpu().numpy() for k in ModelDetector._GRAPH_OUTPUTS} if args.dump_outputs else None
    # the timed region is over (ms is final); the same steps keep the GPU under the same load until the sampler has seen it
    t_load1 = time.time()
    while sampler.count_between(t_load0, t_load1) < 3 and time.time() - t_load0 < 2.0:
        for i in range(max(K, 20)):
            step_resident(i)
        torch.cuda.synchronize()
        t_load1 = time.time()
    clocks = sampler.stop(t_load0, t_load1)
    clocks["timed_region_ms"] = round(ms, 2)
    clouds = 2 * cfg["B"] * world
    value = clouds * K / (ms * 1e-3)

    # ---- end-to-end through the public API: pinned host -> set_input -> forward_loss -> loss.item()
    # Every step copies ITS inputs from pinned host memory and reads ITS loss back; the copy of step i+1 is issued
    # (prefetch_input, a side stream) before step i's loss is awaited, the way a training loop's loader would.
    def batch_args(i):
        b = pinned[i % nb]
        return [b[k] for k in KEYS]

    # The loss of every step is copied to pinned host memory right behind its kernels and READ one step later (the last
    # one before the region closes), so the host never idles the GPU: K input copies, K loss reads, all inside the region.
    loss_pinned = torch.empty(2, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"n": K, "losses": []}

    def step_e2e(i):
        md.set_input(*batch_args(i))                 # adopts the staged copy of this step's batch (or copies it now)
        md.prefetch_input(*batch_args(i + 1))
        md.forward_loss(epoch=0, train_bn=True, graph=use_graph)
        loss_pinned[i % 2].copy_(md.loss, non_blocking=True)
        loss_ev[i % 2].record()
        if i > 0:
            loss_ev[(i - 1) % 2].synchronize(); e2e_state["losses"].append(float(loss_pinned[(i - 1) % 2]))
        if i == e2e_state["n"] - 1:
            loss_ev[i % 2].synchronize(); e2e_state["losses"].append(float(loss_pinned[i % 2]))

    e2e_state["n"] = 3
    for i in range(3):
        step_e2e(i)
    md._staged = None                                # the timed region starts with nothing staged
    e2e_state.update(n=K, losses=[])
    ms_e2e, _ = timed(step_e2e, K)
    assert len(e2e_state["losses"]) == K and all(np.isfinite(e2e_state["losses"]))
    e2e = {"value": clouds * K / (ms_e2e * 1e-3), "unit": "clouds/s", "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K}

    roof = None
    pk = peaks()
    if prof:
        layer_ops = {k: v for k, v in prof.items() if v.get("flops")}
        top = max((layer_ops or prof).items(), key=lambda kv: kv[1]["ms"])
        name, rec = top
        step_ms = sum(r["ms"] for r in prof.values())
        if rec.get("flops"):
            ach = rec["flops"] / (rec["ms"] * 1e-3) / 1e12
            tf32_peak = pk["bf16_tflops"] / 2.0           # the kernel is event-timed on its own: the BURST figure applies
            roof = {"bound": "tensor", "kernel": name, "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s",
                    "frac": ach / tf32_peak, "traffic": None,
                    "note": "achieved = algorithmic flops (2*P*Cin*Cout) / CUDA-event time of that launch; peak = measured BURST "
                            "bf16 cuBLAS rate / 2 (TF32 runs at half the bf16 rate; %s); the kernel issues 3 TF32 MMAs per "
                            "algorithmic MAC (3xTF32), so its tensor-pipe issue fraction is 3x frac" % pk["source"],
                    "frac_vs_sustained_peak": ach / (pk["bf16_tflops_sustained"] / 2.0),
                    "frac_issued_tf32": 3 * ach / tf32_peak, "kernel_ms": rec["ms"], "kernel_share_of_step": rec["ms"] / step_ms,
                    "precision": rec.get("precision", "fp32")}
        else:
            ach = (rec.get("bytes") or 0) / (rec["ms"] * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": name, "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": None, "kernel_ms": rec["ms"],
                    "kernel_share_of_step": rec["ms"] / step_ms, "note": pk["source"]}
        roof["per_op_ms"] = {k: round(v["ms"], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:12]}
        # dram bytes per launch of that kernel from the committed `ncu --set full` capture (profiles/, tools/gpu_profile.sh)
        import glob
        for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_top_kernel_traffic.json")), reverse=True):
            t = json.load(open(f))
            if t.get("kernel", "").split(" ")[0] == roof["kernel"]:
                roof["traffic"] = t["traffic"]
                import re
                m = re.match(r".*\[(\d+)x(\d+)->(\d+)\]", roof["kernel"])
                P_, Ci_, Co_ = (int(x) for x in m.groups())
                roof["traffic_source"] = "%s: dram read %.0f MB + write %.0f MB per launch; compulsory: X %.0f MB read, group max/min %.0f MB written" % (
                    os.path.basename(f), t["dram_bytes_read"] / 1e6, t["dram_bytes_write"] / 1e6, 4e-6 * P_ * Ci_, 8e-6 * (P_ // 16) * Co_)
                break

    # ---- full train step (BASELINE configs[2] / [4]): fwd + loss + backward + Adam (+ NCCL gradient all-reduce, N>1)
    train = None
    if not args.no_train:
        def step_train(i):
            assign(resident[i % nb])
            md.optimize(epoch=0)
        if world > 1:
            md.enable_data_parallel()
        for i in range(W):
            step_train(i)
        ms_t, l_t = timed(step_train, K)
        train = {"value": clouds * K / (ms_t * 1e-3), "unit": "clouds/s", "ms_per_step": ms_t / K, "gpu_launches": l_t,
                 "includes": "fwd (train BN) + loss + backward + Adam" + (" + NCCL all-reduce of the flat 4.79 MB gradient buffer" if world > 1 else ""),
                 "loss_after": float(md.loss)}
        assert np.isfinite(train["loss_after"])

    # ---- the same train step with the backward GEMMs in plain single-pass TF32 (opt.backward_precision = "tf32": the
    # arithmetic PyTorch's default cuDNN path gives the reference's backward).  A labelled extra, never the headline.
    train_tf32 = None
    if not args.no_train and world == 1 and not args.no_tf32_backward:
        opt2 = make_opt(batch_size=cfg["B"], input_pc_num=cfg["N"], node_num=cfg["M"], surface_normal_len=cfg["S"],
                        node_knn_k_1=cfg["Kn"], loss_sigma_lower_bound=cfg["lb"], keypoint_on_pc_alpha=cfg["alpha"],
                        use_tensor_cores=not args.no_tc, device=dev, gpu_ids=[local], backward_precision="tf32")
        md2 = ModelDetector(opt2)
        load_params(md2.detector, P0)
        md_main = md

        def step_train2(i):
            b = resident[i % nb]
            md2.src_pc, md2.src_sn, md2.src_node = b["src_pc"], b["src_sn"], b["src_node"]
            md2.dst_pc, md2.dst_sn, md2.dst_node = b["dst_pc"], b["dst_sn"], b["dst_node"]
            md2.src_R_dst, md2.src_scale_dst, md2.src_shift_dst = b["R"], b["scale"], b["shift"]
            md2.optimize(epoch=0)
        for i in range(W):
            step_train2(i)
        ms_t2, l_t2 = timed(step_train2, K)
        train_tf32 = {"value": clouds * K / (ms_t2 * 1e-3), "unit": "clouds/s", "ms_per_step": ms_t2 / K, "gpu_launches": l_t2,
                      "includes": "as train_step, but dgrad / wgrad GEMMs as one TF32 MMA per MAC (forward stays 3xTF32)",
                      "loss_after": float(md2.loss)}
        del md2
        torch.cuda.empty_cache()

    # ---- N=1 extras: the reference's own GPU path on the same tensors, the descriptor path, the CPU baseline
    ref_gpu = desc = cb = None
    if rank == 0 and world == 1:
        if not args.no_descriptor:
            from tools import bench_descriptor
            desc = bench_descriptor.records(dev, pk if roof else peaks(), quick=True)
        if not args.no_reference_gpu:
            try:
                ref_gpu = reference_gpu_record(cfg, resident, P0, dev, ms / K, None if train is None else train["ms_per_step"])
            except Exception as e:                                  # the denominator is evidence, never a reason to lose the line
                ref_gpu = {"unavailable": "%s: %s" % (type(e).__name__, e)}
        if not args.no_cpu_baseline:
            # own interpreter: the CPU shim of the reference patches torch.cuda.* and cannot share a process with the GPU arm
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1"],
                               capture_output=True, text=True, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
            try:
                cb = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception:
                cb = {"unavailable": (r.stderr or r.stdout)[-300:]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {**_workload_config(cfg, world), "parallelism": "dp%d (independent ranks, no collective on fwd+loss)" % world,
                           "l2": "inputs rotate over %d distinct resident batches (%.0f MB > 126 MB L2); activations per step ~1.5 GB" % (nb, nb * h2d_bytes / 1e6),
                           "matmul_precision": "fp32 SIMT" if args.no_tc else "3xTF32 tcgen05 (fp32-equivalent) + fp32 SIMT for narrow layers",
                           "launch": "CUDA-graph replay of the step (ModelDetector.forward_loss(graph=True))" if use_graph else "eager"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches}
        if roof:
            line["roofline"] = roof
        if cb:
            line["cpu_baseline"] = cb
        if train:
            line["train_step"] = train
        if train_tf32:
            line["train_step_tf32_backward"] = train_tf32
        if ref_gpu:
            line["reference_gpu"] = ref_gpu
        if desc:
            line["descriptor"] = desc
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for k, v in outputs.items():
                np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
        print(json.dumps(line), flush=True)
    if world > 1:
        # the train-step graph holds the captured NCCL all-reduce: graphs first, then the communicator (usip_b200/dp.py);
        # the results are out, so a teardown that does not return within 20 s ends the process with status 0
        from usip_b200.dp import shutdown
        shutdown(md, hard_exit_after=20)


if __name__ == "__main__":
    main()
