#!/usr/bin/env python
"""OFF-unit throughput benchmark (BASELINE.json metric: OFF-unit clips/sec, fwd+bwd; stencil HBM GB/s vs peak).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path (default: BASELINE config 2)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port) on the host cores
    python bench.py --impl eager_cuda ...                    # the reference's ATen/cuDNN ops in torch-eager CUDA on one B200
    python bench.py --config 4 --gpus N                      # BASELINE config 4: 128 clips x 7 segments split over N ranks

A "step" is one forward+backward of the OFF sub-network (RGB_OFF.py:596-860) over one batch of synthetic
BN-Inception taps: config 2 of BASELINE.json (RGB variant, 48 clips x 3 segments per GPU, fp32, train-mode dropout,
cross-entropy on the 7x7 and 14x14 heads as in train_off.py:136-146).  The default arithmetic is the fp32-parity mode on
the tensor cores (3xTF32, --precision fp32); the single-MMA tf32 mode is reported beside it (`tf32_mode`).  For N > 1
every rank processes its own 48 clips (weak scaling; config 4: a fixed 128 clips split over the ranks, strong scaling)
and the OFF-parameter gradients are averaged with a bucketed NCCL all-reduce per step.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "off_unit_clips_per_sec_fwd_bwd"
# dram__bytes_read.sum + dram__bytes_write.sum of the forward stencil launches of one step, from the committed
# ncu --set full capture (profiles/ncu_full_r01t_stencil_summary.txt: read 227.8 MB + write 59.0 MB; 156 MB are written,
# the rest is still dirty in L2 at kernel end)
NCU_STENCIL_TRAFFIC_BYTES = 286.8e6
UNIT = "clips/s"
NOMINAL_HBM_GBS = 8000.0          # north_star: "about 8 TB/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager_cuda"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json config: 2 = RGB 48x3 per GPU (default), 3 = Flow 48x3 per GPU, 4 = RGB 128x7 split over the ranks")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (0 = the config's)")
    ap.add_argument("--length", type=int, default=0, help="segments per clip (0 = the config's)")
    ap.add_argument("--variant", default="", choices=["", "rgb", "flow"])
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32"],
                    help="fp32 = fp32-parity mode on the tensor cores (3xTF32, the BASELINE config-2 arithmetic); tf32 = one "
                         "kind::tf32 MMA per product (stated separately)")
    ap.add_argument("--cpu-clips", type=int, default=0, help="clips per CPU-baseline step (0 = the GPU arm's batch, capped at 48)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the torch-eager CUDA baseline legs")
    ap.add_argument("--no-families", action="store_true", help="skip the per-kernel-family roofline pass")
    ap.add_argument("--no-graphs", action="store_true", help="issue every kernel from the host instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step returned (logits, loss, OFF-parameter "
                         "gradients) as DIR/<name>.npy in float32, to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.config == 4:
        a.variant = a.variant or "rgb"
        a.length = a.length or 7
        a.global_batch = 128
        a.batch = a.batch or max(1, 128 // world)
        a.scaling = "strong"
    else:
        a.variant = a.variant or ("flow" if a.config == 3 else "rgb")
        a.length = a.length or 3
        a.batch = a.batch or 48
        a.global_batch = a.batch * world
        a.scaling = "weak"
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# element data of one --dump-outputs directory; the .npy headers come on top and the files stay under 64 MB in all
DUMP_DATA_BYTES = 60_000_000


def dump_outputs(out_dir, arrays):
    """Write each array as ``out_dir/<name>.npy`` in float32.  Smaller arrays are written whole first; an array larger
    than its share of what is left of DUMP_DATA_BYTES is replaced by a fixed seeded sample of its flattened elements
    (the same indices for the same shapes, so two runs stay comparable element for element)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left, n_left = DUMP_DATA_BYTES // 4, len(arrays)
    for name, a in sorted(arrays.items(), key=lambda kv: kv[1].size):
        a = np.asarray(a, dtype=np.float32)
        share = left // n_left
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left, n_left = left - a.size, n_left - 1


def workload(args):
    return (f"{args.variant.upper()}_OFF OFF sub-network fwd+bwd, {args.batch} clips x {args.length} segments per GPU "
            f"(BASELINE config {args.config}), train-mode dropout, CE loss on the 7x7 and 14x14 heads")


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_oracle_rate(clips: int, length: int, variant: str, steps: int, warmup: int):
    """The reference's CPU path for this hot path (oracle port: the same ATen ops the reference modules call,
    RGB_OFF.py:596-860), fp32, all host threads, fwd+bwd with the same loss.  Returns (clips/s, s/step, threads)."""
    import torch
    import torch.nn.functional as F
    import off_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    taps = O.make_taps(3, clips, length)
    prm = O.make_params(3, variant)
    masks = O.make_dropout_masks(3, clips, length)
    pairs = clips * (length - 1)
    tgt = torch.arange(pairs) % O.NUM_CLASSES
    if variant != "rgb":
        tgt = tgt[:clips]

    def loss(o):
        return F.cross_entropy(o["fc7"].reshape(len(tgt), -1), tgt) + F.cross_entropy(o["fc14"].reshape(len(tgt), -1), tgt)

    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.off_forward_backward(taps, prm, clips, length, variant, masks, torch.float32, loss=loss)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return clips / sec, sec, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the driver's step count is honoured up to a bound that keeps the run within a few minutes (~0.5-1 s per step)
    steps, warmup = max(1, min(args.steps, 40)), max(1, min(args.warmup, 3))
    clips = args.cpu_clips or min(args.batch, 48)
    rate, sec, threads = cpu_oracle_rate(clips, args.length, args.variant, steps, warmup)
    sample = (f"{clips} clips x {args.length} segments per step, fp32, {steps} timed steps after {warmup} "
              f"warm-up ({sec:.2f} s/step)")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": workload(args) + "; CPU arm: a bounded number of steps over " + sample, "sample": sample},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- torch-eager CUDA arm
def eager_cuda_rate(clips: int, length: int, variant: str, allow_tf32: bool, steps: int, warmup: int, device):
    """The honest GPU baseline (SURVEY 2a / 8d): the reference's own ATen / cuDNN ops (the oracle restatement of
    RGB_OFF.py:596-860, which calls exactly the operators the reference modules call) in torch-eager CUDA on one B200,
    same batch, same loss, fwd+bwd, fp32 storage; allow_tf32 toggles cuDNN / cuBLAS TF32.  Returns (clips/s, ms/step)."""
    import torch
    import torch.nn.functional as F
    import off_oracle as O
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = bool(allow_tf32)
    torch.backends.cudnn.benchmark = True
    try:
        g = torch.Generator(device=device).manual_seed(3)
        taps = {t: torch.relu(torch.randn(clips * length, cin, s, s, device=device, generator=g)) for t, (cin, s) in O.LEVELS.items()}
        prm = {k: v.to(device).requires_grad_(True) for k, v in O.make_params(3, variant).items()}
        pairs = clips * (length - 1)
        masks = {t: (torch.rand(pairs, O.DOWN_C, s, s, device=device, generator=g) >= 0.8).to(torch.uint8) for t, (_, s) in O.LEVELS.items()}
        for k, c in (("fc28", 256), ("fc14", 512), ("fc7", 1024)):
            masks[k] = (torch.rand(pairs, c, device=device, generator=g) >= 0.8).to(torch.uint8)
        n_out = pairs if variant == "rgb" else clips
        tgt = torch.arange(n_out, device=device) % O.NUM_CLASSES
        plist = list(prm.values())

        def step():
            out = O.off_forward(taps, prm, clips, length, variant, masks)
            loss = F.cross_entropy(out["fc7"].reshape(n_out, -1), tgt) + F.cross_entropy(out["fc14"].reshape(n_out, -1), tgt)
            torch.autograd.grad(loss, plist, allow_unused=True)      # fc_action_motion_28 receives none (RGB_OFF.py:860)

        for _ in range(warmup):
            step()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        torch.cuda.synchronize(device)
        ms = a.elapsed_time(b) / steps
        return clips / (ms * 1e-3), ms
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old


def run_eager(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    out = {}
    for name, tf32 in (("fp32", False), ("tf32", True)):
        rate, ms = eager_cuda_rate(args.batch, args.length, args.variant, tf32, max(3, args.steps), max(3, args.warmup), dev)
        out[name] = {"value": rate, "ms_per_step": ms}
    key = args.precision
    line = {"impl": "eager_cuda", "metric": METRIC, "value": out[key]["value"], "unit": UNIT, "n_gpus": 1, "steps": max(3, args.steps),
            "warmup": max(3, args.warmup), "ms_per_step": out[key]["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "fp32 (cuDNN/cuBLAS, allow_tf32=%s)" % (key == "tf32"), "data": "synthetic",
            "config": {"workload": workload(args) + "; torch-eager CUDA (ATen/cuDNN) of the reference's operators on one B200"},
            "gpu_baseline": out}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------------------------- rooflines
def _family(name):
    """Kernel family of one plan step (by its launch name)."""
    from off_b200 import spec as S
    base = name.split(".")[0]
    if name.startswith("stencil_fwd"):
        return "stencil_fwd"
    if name.startswith("stencil_bwd"):
        return "stencil_bwd"
    if base.startswith("unit_") or base.startswith("tapT_"):
        return "unit_wgrad" if ".wgrad" in name else ("unit_dgrad" if ".dgrad" in name else "unit_gemm")
    if ".wgrad" in name:
        return "wgrad"
    k = S.CONV_BY_NAME[base][3] if base in S.CONV_BY_NAME else 1
    if ".dgrad" in name:
        return "kxk_dgrad" if k > 1 else "1x1_dgrad"
    if base in S.CONV_BY_NAME:
        return "kxk_fwd" if k > 1 else "1x1_fwd"
    if base.startswith("fc_action"):
        return "1x1_fwd"
    return "glue"


def family_rooflines(eng, pk, precision, reps=3):
    """Per-kernel-family time inside a step and its roofline: every plan step issued on ONE stream with CUDA events
    around it (so concurrency between lanes is removed: these are kernel times, their sum exceeds the step time),
    inputs as the preceding kernels left them (in-step cache state).  GEMM families: algorithmic FLOPs 2*M*N*K of the
    contractions / time against the dense TF32 peak (= half the measured bf16 figure; the fp32 mode issues three MMAs
    per product, so its fraction of the MMA peak is 3x the algorithmic one).  Unit GEMMs and stencils: compulsory bytes /
    time against the measured HBM copy bandwidth."""
    import torch
    from off_b200 import spec as S
    from off_b200.engine import _names
    was = eng.single_stream
    eng.single_stream = True
    h = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fam = {}
    for r in range(reps + 1):
        eng._set_dropout(True, None, 1 + r)
        evs = []
        for sched in (eng.fwd_sched, eng.bwd_sched):
            for stp in sched.steps:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                stp(h)
                b.record()
                evs.append((stp, a, b))
        torch.cuda.synchronize()
        if r == 0:
            continue                                              # warm-up pass
        for stp, a, b in evs:
            name = getattr(stp, "name", None) or _names(stp)[0]
            f = fam.setdefault(_family(name), {"us": 0.0, "flops": 0.0, "launches": 0})
            f["us"] += a.elapsed_time(b) * 1e3 / reps
            if r == 1:
                f["flops"] += float(getattr(stp, "flops", 0.0))
                f["launches"] += len([n for n in _names(stp) if not (n.endswith(".zero") or n.startswith("zero "))])
    eng.single_stream = was
    tf32_peak = 0.5 * pk["bf16_tflops"]
    N, P = eng.N, eng.P
    unit_bytes = sum(4.0 * (N * cin * s * s + N * S.UNIT_C * s * s + S.UNIT_C * cin) for cin, s in S.LEVELS.values())
    unit_wgrad_bytes = sum(4.0 * (N * cin * s * s + N * S.UNIT_C * s * s + S.UNIT_C * cin) for cin, s in S.LEVELS.values())
    st_fwd = sum(4.0 * s * s * (S.GEN_C * N + S.DOWN_C * P + S.UNIT_C * P) for _, s in S.LEVELS.values())
    st_bwd = sum(4.0 * s * s * (S.UNIT_C * P + 2 * S.GEN_C * N + S.DOWN_C * P) for _, s in S.LEVELS.values())
    bytes_of = {"unit_gemm": unit_bytes, "unit_wgrad": unit_wgrad_bytes, "stencil_fwd": st_fwd, "stencil_bwd": st_bwd}
    out = {}
    for k, f in sorted(fam.items(), key=lambda kv: -kv[1]["us"]):
        e = {"us": round(f["us"], 1), "launches": f["launches"]}
        if f["flops"] > 0 and f["us"] > 0:
            tf = f["flops"] / (f["us"] * 1e-6) / 1e12
            e.update(gflop=round(f["flops"] / 1e9, 2), tflops=round(tf, 1), frac_tf32_peak=round(tf / tf32_peak, 3))
            if precision == "fp32":
                e["frac_tf32_peak_mma_issued"] = round(3 * tf / tf32_peak, 3)
        if k in bytes_of and f["us"] > 0:
            gbs = bytes_of[k] / (f["us"] * 1e-6) / 1e9
            e.update(MB=round(bytes_of[k] / 1e6, 1), GBs=round(gbs, 1), frac_hbm=round(gbs / pk["hbm_gbs"], 3),
                     frac_hbm_nominal_8TBs=round(gbs / NOMINAL_HBM_GBS, 3))
        out[k] = e
    return out, tf32_peak


def stencil_roofline(eng, pk, pk_src, dev):
    """The memory-bound kernel BASELINE.json names: the fused stencil.  Forward: one launch per stage group, timed cold
    (L2 evicted and written back before every launch) and in-step; backward: one launch for all nine units, cold."""
    import torch
    from off_b200 import spec as S
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_r = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
    flush_sink = torch.zeros((), dtype=torch.int64, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lvl_bytes = {t: 4.0 * s * s * (S.GEN_C * eng.N + S.DOWN_C * eng.P + S.UNIT_C * eng.P) for t, (cin, s) in S.LEVELS.items()}

    def evict():
        # evict L2 (126 MB): write a 256 MB buffer, then read a second one so that the evicted lines are written back
        # BEFORE the timed launch (dirty lines would otherwise drain during it)
        flush.fill_(1)
        flush_sink.add_(flush_r.view(torch.int64).sum())

    tot_ms, tot_bytes, per_stage = 0.0, 0.0, {}
    eng._set_dropout(True, None, 1)
    for st, step_fn in eng.stencil_fwd_steps.items():
        nbytes = sum(lvl_bytes[t] for t in eng.stencil_fwd_tags[st])
        reps, acc = 10, 0.0
        for _ in range(reps):
            evict()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_fn(stream)
            b.record()
            torch.cuda.synchronize()
            acc += a.elapsed_time(b)
        per_stage[st] = {"MB": round(nbytes / 1e6, 1), "us": round(acc / reps * 1e3, 1), "GBs": round(nbytes / (acc / reps * 1e-3) / 1e9, 1)}
        tot_ms += acc / reps
        tot_bytes += nbytes
    achieved = tot_bytes / (tot_ms * 1e-3) / 1e9
    bwd_bytes = sum(4.0 * s * s * (S.UNIT_C * eng.P + 2 * S.GEN_C * eng.N + S.DOWN_C * eng.P) for _, s in S.LEVELS.values())
    n_lv, acc = len(S.LEVELS), 0.0
    for _ in range(10):
        evict()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.lib.offk_stencil_diff_bwd_batch(n_lv, eng._st_desc, eng._st_io, stream)
        b.record()
        torch.cuda.synchronize()
        acc += a.elapsed_time(b)
    fused_us = acc / 10 * 1e3
    bwd_gbs = bwd_bytes / (fused_us * 1e-6) / 1e9
    return {"bound": "hbm", "kernel": f"stencil_diff_fwd_kernel ({len(per_stage)} launches per step: {' | '.join(per_stage)} stage units; 9 OFF units)",
            "achieved": achieved, "peak": pk["hbm_gbs"], "peak_source": pk_src, "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
            "frac_nominal_8TBs": achieved / NOMINAL_HBM_GBS, "traffic": NCU_STENCIL_TRAFFIC_BYTES, "bytes_per_step": tot_bytes,
            "per_stage": per_stage,
            "backward": {"MB": round(bwd_bytes / 1e6, 1), "us": round(fused_us, 1), "GBs": round(bwd_gbs, 1),
                         "frac": round(bwd_gbs / pk["hbm_gbs"], 3), "frac_nominal_8TBs": round(bwd_gbs / NOMINAL_HBM_GBS, 3),
                         "note": "stencil_diff_bwd_kernel, all nine units in one launch, cold L2"},
            "note": "algorithmic bytes 4*S^2*(128*N + 32*P + 160*P) per level (read G once, read D once, write the 160-channel "
                    "slice once); `achieved` = cold launches, L2 evicted before each; in-step figures: roofline_kernels.stencil_fwd / "
                    "stencil_bwd; traffic = ncu dram__bytes_read+write over the forward stencil launches of one step (profiles/)"}


# ----------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    import off_b200  # noqa: F401
    from off_b200 import spec as S
    from off_b200.modules import OFFSubNetwork
    from off_b200.dist import DataParallelOFF, bind_to_gpu_numa_node

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local)                  # before any pinned allocation: staging buffers on the GPU's node
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, Lg = args.batch, args.length
    graphs = not args.no_graphs
    # the initial weights, the taps and the per-step dropout seeds all follow from this seed: the same arguments give
    # the same inputs in every run
    torch.manual_seed(1234 + rank)
    net = OFFSubNetwork(B, Lg, args.variant, precision=args.precision, device=dev, use_graphs=graphs).train()
    eng = net.engine
    dp = DataParallelOFF(eng, use_graphs=graphs)
    dp.broadcast_parameters()
    taps_dev = net.tap_buffers()
    for t in taps_dev.values():
        t.copy_(torch.relu(torch.randn_like(t)))           # post-ReLU Inception taps (RGB_OFF.py:395)
    n_out = eng.P if not eng.consensus else B
    target = (torch.arange(n_out, device=dev) + rank) % S.NUM_CLASSES   # labels repeated per pair, train_off.py:133
    tap_bytes = sum(t.numel() * 4 for t in taps_dev.values())
    taps_host = {k: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for k, t in taps_dev.items()}
    loss_host = torch.empty((), dtype=torch.float32, pin_memory=True)

    def make_step(net, dp, keep=None):
        def step(inputs=None):
            """One forward+backward.  inputs = None: taps already resident in HBM (device-timed `value`);
            inputs = a prefetch handle: the end-to-end path (taps staged from pinned host memory, loss read back).
            keep: a dict that receives what the step returns to its caller (for --dump-outputs)."""
            fc7, fc28, fc14 = net(net.tap_buffers() if inputs is None else inputs)
            loss = F.cross_entropy(fc7, target) + F.cross_entropy(fc14, target)
            # backward through the module's autograd.Function; the OFF-parameter gradients land in the flat buffer
            g7, g14 = torch.autograd.grad(loss, [fc7, fc14])
            grads = dp.backward(g7, g14)
            if inputs is not None:
                loss_host.copy_(loss.detach(), non_blocking=True)
                torch.cuda.current_stream().synchronize()       # the user reads the loss every step
            if keep is not None:
                keep.update(fc7=fc7, fc28=fc28, fc14=fc14, loss=loss, grads=grads)
            return loss
        return step

    last = {} if args.dump_outputs else None
    step = make_step(net, dp, last)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step, net, n, e2e):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        if e2e:
            # public API: net.prefetch(host taps) starts the H2D copy of step i+1 into the idle input set while
            # step i computes; every step's tap copy and 4-byte loss read-back are inside the timed region
            h = net.prefetch(taps_host)
            for i in range(n):
                h_next = net.prefetch(taps_host) if i + 1 < n else None
                step(h)
                h = h_next
        else:
            for _ in range(n):
                step()
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for _ in range(max(3, args.warmup)):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(step, net, args.steps, False)
    sampler.stop_flag = True
    if last is not None and rank == 0:
        # before any further step: the gradients are views of the engine's flat buffer, which the next step overwrites
        out = {k: last[k].detach().cpu().numpy() for k in ("fc7", "fc28", "fc14", "loss")}
        out.update({"grad." + n: g.cpu().numpy() for n, g in last["grads"].items()})
        dump_outputs(args.dump_outputs, out)
    timed(step, net, 2, True)                                 # warm the staged path
    n_e2e = max(3, args.steps // 2)
    ms_e2e = timed(step, net, n_e2e, True) / n_e2e * args.steps

    clips_total = B * world * args.steps
    value = clips_total / (ms * 1e-3)
    e2e_value = clips_total / (ms_e2e * 1e-3)

    pk, pk_src = peaks()
    roof = families = None
    tf32_peak = 0.5 * pk["bf16_tflops"]
    if rank == 0:
        stencil = stencil_roofline(eng, pk, pk_src, dev)
        if not args.no_families:
            families, tf32_peak = family_rooflines(eng, pk, args.precision)
            for k in ("stencil_fwd", "stencil_bwd"):
                if k in families:
                    families[k]["cold"] = ({"GBs": round(stencil["achieved"], 1), "frac_hbm": round(stencil["frac"], 3)} if k == "stencil_fwd"
                                           else {"GBs": stencil["backward"]["GBs"], "frac_hbm": stencil["backward"]["frac"]})
            dom = next(k for k in families if "tflops" in families[k])          # families are sorted by time
            d = families[dom]
            roof = {"bound": "tensor", "kernel": f"{dom} family ({d['launches']} launches per step, {d['us']} us of kernel time)",
                    "achieved": d["tflops"], "peak": tf32_peak, "unit": "TFLOP/s", "frac": d["frac_tf32_peak"],
                    "peak_source": f"dense TF32 = 0.5 x {pk_src} bf16 burst ({pk['bf16_tflops']} TFLOP/s)", "traffic": None,
                    "note": "the dominant kernel family of the step; algorithmic FLOPs 2*M*N*K of its contractions / its in-step "
                            "kernel time (CUDA events, single-stream issue)" +
                            ("; the fp32 mode issues 3 kind::tf32 MMAs per product (3xTF32): fraction of the MMA peak actually "
                             f"issued = {d.get('frac_tf32_peak_mma_issued')}" if args.precision == "fp32" else "")}
        else:
            roof = stencil

    # ---- the other precision mode, stated separately (same shapes, same loss; bounded: 10 steps)
    other = None
    if rank == 0 and world == 1:
        oprec = "tf32" if args.precision == "fp32" else "fp32"
        del step
        net2 = OFFSubNetwork(B, Lg, args.variant, precision=oprec, device=dev, use_graphs=graphs).train()
        net2.engine.params_flat.copy_(eng.params_flat)
        for k, t in net2.tap_buffers().items():
            t.copy_(taps_dev[k])
        step2 = make_step(net2, DataParallelOFF(net2.engine, use_graphs=graphs))
        for _ in range(3):
            step2()
        ms2 = timed(step2, net2, 10, False) / 10
        other = {"precision": oprec, "value": B / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2,
                 "dtype": "tf32 (one tcgen05 kind::tf32 MMA per product, fp32 accumulate)" if oprec == "tf32" else "fp32 (3xTF32)",
                 "tolerance": "tests/test_gpu_parity.py: tf32 <= 5e-3 of the tensor max per level, 1e-2 on logits (fp32 mode: 2e-5 / 5e-5)"}
        del net2, step2
        torch.cuda.empty_cache()

    gpu_base = None
    if rank == 0 and world == 1 and not args.no_gpu_baseline:
        gpu_base = {}
        for name, tf32 in (("fp32", False), ("tf32", True)):
            try:
                rate, ms_b = eager_cuda_rate(B, Lg, args.variant, tf32, 10, 5, dev)
                gpu_base[name] = {"value": rate, "unit": UNIT, "ms_per_step": ms_b}
            except Exception as e:                          # e.g. out of memory at a large custom batch: report, do not die
                gpu_base[name] = {"error": repr(e)[:200]}
        gpu_base["what"] = ("torch-eager CUDA (ATen/cuDNN, cudnn.benchmark) of the reference's operators (RGB_OFF.py:596-860 via the "
                            "oracle restatement), same batch, loss and fwd+bwd on this B200; fp32 = allow_tf32 off, tf32 = on")
        torch.cuda.empty_cache()

    # ---- deployment shape of the boundary (extra, N = 1): IMAGES from pinned host memory through the built-in frozen
    # BN-Inception extractor (stock cuDNN ops, out of the accelerated scope) into the OFF path -- the taps never cross PCIe
    from_images = None
    if rank == 0 and world == 1 and not args.no_gpu_baseline:
        try:
            from off_b200.models import BNInception_OFF
            old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = (args.precision == "tf32")
            full = BNInception_OFF(S.NUM_CLASSES, B, Lg, variant=args.variant, backbone="bninception", precision=args.precision,
                                   device=dev).train()
            cin = 10 if args.variant == "flow" else 3
            img_host = torch.randn(B * Lg, cin, 224, 224).pin_memory()

            def istep():
                x = img_host.to(dev, non_blocking=True)
                out = full.RGB_OFF_forward(x) if args.variant == "rgb" else full(x)
                loss = F.cross_entropy(out[0], target) + F.cross_entropy(out[2], target)
                loss.backward()
                loss_host.copy_(loss.detach(), non_blocking=True)
                torch.cuda.current_stream().synchronize()
            for _ in range(3):
                istep()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                istep()
            b.record()
            torch.cuda.synchronize()
            ims = a.elapsed_time(b) / 10
            from_images = {"value": B / (ims * 1e-3), "unit": UNIT, "ms_per_step": ims, "h2d_bytes_per_step": img_host.numel() * 4,
                           "note": "full model: images copied from pinned host memory, frozen BN-Inception extractor on stock cuDNN ops "
                                   f"(allow_tf32={args.precision == 'tf32'}), OFF fwd+bwd on liboffk, loss read back; the extractor is "
                                   "outside the accelerated scope (SURVEY 8f-2)"}
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
            del full
            torch.cuda.empty_cache()
        except Exception as e:
            from_images = {"error": repr(e)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # the CPU baseline is timed at N = 1 only
        clips = args.cpu_clips or min(B, 48)
        rate, sec, threads = cpu_oracle_rate(clips, Lg, args.variant, 6, 1)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{clips} clips x {Lg} segments, fwd+bwd, fp32, 6 timed steps after 1 warm-up ({sec:.2f} s/step)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": ("tf32 (tcgen05 kind::tf32 multiply, fp32 accumulate, fp32 storage)" if args.precision == "tf32" else
                      "fp32 (3xTF32: error-compensated tcgen05 kind::tf32 MMAs, fp32 accumulate, fp32 storage)"),
            "data": "synthetic",
            "config": {"workload": workload(args), "clips_per_gpu": B, "segments": Lg, "precision": args.precision,
                       "global_clips": B * world,
                       "l2": f"inputs larger than L2: {tap_bytes / 1e6:.0f} MB of taps per step vs 126 MB L2",
                       "parallelism": f"dp{world} (clip-sharded, NCCL all-reduce of {eng.n_flat} fp32 gradients)",
                       "numa": numa,
                       "issue": ("forward and backward replayed as one captured CUDA graph each (multi-stream capture of the plan)"
                                 if graphs else "every kernel issued from the host") + ("; gradient all-reduce buckets issued eagerly "
                                 "between the unit weight-gradient kernels" if world > 1 else "")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": tap_bytes, "d2h_bytes_per_step": 4,
                    "note": "taps copied from pinned host memory every step (copy of step i+1 overlaps compute of step i: "
                            "two input sets), loss read back every step"},
            "gpu_launches": (eng.launches_fwd + eng.launches_bwd) * args.steps,
            "clocks": sampler.summary(),
            "roofline": roof,
            "roofline_kernels": families,
            "roofline_stencil": stencil if not args.no_families else None,
            "cpu_baseline": cpu,
            "gpu_baseline": gpu_base,
            "e2e_from_images": from_images,
            ("tf32_mode" if args.precision == "fp32" else "fp32_mode"): other,
            "flops_per_step": {"fwd": eng.flops_fwd, "bwd": eng.flops_bwd,
                               "tflops_achieved": (eng.flops_fwd + eng.flops_bwd) / (ms / args.steps * 1e-3) / 1e12,
                               "frac_tf32_peak": (eng.flops_fwd + eng.flops_bwd) / (ms / args.steps * 1e-3) / 1e12 / tf32_peak},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "eager_cuda":
        run_eager(a)
    else:
        run_ours(a)
