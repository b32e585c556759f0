"""Time the fused BN-Inception extractor (extractor.py) at config-2 size and print ONE JSON line.

    python tools/bench_extractor.py [--batch 48 --length 3 --variant rgb] [--parent-lib OTHER/liboffk.so]

Reported, all with CUDA events after warm-up on the same card, whose name and power limit are read in the same run:
  * extractor:   the extractor pass alone (batch*length frames, inputs already on the device): the stock module with
                 allow_tf32 off and on, the fused plan in the fp32 (3xTF32) and tf32 modes (eager issue and graph replay);
                 algorithmic FLOP/s from the plan's shapes, and its share of the dense TF32 data-sheet rate (1125 TFLOP/s);
  * from_images: the full fwd+bwd training step from pinned host images, measured like bench.py's e2e_from_images
                 (copy, model forward, CE loss on the 7x7 and 14x14 heads, backward, loss read back), for both backbones;
  * maxpool28:   with --parent-lib (a liboffk.so that still exports offk_maxpool3s2_fwd): the config-2 OFF training step
                 with motion_pool_trans_28 on offk_pool3_nhwc and on offk_maxpool3s2_fwd, alternating, and whether the two
                 kernels write bit-identical pooled features from the same input.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                       # noqa: E402
import torch.nn.functional as F    # noqa: E402

TF32_DENSE = 1125e12               # HGX B200 data sheet, per GPU, dense, at 1000 W


def _timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def _card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else None
    except Exception as e:         # the numbers stay valid without it; say why it is missing
        out["power_limit_and_max_sm_clock"] = "unavailable: " + repr(e)[:100]
    return out


def extractor_times(n, cin, iters, warmup, dev):
    from off_b200.backbone import BNInceptionBackbone
    from off_b200.extractor import FusedBNInception
    x = torch.randn(n, cin, 224, 224, device=dev)
    res = {}
    stock = BNInceptionBackbone(101, cin).to(dev)
    torch.backends.cudnn.benchmark = True
    for name, tf32 in (("stock_fp32", False), ("stock_tf32", True)):
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = tf32
        res[name] = {"ms": _timed(lambda: stock(x), iters, warmup)}
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    del stock
    for prec in ("fp32", "tf32"):
        fx = FusedBNInception(101, cin, n, prec, dev)
        flops = fx.plan.flops_fwd
        for graph in (False, True):
            fx.use_graphs = graph
            ms = _timed(lambda: fx(x), iters, warmup)
            res[f"fused_{prec}" + ("_graph" if graph else "")] = {
                "ms": ms, "tflops": flops / (ms * 1e-3) / 1e12, "share_of_dense_tf32": flops / (ms * 1e-3) / TF32_DENSE}
        res["gflop_per_pass"] = flops / 1e9
        del fx
        torch.cuda.empty_cache()
    return res


def from_images(B, Lg, variant, backbone, precision, iters, warmup, dev):
    from off_b200.models import BNInception_OFF
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
    full = BNInception_OFF(101, B, Lg, variant=variant, backbone=backbone, precision=precision, device=dev).train()
    cin = 10 if variant == "flow" else 3
    img_host = torch.randn(B * Lg, cin, 224, 224).pin_memory()
    n_out = B * (Lg - 1) if variant == "rgb" else B
    target = torch.randint(0, 101, (n_out,), device=dev)
    loss_host = torch.zeros((), pin_memory=True)

    def istep():
        x = img_host.to(dev, non_blocking=True)
        out = full.RGB_OFF_forward(x) if variant == "rgb" else full(x)
        loss = F.cross_entropy(out[0], target) + F.cross_entropy(out[2], target)
        loss.backward()
        loss_host.copy_(loss.detach(), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms = _timed(istep, iters, warmup)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    del full
    torch.cuda.empty_cache()
    return {"ms_per_step": ms, "clips_per_s": B / (ms * 1e-3)}


def maxpool28_ab(B, Lg, precision, parent_lib, iters, warmup, rounds, dev):
    """The OFF training step with the maxpool28 launch on either kernel; the rest of the plan is the same object."""
    from off_b200 import _lib as L, plan as PL, spec as S
    from off_b200.modules import OFFSubNetwork
    import off_oracle as O
    old = C.CDLL(parent_lib)
    old.offk_maxpool3s2_fwd.restype = C.c_int
    old.offk_maxpool3s2_fwd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    net = OFFSubNetwork(B, Lg, "rgb", precision=precision, device=dev)
    eng = net.engine
    i = [k for k, st in enumerate(eng.fwd_sched.steps) if PL._names(st) == ["maxpool28"]][0]
    new_step = eng.fwd_sched.steps[i]
    f14, p28, P = eng.buf["F14"], eng.buf["p28"], eng.P

    def old_fn(stream):
        L.check(old.offk_maxpool3s2_fwd(PL._ptr(f14), P, 256, 14, 14, 1056, 800, PL._ptr(p28), stream), "maxpool3s2")
    old_step = PL._nm(old_fn, "maxpool28", reads=new_step.reads, writes=new_step.writes, lane=new_step.lane)
    taps = {k: v.to(dev) for k, v in O.make_taps(3, B, Lg).items()}
    target = torch.randint(0, 101, (B * (Lg - 1),), device=dev)

    def use(step):
        eng.fwd_sched.steps[i] = step

    # both kernels on the same F14 (the stage convs before it use split-K with fp32 atomics, so two forwards differ in the
    # last bits whatever the pool kernel; the pool itself must be exact)
    net.eval()
    with torch.no_grad():
        net(taps)
    torch.cuda.synchronize()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    new_step(stream)
    got_new = p28.clone()
    old_step(stream)
    torch.cuda.synchronize()
    same = torch.equal(got_new, p28)
    net.train()

    def tstep():
        fc7, _, fc14 = net(taps)
        (F.cross_entropy(fc7, target) + F.cross_entropy(fc14, target)).backward()
    times = {"pool3_nhwc": [], "maxpool3s2": []}
    for _ in range(rounds):
        for name, step in (("pool3_nhwc", new_step), ("maxpool3s2", old_step)):
            use(step)
            times[name].append(_timed(tstep, iters, warmup))
    use(new_step)
    return {"precision": precision, "bit_identical_pool_outputs": same, "ms_per_step": times,
            "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()}}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batch", type=int, default=48)
    ap.add_argument("--length", type=int, default=3)
    ap.add_argument("--variant", default="rgb", choices=["rgb", "flow"])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--parent-lib", default=None, help="a liboffk.so exporting offk_maxpool3s2_fwd, for the maxpool28 A/B")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_extractor.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import off_b200  # noqa: F401
    dev = torch.device("cuda")
    torch.manual_seed(0)
    B, Lg = a.batch, a.length
    cin = 10 if a.variant == "flow" else 3
    out = {"card": _card(), "frames": B * Lg, "variant": a.variant}
    out["extractor"] = extractor_times(B * Lg, cin, a.iters, a.warmup, dev)
    out["from_images"] = {f"{bb}_{p}": from_images(B, Lg, a.variant, bb, p, a.iters, a.warmup, dev)
                          for bb in ("bninception", "bninception_fused") for p in ("fp32", "tf32")}
    if a.parent_lib:
        out["maxpool28"] = [maxpool28_ab(B, Lg, p, a.parent_lib, a.iters, a.warmup, 3, dev) for p in ("fp32", "tf32")]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
