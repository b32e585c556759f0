"""Pin the oracle against the REAL reference and write tests/golden/*.npz.

Needs a checkout of the reference repository (JoeHEZHAO/Optical-Flow-Guided-Feature-Pytorch),
read-only.  The reference classes are imported unmodified; the OFF section is isolated with
forward-pre-hooks that replace the inputs of the 18 tap consumers
(SURVEY.md section 8c): ``motion_conv_gen_X <- taps[X]`` and
``motion_spatial_down_X <- taps[X][:B*(L-1)]`` (mirrors RGB_OFF.py:609).
Shims applied at run time, never by editing the reference:
  * ``consensus``  -> ``x.mean(1, keepdim=True)`` (basic_ops.py:22; the legacy
    autograd.Function no longer runs on torch >= 1.5),
  * ``dropout``    -> a module replaying injected keep-masks in call order
    (RGB_OFF.py:612,632,651,701,719,737,755,785,791,809,827,845).

Usage:  python oracle/make_golden.py REFERENCE_DIR      (writes tests/golden/*)
"""
from __future__ import annotations

import os
import sys
from collections import OrderedDict

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import off_oracle as O  # noqa: E402

REF = ""                      # the reference checkout, from the command line
GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")

DROP_ORDER = ["3a", "3b", "3c", "4a", "4b", "4c", "4d", "fc28", "fc14", "5a", "5b", "fc7"]


class _Mean(torch.nn.Module):
    def forward(self, x):
        return x.mean(dim=1, keepdim=True)


class _ReplayDropout(torch.nn.Module):
    def __init__(self, masks, p):
        super().__init__()
        self.masks, self.p, self.i = masks, p, 0

    def forward(self, x):
        m = self.masks[DROP_ORDER[self.i]]
        self.i += 1
        return x * m.to(x.dtype).reshape(x.shape) / (1.0 - self.p)


def run_reference(variant, batch, length, taps, prm, masks=None, dtype=torch.float32, backward=True):
    sys.path.insert(0, REF)
    import importlib
    mod = importlib.import_module({"rgb": "RGB_OFF", "flow": "Flow_OFF", "v2": "RGB_OFF_v2"}[variant])
    net = mod.bninception_off(O.NUM_CLASSES, batch, length)
    net.eval()
    sd = net.state_dict()
    for k, v in prm.items():
        assert sd[k].shape == v.shape, (k, sd[k].shape, v.shape)
    net.load_state_dict({**sd, **prm})
    net = net.to(dtype)
    if variant != "rgb":
        net.consensus = _Mean()
    if masks is not None:
        net.dropout = _ReplayDropout(masks, 0.8)
    for p in net.parameters():
        p.requires_grad_(False)
    for n, p in net.named_parameters():
        if "motion" in n:                       # train_off.py:40
            p.requires_grad_(True)
    pairs = batch * (length - 1)
    taps = OrderedDict((k, v.to(dtype)) for k, v in taps.items())
    caught = {}
    hooks = []
    for tag in O.LEVELS:
        hooks.append(getattr(net, "motion_conv_gen_" + tag).register_forward_pre_hook(
            lambda m, inp, t=tag: (taps[t],)))
        hooks.append(getattr(net, "motion_spatial_down_" + tag).register_forward_pre_hook(
            lambda m, inp, t=tag: (taps[t][:pairs],)))
    for name, key in (("motion_conv_trans_28", "fusion28"), ("motion_conv_trans_14", "fusion14"),
                      ("motion_conv_trans", "fusion7")):
        hooks.append(getattr(net, name).register_forward_pre_hook(
            lambda m, inp, k=key: caught.__setitem__(k, inp[0].detach())))
    hooks.append(net.fc_action_motion_28.register_forward_hook(
        lambda m, inp, out: caught.__setitem__("fc28_pairs", out.detach())))
    cin = 10 if variant == "flow" else 3
    dummy = torch.zeros(batch * length, cin, 224, 224, dtype=dtype)
    fwd = net.RGB_OFF_forward if variant == "rgb" else net.forward
    res = fwd(dummy)
    fc7, fc14 = res[0], res[2]
    grads = None
    if backward:
        (fc7.sum() + fc14.sum()).backward()
        grads = OrderedDict()
        for n, p in net.named_parameters():
            if n in prm:
                grads[n] = (p.grad if p.grad is not None else torch.zeros_like(p)).detach()
    for h in hooks:
        h.remove()
    out = dict(fc7=fc7.detach(), fc14=fc14.detach(), **caught)
    return out, grads


def digest(t: torch.Tensor, n=64):
    t = t.detach().double().reshape(-1)
    idx = torch.linspace(0, t.numel() - 1, min(n, t.numel())).long()
    return dict(sum=float(t.sum()), abssum=float(t.abs().sum()), l2=float(t.norm()),
                idx=idx.numpy(), val=t[idx].numpy())


CASES = [
    # name, variant, batch, length, train-mode masks?
    ("rgb_b1_l3", "rgb", 1, 3, False),      # BASELINE config 1 geometry
    ("rgb_b2_l3", "rgb", 2, 3, False),      # exercises the flat-index quirk (SURVEY 3.3)
    ("flow_b2_l3", "flow", 2, 3, False),    # diagonal Sobel + consensus
    ("rgb_b2_l2_train", "rgb", 2, 2, True), # injected dropout masks
    ("flow_b1_l4", "flow", 1, 4, False),
    ("v2_b2_l3", "v2", 2, 3, False),        # RGB_OFF_v2: Flow's graph on RGB input (4-tuple return, RGB_OFF_v2.py:891)
    ("rgb_b1_l2", "rgb", 1, 2, False),      # ONE frame pair: torch.squeeze drops the batch dimension too (RGB_OFF.py:786,792,846)
]


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    report = []
    for name, variant, batch, length, train in CASES:
        seed = 1 + CASES.index((name, variant, batch, length, train))
        taps = O.make_taps(seed, batch, length)
        prm = O.make_params(seed, variant)
        masks = O.make_dropout_masks(seed, batch, length) if train else None
        ref64, g64 = run_reference(variant, batch, length, taps, prm, masks, torch.float64)
        ref32, g32 = run_reference(variant, batch, length, taps, prm, masks, torch.float32)
        ora64, og64 = O.off_forward_backward(taps, prm, batch, length, variant, masks, torch.float64)
        ora32, og32 = O.off_forward_backward(taps, prm, batch, length, variant, masks, torch.float32)

        # -- pin: restatement == reference (fp64 exact to 1e-12 rel, fp32 to round-off)
        def cmp(a, b):
            return float((a.double() - b.double()).abs().max()), float(b.double().abs().max())
        worst = 0.0
        for k in ("fc7", "fc14", "fusion28", "fusion14", "fusion7"):
            e, s = cmp(ora64[k].reshape(ref64[k].shape), ref64[k])
            assert e <= 1e-10 * max(s, 1.0), (name, k, e, s)
            e32, _ = cmp(ora32[k].reshape(ref32[k].shape), ref32[k])
            assert e32 <= 2e-5 * max(s, 1.0), (name, k, e32, s)
            worst = max(worst, e32 / max(s, 1.0))
        fc28_ref = ref64["fc28_pairs"]
        if variant != "rgb":
            fc28_ref = fc28_ref.view(batch, length - 1, -1).mean(1)
        e, s = cmp(ora64["fc28"].reshape(fc28_ref.shape), fc28_ref)
        assert e <= 1e-10 * max(s, 1.0), (name, "fc28", e)
        for k in g64:
            e, s = cmp(og64[k], g64[k])
            assert e <= 1e-9 * max(s, 1.0), (name, "grad " + k, e, s)
        zero_grad = [k for k in g64 if float(g64[k].abs().max()) == 0.0]
        assert sorted(zero_grad) == ["fc_action_motion_28.bias", "fc_action_motion_28.weight"], zero_grad
        # fp32 reference noise floor vs fp64 (what "fp32 parity" can mean at best)
        floor = {k: cmp(ref32[k], ref64[k])[0] for k in ("fc7", "fc14", "fusion28", "fusion14", "fusion7")}

        fix = dict(variant=variant, batch=batch, length=length, seed=seed, train=int(train))
        for k in ("fc7", "fc14"):
            fix[k] = ref64[k].numpy()
        fix["fc28"] = fc28_ref.numpy()
        for k in ("fusion28", "fusion14", "fusion7"):
            d = digest(ref64[k], 256)
            for kk, vv in d.items():
                fix[f"{k}.{kk}"] = vv
            fix[f"{k}.fp32_floor"] = floor[k]
        for k, g in g64.items():
            d = digest(g, 32)
            for kk, vv in d.items():
                fix[f"grad.{k}.{kk}"] = vv
        np.savez_compressed(os.path.join(GOLD, f"off_{name}.npz"), **fix)
        report.append((name, worst, floor))
        print(f"[golden] {name}: oracle==reference (fp32 rel err {worst:.2e}); fp32-vs-fp64 floor {floor}")

    # -- known-answer vectors for the fixed stencils (util.py:29-30,61), computed with the reference classes
    sys.path.insert(0, REF)
    import util as RU
    x = torch.arange(5.0).repeat(5, 1).view(1, 1, 5, 5)
    gx, gy = RU.SobelFilter(1, 1)(x)
    gd = RU.SobelFilter_Diagonal(1, 1)(x)
    ox, oy = O.sobel_xy(x)
    assert torch.equal(gx, ox) and torch.equal(gy, oy) and torch.equal(gd, O.sobel_diagonal(x))
    xr = O.hash_normal(99, (2, 4, 9, 7))
    rx, ry = RU.SobelFilter(4, 4)(xr)
    rd = RU.SobelFilter_Diagonal(4, 4)(xr)
    np.savez_compressed(os.path.join(GOLD, "sobel_kat.npz"), ramp_gx=gx.detach().numpy(), ramp_gy=gy.detach().numpy(),
                        ramp_diag=gd.detach().numpy(), rand_seed=99, rand_gx=rx.detach().numpy(),
                        rand_gy=ry.detach().numpy(), rand_diag=rd.detach().numpy())
    print("[golden] sobel KAT centre rows:", gx[0, 0, 2].tolist(), gy[0, 0, 0].tolist(), gd[0, 0, 2].tolist())

    # -- state_dict key/shape contract (SURVEY 8b)
    import RGB_OFF, Flow_OFF
    for variant, mod in (("rgb", RGB_OFF), ("flow", Flow_OFF)):
        sd = mod.bninception_off(101, 1, 3).state_dict()
        with open(os.path.join(GOLD, f"state_dict_keys_full_{variant}.txt"), "w") as f:      # all 593 / 576 entries
            for k, v in sd.items():
                f.write(f"{k} {' '.join(map(str, v.shape))}\n")
        keys = OrderedDict((k, tuple(v.shape)) for k, v in sd.items() if "motion" in k or "sobel" in k)
        mine = O.param_shapes(variant)
        for k, shp in mine.items():
            assert keys[k] == tuple(shp), (k, keys[k], shp)
        extra = set(keys) - set(mine)
        assert extra <= {"sobel_edge_diagonal.conv.weight"}, extra
        with open(os.path.join(GOLD, f"state_dict_keys_{variant}.txt"), "w") as f:
            for k, shp in keys.items():
                f.write(f"{k} {' '.join(map(str, shp))}\n")
    # -- the whole reference model, images in (SURVEY 8f-2): backbone taps + score + OFF heads of RGB_OFF_forward /
    # Flow_OFF.forward with a seeded FULL state_dict, for the drop-in test of BNInception_OFF(backbone="bninception")
    for variant, mod, cin in (("rgb", RGB_OFF, 3), ("flow", Flow_OFF, 10)):
        B, Lg, seed = 1, 3, 31
        net = mod.bninception_off(O.NUM_CLASSES, B, Lg).eval()
        keys = [(k, tuple(v.shape)) for k, v in net.state_dict().items()]
        net.load_state_dict(O.make_state_dict(seed, keys))
        net = net.double()
        if variant != "rgb":
            net.consensus = _Mean()
        x = O.hash_normal(seed, (B * Lg, cin, 224, 224)).double()
        caught = {}
        hooks = [getattr(net, "motion_conv_gen_" + t).register_forward_pre_hook(lambda m, inp, t=t: caught.__setitem__(t, inp[0].detach()))
                 for t in O.LEVELS]
        with torch.no_grad():
            res = net.RGB_OFF_forward(x) if variant == "rgb" else net(x)
        for h in hooks:
            h.remove()
        fix = dict(variant=variant, batch=B, length=Lg, seed=seed, fc7=res[0].numpy(), score=res[1].numpy(), fc14=res[2].numpy())
        for t, v in caught.items():
            for kk, vv in digest(v, 128).items():
                fix[f"tap{t}.{kk}"] = vv
        np.savez_compressed(os.path.join(GOLD, f"backbone_{variant}_b1_l3.npz"), **fix)
        print(f"[golden] full model {variant}: fc7 {tuple(res[0].shape)} score {tuple(res[1].shape)} taps {[tuple(v.shape) for v in caught.values()][:2]}...")
    print("[golden] done")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        sys.exit("usage: python oracle/make_golden.py REFERENCE_DIR")
    REF = os.path.abspath(sys.argv[1])
    main()
