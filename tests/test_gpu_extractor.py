"""GPU: the fused BN-Inception extractor (extractor.py) -- its pools and image conversion, the extractor against the
reference fixtures and against the stock module, the full model on it, zero-copy taps, training from images and graph
replay.

Errors are max-abs relative to the tensor's max (as in test_full_model_is_a_drop_in_of_the_reference_class).  fp32 mode
(3xTF32) is held to that test's 1e-4 gate.  TOL_TF32 is the gate of the tf32 mode (one kind::tf32 MMA per product through
the 22 conv layers of the deepest path), see DESIGN.md section 4 for the measured values."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import off_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL_FP32 = 1e-4
TOL_TF32 = 5e-3


@pytest.fixture(scope="module")
def dev():
    import off_b200  # noqa: F401
    return torch.device("cuda")


@pytest.fixture(autouse=True)
def _no_tf32_in_torch():
    """The stock module is the reference here: cuDNN in plain fp32."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _rel(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return (got - want).abs().max().item() / want.abs().max().item()


def _keys(variant):
    return [(l.split()[0], tuple(int(x) for x in l.split()[1:])) for l in open(os.path.join(GOLD, f"state_dict_keys_full_{variant}.txt"))]


def _own(sd, module):
    own = module.state_dict()
    return {k: sd[k] for k in own}


def _report(what, err):
    print(f"[extractor-err] {what} {err:.3e}")


@pytest.mark.parametrize("kind", ["max_s2_p0", "max_s1_p1", "avg_s1_p1"])
@pytest.mark.parametrize("size", [112, 56, 28, 14, 7])
def test_pool3_nhwc_matches_torch(dev, kind, size):
    """offk_pool3_nhwc between channel slices, against F.max_pool2d / F.avg_pool2d (ceil mode, count_include_pad=True);
    max pools are exact."""
    from off_b200 import _lib as L
    lib = L.lib()
    n, ctot, coff, c, y_ctot, y_coff = 3, 40, 8, 24, 36, 4
    x = torch.randn(n, size, size, ctot, device=dev)
    mode, stride, pad = kind.split("_")[0], int(kind[-4]), int(kind[-1])
    xin = x[..., coff:coff + c].permute(0, 3, 1, 2)
    if mode == "max":
        want = F.max_pool2d(xin, 3, stride, pad, 1, ceil_mode=True)
    else:
        want = F.avg_pool2d(xin, 3, stride, pad, ceil_mode=True, count_include_pad=True)
    ho = want.shape[-1]
    y = torch.full((n, ho, ho, y_ctot), 7.0, device=dev)
    L.check(lib.offk_pool3_nhwc(x.data_ptr(), n, size, size, ctot, coff, c, stride, pad,
                                L.POOL_MAX if mode == "max" else L.POOL_AVG, y.data_ptr(), y_ctot, y_coff, None), "pool3")
    torch.cuda.synchronize()
    got = y[..., y_coff:y_coff + c].permute(0, 3, 1, 2)
    if mode == "max":
        assert torch.equal(got, want)
    else:
        assert (got - want).abs().max().item() < 1e-6
    assert torch.all(y[..., :y_coff] == 7.0) and torch.all(y[..., y_coff + c:] == 7.0)       # only the slice is written


@pytest.mark.parametrize("c,c_pad", [(3, 4), (10, 12)])
def test_image_to_nhwc(dev, c, c_pad):
    from off_b200 import _lib as L
    x = torch.randn(2, c, 224, 224, device=dev)
    y = torch.full((2, 224, 224, c_pad), 5.0, device=dev)
    L.check(L.lib().offk_image_to_nhwc(x.data_ptr(), y.data_ptr(), 2, c, 224 * 224, c_pad, None), "image_to_nhwc")
    torch.cuda.synchronize()
    assert torch.equal(y[..., :c], x.permute(0, 2, 3, 1)) and torch.all(y[..., c:] == 0)


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_fused_extractor_matches_the_reference_fixture(dev, variant, precision):
    """Against the reference class run in fp64 on the seeded full state_dict and images (tests/golden/backbone_*.npz): the
    nine taps and Feature_Generation_Score; then the whole model on the fused extractor, images in."""
    from off_b200 import RGB_OFF, Flow_OFF
    from off_b200.extractor import FusedBNInception
    fix = np.load(os.path.join(GOLD, f"backbone_{variant}_b1_l3.npz"))
    B, Lg, seed = int(fix["batch"]), int(fix["length"]), int(fix["seed"])
    cin = 10 if variant == "flow" else 3
    tol = TOL_FP32 if precision == "fp32" else TOL_TF32
    sd = O.make_state_dict(seed, _keys(variant))
    x = O.hash_normal(seed, (B * Lg, cin, 224, 224)).to(dev)
    fx = FusedBNInception(101, cin, B * Lg, precision, dev)
    fx.load_state_dict(_own(sd, fx), strict=True)
    taps, score, conv2 = fx(x)
    torch.cuda.synchronize()
    assert conv2.shape == (B * Lg, 192, 56, 56)
    for t, v in taps.items():
        flat = v.reshape(-1).cpu()
        idx = torch.from_numpy(fix[f"tap{t}.idx"])
        val = torch.from_numpy(fix[f"tap{t}.val"])
        err = (flat[idx].double() - val).abs().max().item() / val.abs().max().item()
        _report(f"{variant} {precision} tap{t}", err)
        assert err < tol, (t, err)
        l2 = float(fix[f"tap{t}.l2"])
        assert abs(float(v.double().norm()) - l2) / l2 < tol, t
    want = torch.from_numpy(fix["score"])
    got = score if variant == "rgb" else score.view(B, Lg, -1).mean(1)
    _report(f"{variant} {precision} score", _rel(got, want))
    assert _rel(got, want) < tol
    # the full model, images in: RGB_OFF.RGB_OFF_forward / Flow_OFF.forward
    mod = RGB_OFF if variant == "rgb" else Flow_OFF
    m = mod.bninception_off(101, B, Lg, device=dev, backbone="bninception_fused", precision=precision).eval()
    m.load_state_dict(sd, strict=True)
    with torch.no_grad():
        out = m.RGB_OFF_forward(x) if variant == "rgb" else m(x)
    for got, key in zip(out[:3], ("fc7", "score", "fc14")):
        want = torch.from_numpy(fix[key])
        assert tuple(got.shape) == tuple(want.shape), key
        _report(f"{variant} {precision} model {key}", _rel(got, want))
        assert _rel(got, want) < tol, key


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("cin", [3, 10])
def test_fused_extractor_matches_the_stock_module_after_a_reload(dev, cin, precision):
    """B=2, L=3: fused vs stock after load_state_dict of different weights (the fold is redone), every tap, the score and
    conv2; the fixture's BatchNorm statistics are far from (0, 1), so folding is not the identity."""
    from off_b200.backbone import BNInceptionBackbone
    from off_b200.extractor import FusedBNInception
    variant = "flow" if cin == 10 else "rgb"
    tol = TOL_FP32 if precision == "fp32" else TOL_TF32
    n = 6
    fx = FusedBNInception(101, cin, n, precision, dev)
    stock = BNInceptionBackbone(101, cin).to(dev)
    x = O.hash_normal(21, (n, cin, 224, 224)).to(dev)
    fx.load_state_dict(_own(O.make_state_dict(1, _keys(variant)), fx), strict=True)
    first = fx(x)[1]
    sd = _own(O.make_state_dict(2, _keys(variant)), fx)
    for k, v in sd.items():
        if k.endswith("running_var"):
            assert (v - 1).abs().min() > 0 and v.std() > 0.1, k
        if k.endswith("running_mean"):
            assert v.abs().max() > 0.1, k
    fx.load_state_dict(sd, strict=True)
    stock.load_state_dict(sd, strict=True)
    taps, score, conv2 = fx(x)
    with torch.no_grad():
        rtaps, rscore, rconv2 = stock(x)
    torch.cuda.synchronize()
    assert _rel(first, rscore) > 0.2                        # the reload changed the result: the plan did refold
    for t in rtaps:
        assert taps[t].shape == rtaps[t].shape and taps[t].is_contiguous(memory_format=torch.channels_last)
        _report(f"stock {variant} {precision} tap{t}", _rel(taps[t], rtaps[t]))
        assert _rel(taps[t], rtaps[t]) < tol, t
    _report(f"stock {variant} {precision} score", _rel(score, rscore))
    _report(f"stock {variant} {precision} conv2", _rel(conv2, rconv2))
    assert _rel(score, rscore) < tol and _rel(conv2, rconv2) < tol
    with pytest.raises(RuntimeError):
        fx(x.double())
    with pytest.raises(RuntimeError):
        fx(x[:3])


def test_rgb_v2_returns_conv2_and_the_taps_are_the_engines(dev):
    """RGB_OFF_v2 on the fused extractor returns conv2_relu_3x3_out as its 4th output; the taps the extractor returns ARE the
    OFF engine's input buffers (no copy between the two networks)."""
    from off_b200 import RGB_OFF_v2
    from off_b200.backbone import BNInceptionBackbone
    B, Lg = 2, 3
    m = RGB_OFF_v2.bninception_off(101, B, Lg, device=dev, backbone="bninception_fused", precision="fp32").eval()
    sd = O.make_state_dict(4, [(k, tuple(v.shape)) for k, v in m.state_dict().items()])
    m.load_state_dict(sd, strict=True)
    x = O.hash_normal(8, (B * Lg, 3, 224, 224)).to(dev)
    out = m(x)
    assert len(out) == 4
    stock = BNInceptionBackbone(101, 3).to(dev)
    stock.load_state_dict(_own(sd, stock))
    with torch.no_grad():
        _, _, rconv2 = stock(x)
    assert _rel(out[3], rconv2) < TOL_FP32
    taps, _, _ = m.backbone(x)
    for tag, t in taps.items():
        buf = m.off.engine.taps[tag]
        assert t.data_ptr() == buf.data_ptr() and t.untyped_storage().data_ptr() == buf.untyped_storage().data_ptr()


def test_training_from_images_matches_the_stock_taps(dev):
    """model.train() on the fused extractor with injected dropout masks: OFF parameter gradients within the fp32-mode
    gradient gate (test_gpu_parity.TOL_FP32: worst relative L2 5e-2, a bound on ReLU gate flips) of an NCHW OFFSubNetwork
    fed the stock extractor's eval-mode taps, and within 1e-2 of the same NCHW network fed the fused extractor's own taps
    (the channels-last unit path alone; the NCHW network run twice on identical taps already differs by up to 1e-3 on the
    most strongly gated unit, through the order of its split-K fp32 atomics).

    A parameter's error is taken relative to its own gradient norm, floored at 1e-6 of the norm of all OFF gradients (fp32
    round-off of the whole gradient).  Without the floor, gradients that cancel to round-off are compared digit by digit:
    with these weights nearly every 4d-level gen unit is gated off, its bias gradient is ~3e-8 against a total norm of
    ~1e2, and the NCHW network run twice on identical taps already disagrees on it by ~100 %."""
    from off_b200 import RGB_OFF
    from off_b200.backbone import BNInceptionBackbone
    from off_b200.modules import OFFSubNetwork
    B, Lg, seed = 2, 3, 6
    sd = O.make_state_dict(seed, _keys("rgb"))
    x = O.hash_normal(seed, (B * Lg, 3, 224, 224)).to(dev)
    masks = O.make_dropout_masks(seed, B, Lg)
    r7, r14 = O.hash_normal(77, (B * (Lg - 1), 101)).to(dev), O.hash_normal(78, (B * (Lg - 1), 101)).to(dev)

    def grads(net, taps):
        net.zero_grad(set_to_none=True)
        a, _, b = net(taps, masks=masks)
        ((a * r7).sum() + (b * r14).sum()).backward()
        torch.cuda.synchronize()
        return {n: p.grad.clone() if p.grad is not None else None for n, p in net.named_parameters()}

    m = RGB_OFF.bninception_off(101, B, Lg, device=dev, backbone="bninception_fused", precision="fp32")
    m.load_state_dict(sd, strict=True)
    m.train()
    taps, _, _ = m.backbone(x)
    fused_taps = {t: v.contiguous() for t, v in taps.items()}                # NCHW copies of the fused extractor's taps
    got = grads(m.off, taps)
    ref = OFFSubNetwork(B, Lg, "rgb", precision="fp32", device=dev)
    ref.load_state_dict(m.off.state_dict())
    ref.train()
    same_taps = grads(ref, fused_taps)
    stock = BNInceptionBackbone(101, 3).to(dev)
    stock.load_state_dict(_own(sd, stock))
    with torch.no_grad():
        staps, _, _ = stock(x)
    stock_taps = grads(ref, staps)
    floor = 1e-6 * torch.cat([g.reshape(-1) for g in stock_taps.values() if g is not None]).norm().item()
    worst = {"stock": 0.0, "same": 0.0}
    for n, g in got.items():
        if stock_taps[n] is None:
            assert g is None and same_taps[n] is None, n
            continue
        for key, want, tol in (("stock", stock_taps[n], 5e-2), ("same", same_taps[n], 1e-2)):
            e = (g - want).norm().item() / max(want.norm().item(), floor)
            worst[key] = max(worst[key], e)
            assert e < tol, (key, n, e)
    _report("train grad worst rel-L2 vs stock taps", worst["stock"])
    _report("train grad worst rel-L2 vs the same taps in NCHW", worst["same"])


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_graph_replay_is_bit_identical_to_eager(dev, precision):
    """The captured extractor pass replays the eager launches: bit-identical outputs for every tap that no split-K
    accumulation (order-dependent fp32 atomics) feeds; the rest within the precision's gate."""
    from off_b200.extractor import FusedBNInception
    n = 6
    fx = FusedBNInception(101, 3, n, precision, dev)
    fx.load_state_dict(_own(O.make_state_dict(9, _keys("rgb")), fx))
    x = O.hash_normal(10, (n, 3, 224, 224)).to(dev)
    taps, score, conv2 = fx(x)
    eager = ({t: v.clone() for t, v in taps.items()}, score.clone(), conv2.clone())
    fx.use_graphs = True
    for _ in range(2):
        taps, score, conv2 = fx(x.clone())                     # the graph reads its own copy of the input
        torch.cuda.synchronize()
        split = [i for i, st in enumerate(fx.plan.steps) if getattr(getattr(st, "gemm", st), "desc", None) is not None
                 and getattr(st, "gemm", st).desc.split_k > 1]
        first = min(split) if split else len(fx.plan.steps)
        names = [getattr(st, "name", None) or st.launches[0] for st in fx.plan.steps]
        exact = 0
        assert torch.equal(conv2, eager[2])
        for t, v in taps.items():
            mine = [i for i, nm in enumerate(names) if nm.startswith(f"inception_{t}_")]
            if max(mine) < first:
                assert torch.equal(v, eager[0][t]), t
                exact += 1
            else:
                assert _rel(v, eager[0][t]) < (TOL_FP32 if precision == "fp32" else TOL_TF32), t
        assert exact >= 2
        if not split:
            assert torch.equal(score, eager[1])
