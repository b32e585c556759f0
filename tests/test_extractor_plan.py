"""CPU: the launch plan of the fused BN-Inception extractor (extractor.py) and the channels-last tap mode of the OFF engine.
Both are host logic (tables, descriptors, launch lists); nothing here launches a kernel."""
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _full_keys(variant):
    gold = os.path.join(ROOT, "tests", "golden")
    return [(l.split()[0], tuple(int(x) for x in l.split()[1:])) for l in open(os.path.join(gold, f"state_dict_keys_full_{variant}.txt"))]


def _stock_conv_flops(cin):
    """Forward FLOPs of one frame, counted with hooks on the stock module's convs and Linear (2 per multiply-add)."""
    from off_b200.backbone import BNInceptionBackbone
    bb = BNInceptionBackbone(101, cin)
    total = [0.0]

    def hook(mod, inp, out):
        if isinstance(mod, torch.nn.Conv2d):
            k = mod.kernel_size[0] * mod.kernel_size[1] * mod.in_channels
            total[0] += 2.0 * out.numel() * k
        else:
            total[0] += 2.0 * out.numel() * mod.in_features
    hs = [m.register_forward_hook(hook) for m in bb.modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear))]
    bb(torch.zeros(1, cin, 224, 224))
    for h in hs:
        h.remove()
    return total[0]


@pytest.mark.parametrize("cin", [3, 10])
def test_fused_extractor_plan_builds_without_a_gpu(cin):
    from off_b200 import plan as PL
    from off_b200.backbone import BNInceptionBackbone
    from off_b200.extractor import FusedBNInception
    n = 6
    fx = FusedBNInception(101, cin, n_frames=n, precision="tf32", device="cpu")
    plan = fx.plan
    assert plan.c_pad == (4 if cin == 3 else 12)
    # the module is a BNInceptionBackbone: same children, parameters, buffers, state_dict keys
    stock = BNInceptionBackbone(101, cin)
    assert [(k, tuple(v.shape)) for k, v in fx.state_dict().items()] == [(k, tuple(v.shape)) for k, v in stock.state_dict().items()]
    # launch list: the image conversion, ONE gather-fed stem GEMM, one TMA-fed GEMM per other conv of backbone.py's table,
    # the two stem pools and one pool per Inception module, the global pool and last_linear
    steps = {getattr(st, "name", None) or st.launches[0]: st for st in plan.steps}
    gathers = [st for st in plan.steps if isinstance(st, PL.Gemm) and not isinstance(st, PL.TGemm)]
    assert [g.name for g in gathers] == ["conv1_7x7_s2"]
    assert gathers[0].spec.a_mode == gathers[0].spec.b_mode == 2           # LOAD_VEC_K x LOAD_VEC_K
    convs = [name for name, m in stock.named_children() if isinstance(m, torch.nn.Conv2d)]
    assert len(convs) == 69
    for name in convs[1:]:
        st = steps[name]
        assert isinstance(getattr(st, "gemm", st), PL.TGemm), name
    pools = [n for n in steps if (n.startswith("inception_") and n.endswith("_pool")) or n in ("pool1", "pool2")]
    assert pools == ["pool1", "pool2"] + [f"inception_{t}_pool" for t in ("3a", "3b", "3c", "4a", "4b", "4c", "4d", "4e",
                                                                           "5a", "5b")]
    assert list(steps)[0] == "image_to_nhwc" and list(steps)[-2:] == ["global_pool", "last_linear"]
    assert len(plan.steps) == 1 + 69 + 12 + 2
    # algorithmic forward FLOPs from the plan's shapes agree with a hook count over the stock module (SURVEY: 4.06
    # GFLOP per RGB frame)
    want = _stock_conv_flops(cin) * n
    assert abs(plan.flops_fwd - want) / want < 1e-9
    if cin == 3:
        assert abs(plan.flops_fwd / n / 1e9 - 4.06) < 0.01
    # the nine taps are channels-last [N, C, S, S] tensors
    for t in plan.taps.values():
        assert t.shape[0] == n and t.is_contiguous(memory_format=torch.channels_last)


def test_fused_extractor_plan_keeps_the_fp32_weight_residuals_behind_the_weights():
    from off_b200 import _lib as L
    from off_b200.extractor import FusedBNInception
    fx = FusedBNInception(101, 3, n_frames=2, precision="fp32", device="cpu")
    plan = fx.plan
    assert plan.prec == L.PREC_TF32X3 and plan.w_lo.data_ptr() == plan.w_flat.data_ptr() + 4 * plan.w_flat.numel()
    tg = [getattr(st, "gemm", st) for st in plan.steps if hasattr(getattr(st, "gemm", st), "tdesc")]
    assert tg and all(g.tdesc.b_lo_delta == plan.w_flat.numel() for g in tg)


def test_channels_last_taps_in_the_off_engine():
    from off_b200 import _lib as L, engine as E, spec as S
    ref = E.OFFEngine(2, 3, "rgb", "cpu", "tf32")
    cl = E.OFFEngine(2, 3, "rgb", "cpu", "tf32", tap_layout="channels_last")
    names, cl_names = ref.launch_names(), cl.launch_names()
    assert not any(n.startswith("tapT_") for n in cl_names)
    assert [n for n in names if not n.startswith("tapT_")] == cl_names
    for tag in S.LEVELS:
        t = cl.taps[tag]
        assert t.shape == ref.taps[tag].shape and t.is_contiguous(memory_format=torch.channels_last)
        # forward: a dense tensor map over the tap; weight gradient: the im2col form; both re-bound by select_taps
        users = cl._tap_users[tag]
        kinds = sorted(g.tdesc.a_kind for g in users)
        assert kinds == [L.TMA_A_DENSE, L.TMA_A_IM2COL_T], tag
        assert all(g.tdesc.g.a_src == t.data_ptr() for g in users)
    cl.select_taps(1)
    for tag in S.LEVELS:
        assert all(g.tdesc.g.a_src == cl.tap_sets[1][tag].data_ptr() for g in cl._tap_users[tag])
    # the NCHW plan keeps its in-place NCHW route for the 28 / 14 levels
    assert all(g.tdesc.a_kind in (L.TMA_A_NCHW, L.TMA_A_NCHW_T) for g in ref._tap_users["3a"])
    with pytest.raises(ValueError):
        E.OFFEngine(1, 3, "flow", "cpu", "tf32", tap_grads=True, tap_layout="channels_last")
    with pytest.raises(ValueError):
        E.OFFEngine(1, 3, "flow", "cpu", "tf32", tap_layout="nhwc")


@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_fused_backbone_model_surface(variant):
    """BNInception_OFF(backbone='bninception_fused'): the reference's full state_dict, strict loading, the extractor's taps are
    the OFF engine's first input set, and CPU input is refused (no fallback)."""
    import off_oracle as O
    from off_b200 import RGB_OFF, Flow_OFF, RGB_OFF_v2
    from off_b200.extractor import FusedBNInception
    mod = RGB_OFF if variant == "rgb" else Flow_OFF
    m = mod.bninception_off(101, 1, 3, device="cpu", backbone="bninception_fused")
    assert isinstance(m.backbone, FusedBNInception) and m.off.engine.tap_layout == "channels_last"
    want = _full_keys(variant)
    got = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert dict(got) == dict(want) and len(got) == len(want) == (593 if variant == "rgb" else 576)
    m.load_state_dict(O.make_state_dict(3, want), strict=True)
    for tag, t in m.backbone.plan.taps.items():
        assert t.data_ptr() == m.off.engine.tap_sets[0][tag].data_ptr()
    assert all("motion" in n for n, p in m.named_parameters() if p.requires_grad)
    with pytest.raises(RuntimeError):
        m.backbone(torch.zeros(3, 10 if variant == "flow" else 3, 224, 224))
    with pytest.raises(ValueError):
        mod.bninception_off(101, 1, 3, device="cpu", backbone="bninception_fused", tap_grads=True)
    with pytest.raises(ValueError):
        mod.bninception_off(101, 1, 3, device="cpu", backbone="inception")
    assert RGB_OFF_v2.bninception_off(101, 1, 3, device="cpu", backbone="bninception_fused").off.engine.tap_layout == "channels_last"
