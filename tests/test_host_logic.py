"""CPU: host-side logic of the product package (no kernel launches)."""
import ctypes as C
import math
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import off_b200  # noqa: F401
from off_b200 import _lib as L, spec as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_state_dict_contract(variant):
    """Parameter names / shapes equal the reference's state_dict (captured from the reference classes)."""
    want = {}
    for line in open(os.path.join(GOLD, f"state_dict_keys_{variant}.txt")):
        f = line.split()
        want[f[0]] = tuple(int(x) for x in f[1:])
    mine = S.param_shapes(variant)
    frozen = {"sobel_edge_diagonal.conv.weight"}
    assert set(mine) == set(want) - frozen
    for k, shp in mine.items():
        assert tuple(shp) == want[k], k
    assert sum(int(np.prod(s)) for s in mine.values()) == (9872975 if variant == "rgb" else 9870095)   # SURVEY 8a12


@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_flat_layout(variant):
    layout, total = S.flat_layout(variant)
    spans = sorted((off, off + int(np.prod(shp))) for off, shp in layout.values())
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 <= b0                                        # no overlap
    assert spans[-1][1] <= total
    for tag, (cin, _) in S.LEVELS.items():                     # gen|down adjacent -> one [160, cin] GEMM operand
        g, d = layout[f"motion_conv_gen_{tag}.weight"][0], layout[f"motion_spatial_down_{tag}.weight"][0]
        assert d == g + S.GEN_C * cin and g % 4 == 0
        gb, db = layout[f"motion_conv_gen_{tag}.bias"][0], layout[f"motion_spatial_down_{tag}.bias"][0]
        assert db == gb + S.GEN_C and gb % 4 == 0


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "offk.h")).read()
    declared = set(re.findall(r"\b(offk_[a-z0-9_]+)\s*\(", hdr))
    lib = L.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/offk.h but not exported by liboffk.so"
    assert declared == set(L.exported_symbols()), declared ^ set(L.exported_symbols())
    assert lib.offk_version() == 100
    assert lib.offk_drop_keep_host(1, 2, 0.0) == 1 and lib.offk_drop_keep_host(1, 2, 1.0) == 0


def test_ctypes_structs_match_the_c_header():
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "offk.h"
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(offk_idx_t), sizeof(offk_gemm_t), offsetof(offk_gemm_t, out),
             offsetof(offk_gemm_t, split_k), sizeof(offk_stencil_t), offsetof(offk_stencil_t, seed),
             offsetof(offk_stencil_t, keep_mask), sizeof(offk_stencil_io_t), offsetof(offk_stencil_io_t, dg_fs),
             offsetof(offk_stencil_io_t, dbias));
      printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(offk_tgemm_t), offsetof(offk_tgemm_t, a_kind), offsetof(offk_tgemm_t, wout),
             offsetof(offk_tgemm_t, geom_flags), offsetof(offk_tgemm_t, precision), offsetof(offk_tgemm_t, tmap_a),
             sizeof(offk_permute_t));
      return 0;
    }'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", os.path.join(d, "t")])
        out = subprocess.check_output([os.path.join(d, "t")]).split()
    got = [int(x) for x in out]
    assert got == [C.sizeof(L.OffkIdx), C.sizeof(L.OffkGemm), L.OffkGemm.out.offset, L.OffkGemm.split_k.offset,
                   C.sizeof(L.OffkStencil), L.OffkStencil.seed.offset, L.OffkStencil.keep_mask.offset,
                   C.sizeof(L.OffkStencilIO), L.OffkStencilIO.dg_fs.offset, L.OffkStencilIO.dbias.offset,
                   C.sizeof(L.OffkTGemm), L.OffkTGemm.a_kind.offset, L.OffkTGemm.wout.offset, L.OffkTGemm.geom_flags.offset,
                   L.OffkTGemm.precision.offset, L.OffkTGemm.tmap_a.offset, C.sizeof(L.OffkPermute)]


def test_cpu_calls_fail_loudly():
    """No CPU fallback: bad arguments give error codes + messages, not silent success."""
    lib = L.lib()
    g = L.OffkGemm()
    assert lib.offk_gather_gemm(C.byref(g), L.PREC_TF32, None) == -1
    assert b"empty problem" in lib.offk_last_error_string()
    s = L.OffkStencil()
    assert lib.offk_stencil_diff_fwd(C.byref(s), None, None, None, None, None, None) == -1
    with pytest.raises(RuntimeError):
        L.check(-1, "probe")


def test_engine_plan_builds_without_a_gpu():
    """The plan (tables, descriptors, launch list) is pure host logic."""
    from off_b200 import engine as E, tables as T
    eng = E.OFFEngine(2, 3, "rgb", "cpu", "tf32")
    assert eng.launches_fwd > 40 and eng.launches_bwd > 60
    assert eng.unit_range[1] == eng.stage_range[0] and eng.stage_range[1] == eng.n_flat
    # forward FLOPs follow the survey's scaling law 0.28897*N + 1.29305*P GFLOP (+ the down rows of the N-P extra frames)
    gf = 0.28897 * eng.N + 1.29305 * eng.P + 0.07235 * (eng.N - eng.P)
    assert abs(eng.flops_fwd / 1e9 - gf) / gf < 0.01
    flow = E.OFFEngine(1, 4, "flow", "cpu", "tf32", tap_grads=True)
    assert flow.consensus and "motion_spatial_grad_3a.weight" not in flow.params
    # tf32 plan: the 7x7 taps go through a channels-last copy, every stride-2 data-gradient class has its own weight
    # block, the forward stencil is two launches and all KxK weight gradients are un-permuted by one
    names = eng.launch_names()
    assert "tapT_5a" in names and "tapT_5b" in names and "tapT_3a" not in names
    assert [n for n in names if n.startswith("stencil_fwd_")] == ["stencil_fwd_28", "stencil_fwd_14+7"]
    assert names.count("unpermute_kxk_weight_grads") == 1 and "stencil_bwd" in names
    for conv in ("motion_conv_trans_28", "motion_conv_trans_14"):
        assert all((conv, a, b) in eng.wd for a in (0, 1) for b in (0, 1))
    # tap gradients: every unit's data gradient into its NCHW tap is launched; the 7x7 units read a channels-last tap copy
    flow_names = flow.launch_names()
    for tag in S.LEVELS:
        assert any(n.startswith(f"unit_{tag}.dgrad") for n in flow_names), tag
    assert "tapT_5a" in flow_names and "tapT_5b" in flow_names
    with pytest.raises(KeyError):
        E.OFFEngine(1, 4, "flow", "cpu", "fp32_simt")
    # precision='fp32' is the 3xTF32 tensor-core mode: the same TMA-fed plan as 'tf32', launch for launch, plus the two
    # per-step weight-residual passes (the GEMMs then receive both weight tiles by TMA)
    x3 = E.OFFEngine(2, 3, "rgb", "cpu", "fp32")
    extra = {"weight_residuals_params", "weight_residuals_copies"}
    assert x3.prec == L.PREC_TF32X3 and [n for n in x3.launch_names() if n not in extra] == names
    assert extra <= set(x3.launch_names()) and x3.params_lo.data_ptr() == x3.params_flat.data_ptr() + 4 * x3.n_flat
    # hazard analysis: a step never waits on its own lane, and every cross-lane wait points backwards
    for sched in (eng.fwd_sched, eng.bwd_sched):
        for i, ws in enumerate(sched.waits):
            assert all(j < i and sched.lanes[j] != sched.lanes[i] for j in ws)


def test_reference_model_surface_builds_without_a_gpu():
    """BNInception_OFF(num_classes, batch, length) / bninception_off(num_classes, batch, num_seg) under the reference's
    module names (RGB_OFF.py:30-36,1346-1377; Flow_OFF.py:38-51,1371-1385; RGB_OFF_v2.py:43-58,1378-1392): constructor
    signature, attributes, state_dict keys of the OFF section, the 'motion' parameter filter of train_off.py:40."""
    import inspect
    import torch
    from off_b200 import RGB_OFF, Flow_OFF, RGB_OFF_v2
    gold = os.path.join(ROOT, "tests", "golden")
    keys = lambda v: {l.split()[0]: tuple(int(x) for x in l.split()[1:]) for l in open(os.path.join(gold, f"state_dict_keys_{v}.txt"))}
    for mod, gv in ((RGB_OFF, "rgb"), (Flow_OFF, "flow"), (RGB_OFF_v2, "flow")):
        assert list(inspect.signature(mod.bninception_off).parameters)[:3] == ["num_classes", "batch", "num_seg"]
        assert list(inspect.signature(mod.BNInception_OFF.__init__).parameters)[1:4] == ["num_classes", "batch", "length"]
        m = mod.bninception_off(101, 2, 3, device="cpu")
        assert isinstance(m, mod.BNInception_OFF) and (m.batch, m.length) == (2, 3) and m.modality_fuse is False
        assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == keys(gv)
        assert all("motion" in n for n, p in m.named_parameters() if p.requires_grad)
        assert m.consensus.consensus_type == "avg"
        m.eval()
        assert not m.off.training
        with pytest.raises(RuntimeError):
            m.forward(torch.zeros(6, 3, 8, 8)) if gv != "rgb" else m.RGB_OFF_forward(torch.zeros(6, 3, 8, 8))
    assert RGB_OFF.bninception_off_sobel(101, 1, 3, device="cpu").variant == "rgb"
    # one frame pair: torch.squeeze in the reference drops the batch dimension as well (RGB_OFF.py:786,792,846;
    # tests/golden/off_rgb_b1_l2.npz holds [101]-shaped heads produced by the reference itself)
    one = RGB_OFF.bninception_off(101, 1, 2, device="cpu")
    object.__setattr__(one, "off", lambda taps: (torch.ones(1, 101), torch.zeros(1, 101), torch.ones(1, 101)))
    f7, _, f14 = one.RGB_OFF_forward({})
    assert f7.shape == (101,) and f14.shape == (101,)
    assert np.load(os.path.join(gold, "off_rgb_b1_l2.npz"))["fc7"].shape == (101,)
    # data flow of the three forwards with the device work stubbed out (shapes and return structure of
    # RGB_OFF.py:860, Flow_OFF.py:879-884, RGB_OFF_v2.py:891)
    B, Lg, NC = 2, 3, 101

    class Backbone(torch.nn.Module):
        def forward(self, x):
            return {"taps": x.shape[0]}, torch.arange(B * Lg * NC, dtype=torch.float32).reshape(B * Lg, NC), "conv2"

    class Mean(torch.nn.Module):
        def forward(self, t):
            return t.mean(dim=1, keepdim=True)

    for mod, per_pair in ((RGB_OFF, True), (Flow_OFF, False), (RGB_OFF_v2, False)):
        m = mod.bninception_off(NC, B, Lg, device="cpu", backbone=Backbone())
        n_out = B * (Lg - 1) if per_pair else B
        object.__setattr__(m, "off", lambda taps, n_out=n_out: (torch.ones(n_out, NC), torch.zeros(n_out, NC), 2 * torch.ones(n_out, NC)))
        m.consensus = Mean()                                       # CPU stand-in for offk_segment_mean (basic_ops.py:22)
        x = torch.zeros(B * Lg, 3, 8, 8)
        if per_pair:
            fc7, score, fc14 = m.RGB_OFF_forward(x)
            assert fc7.shape == (B * (Lg - 1), NC) and score.shape == (B * Lg, NC) and fc14[0, 0] == 2
            assert m(x).shape == (B * Lg, NC)                      # RGB_OFF.forward = backbone classifier (:1340-1344)
        else:
            out = m(x)
            assert len(out) == (4 if mod is RGB_OFF_v2 else 3)
            fc7, score, fc14 = out[:3]
            want = torch.arange(B * Lg * NC, dtype=torch.float32).reshape(B, Lg, NC).mean(1)
            assert fc7.shape == (B, NC) and torch.equal(score, want)
            if mod is RGB_OFF_v2:
                assert out[3] == "conv2"
            m.modality_fuse = True
            assert torch.equal(m(x), 1 + want + 2)


def test_checkpoint_compatibility(tmp_path):
    """Reference-style checkpoints: plain state_dict files (train_off.py:155-156), 'module.' / 'base_model.' prefixes
    (test_flow_off.py:52-58, Flow_OFF.py:1399), key-filtered partial merges (model_utils.py:200,240)."""
    import torch
    from off_b200 import RGB_OFF, checkpoint as CK
    a = RGB_OFF.bninception_off(101, 1, 3, device="cpu")
    b = RGB_OFF.bninception_off(101, 1, 3, device="cpu")
    assert not torch.equal(a.off.engine.params_flat, b.off.engine.params_flat)
    path = str(tmp_path / "2019-01-08_22-42-50.pth")
    keys = CK.save_checkpoint(a, path, data_parallel_prefix=True)
    assert all(k.startswith("module.") for k in keys) and len(keys) == 108
    loaded, missing, ignored = CK.load_checkpoint(b, path)
    assert len(loaded) == 108 and not missing and not ignored
    assert torch.equal(a.off.engine.params_flat, b.off.engine.params_flat)
    # partial merge: keep b's own FC heads, take the rest (the 'fc-action' / 'motion' style filters of model_utils.py)
    c = RGB_OFF.bninception_off(101, 1, 3, device="cpu")
    fc_before = c.fc_action_motion.weight.detach().clone()
    ck = {"module.base_model." + k: v for k, v in a.state_dict().items()}
    ck["module.base_model.conv1_7x7_s2.weight"] = torch.zeros(64, 3, 7, 7)        # a backbone entry the OFF module lacks
    loaded, missing, ignored = CK.merge_state_dict(c, ck, keep=lambda k: "fc_action" not in k)
    assert torch.equal(c.fc_action_motion.weight, fc_before)
    assert torch.equal(c.motion_conv_trans_28.weight, a.motion_conv_trans_28.weight)
    assert set(missing) == {k for k in a.state_dict() if "fc_action" in k} and "conv1_7x7_s2.weight" in ignored
    bad = dict(a.state_dict())
    bad["motion_conv_trans.weight"] = torch.zeros(3, 3)
    with pytest.raises(RuntimeError):
        CK.merge_state_dict(c, bad)


def test_seeded_dropout_uses_every_seed_bit():
    """ADVICE r1 (high): the keep decisions of ALL four elements of a channel quad must change with the seed, also for
    small seeds and for seeds that differ only in their low or only in their high word; the keep rate stays 1 - p."""
    lib = L.lib()
    n = 4096

    def mask(seed):
        return [[lib.offk_drop_keep_host(seed, 4 * q + lane, 0.8) for q in range(n // 4)] for lane in range(4)]

    base = mask(1)
    for other in (2, 3, 1 + (1 << 32), 1 + (5 << 40), 73, 137, 4928):
        m = mask(other)
        for lane in range(4):
            same = sum(a == b for a, b in zip(base[lane], m[lane])) / len(m[lane])
            assert same < 0.80, (other, lane, same)          # independent masks agree on 0.8^2 + 0.2^2 = 0.68 of the elements
    rate = sum(sum(r) for r in base) / n
    assert 0.17 < rate < 0.23
    # the engine's per-site salts (the kernels add the step seed held in device memory): 12 distinct 64-bit values
    from off_b200 import engine as E
    salts = {E.OFFEngine._site_salt(i) for i in range(12)}
    assert len(salts) == 12 and all(0 <= v < 1 << 64 for v in salts)


def test_backbone_layers_live_at_the_top_level_like_the_reference(tmp_path):
    """ADVICE r1 (medium): the reference's checkpoints carry the BN-Inception layers at the top level
    (``conv1_7x7_s2.weight``, RGB_OFF.py:43); a model built with a feature extractor must expose, load and save them under
    exactly those keys, and a merge that would load nothing must not pass silently.  ``.to()`` / ``.float()`` move the
    extractor only: the OFF parameters stay views of the engine's flat buffer (ADVICE r1, low)."""
    import torch
    import warnings
    from off_b200 import RGB_OFF, checkpoint as CK

    class Backbone(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.conv1_7x7_s2 = torch.nn.Conv2d(3, 64, 7, 2, 3)
            self.conv1_7x7_s2_bn = torch.nn.BatchNorm2d(64)

        def forward(self, x):
            return {}, None

    m = RGB_OFF.bninception_off(101, 1, 3, device="cpu", backbone=Backbone())
    keys = list(m.state_dict())
    assert "conv1_7x7_s2.weight" in keys and "conv1_7x7_s2_bn.num_batches_tracked" in keys
    assert not any(k.startswith("backbone.") for k in keys)
    assert sum("motion" in k for k in keys) == 108
    # model_utils.py:240 style merge: everything but the OFF branch comes from the checkpoint
    ck = {"module." + k: torch.full_like(v, 0.5) for k, v in m.state_dict().items()}
    off_before = m.motion_conv_trans.weight.detach().clone()
    loaded, missing, ignored = CK.merge_state_dict(m, ck, keep=lambda k: "motion" not in k)
    assert "conv1_7x7_s2.weight" in loaded and float(m.backbone.conv1_7x7_s2.weight.mean()) == 0.5
    assert torch.equal(m.motion_conv_trans.weight, off_before)
    path = str(tmp_path / "full.pth")
    assert "conv1_7x7_s2.weight" in CK.save_checkpoint(m, path)
    # a backbone-only checkpoint into a model WITHOUT a backbone: nothing would be loaded -> error, not silence
    bare = RGB_OFF.bninception_off(101, 1, 3, device="cpu")
    with pytest.raises(RuntimeError, match="loaded nothing"):
        CK.merge_state_dict(bare, {"conv1_7x7_s2.weight": torch.zeros(64, 3, 7, 7)})
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        CK.merge_state_dict(bare, ck)                       # OFF keys load, backbone keys are reported
        assert any("not in the model" in str(x.message) for x in w)
    # placement / casting
    m.float().to("cpu")
    assert m.motion_conv_trans.weight.data_ptr() == m.off.engine.params["motion_conv_trans.weight"].data_ptr()
    with pytest.raises(RuntimeError, match="flat"):
        m.double()
    assert m.motion_conv_trans.weight.dtype == torch.float32
    assert list(m._modules)[:3] == list(RGB_OFF.bninception_off(101, 1, 3, device="cpu", backbone=Backbone())._modules)[:3]


def test_eval_protocol_fusion_accuracy_and_npz(tmp_path):
    """SURVEY 8f-4: the reference's video-level protocol (test_rgb_off.py:83-236): crops as the batch axis, crop means fused
    as rst1 + 2*rst2 + rst3, arg-max prediction, mean per-class accuracy from the confusion matrix, npz score layout."""
    import torch
    from off_b200 import Flow_OFF, evaluate as EV
    crops, segs, NC = 10, 25, 101

    class Backbone(torch.nn.Module):
        def forward(self, x):
            return {"n": x.shape[0]}, x.new_zeros(crops * segs, NC) + x.reshape(crops * segs, -1)[:, :1], None

    m = Flow_OFF.bninception_off(NC, crops, segs, device="cpu", backbone=Backbone())

    class Mean(torch.nn.Module):
        def forward(self, t):
            return t.mean(dim=1, keepdim=True)
    m.consensus = Mean()
    videos, want_scores = [], []
    g = torch.Generator().manual_seed(0)
    for label in (3, 3, 7, 50):
        s7, s14 = torch.randn(crops, NC, generator=g), torch.randn(crops, NC, generator=g)
        s7[:, label] += 5.0
        data = torch.full((crops * segs, 3, 2, 2), 0.25 * label)
        videos.append(((data, s7, s14), label))
        want_scores.append((s7, s14))
    state = {}
    class Off:                                   # CPU stand-in for the liboffk-backed OFF section
        training = False

        def train(self, mode=True):
            self.training = mode

        def __call__(self, taps):
            assert not self.training             # eval_video switches the model to eval mode (no dropout)
            return state["s7"], torch.zeros(crops, NC), state["s14"]
    object.__setattr__(m, "off", Off())

    def gen():
        for (data, s7, s14), label in videos:
            state.update(s7=s7, s14=s14)
            yield data, label
    res = EV.evaluate(m, gen(), save_path=str(tmp_path / "rgb_save_score_3"))
    assert res["pred"] == [3, 3, 7, 50] and res["accuracy"] == 1.0
    z = np.load(str(tmp_path / "rgb_save_score_3.npz"))
    assert sorted(z.files) == ["label", "scores1", "scores2", "scores3"]               # test_rgb_off.py:236
    assert z["scores1"].shape == (4, crops, NC) and z["label"].tolist() == [3, 3, 7, 50]
    s7, s14 = want_scores[2]
    rgb = np.full((crops, NC), 0.25 * 7)
    fused = EV.fuse_video_scores(s7.numpy(), rgb, s14.numpy())
    np.testing.assert_allclose(fused[0], s7.numpy().mean(0) + 2 * rgb.mean(0) + s14.numpy().mean(0), rtol=1e-6)
    # per-class accuracy is the mean over the classes that occur, not over videos
    acc, per_class, cf = EV.per_class_accuracy([0, 0, 0, 1], [0, 0, 1, 0], 3)
    assert abs(acc - (2 / 3 + 0) / 2) < 1e-12 and cf[0, 1] == 1 and np.isnan(per_class[2])


def _full_keys(variant):
    gold = os.path.join(ROOT, "tests", "golden")
    return [(l.split()[0], tuple(int(x) for x in l.split()[1:])) for l in open(os.path.join(gold, f"state_dict_keys_full_{variant}.txt"))]


@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_full_model_state_dict_equals_the_reference_key_for_key(variant, tmp_path):
    """SURVEY 8b / 8f-2,4: with the built-in feature extractor the model exposes EXACTLY the reference's state_dict (593
    entries RGB, 576 Flow / v2: names, shapes, BatchNorm buffers; generated from the reference classes by make_golden.py), and
    a DataParallel-style checkpoint of a full reference model loads strictly: everything loaded, nothing missing or ignored."""
    import torch
    import off_oracle as O
    from off_b200 import RGB_OFF, Flow_OFF, checkpoint as CK
    want = _full_keys(variant)
    assert len(want) == (593 if variant == "rgb" else 576)
    mod = RGB_OFF if variant == "rgb" else Flow_OFF
    m = mod.bninception_off(101, 1, 3, device="cpu", backbone="bninception")
    got = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert dict(got) == dict(want) and len(got) == len(want)
    assert all("motion" in n for n, p in m.named_parameters() if p.requires_grad)        # train_off.py:40: the backbone is frozen
    sd = O.make_state_dict(31, want)
    path = str(tmp_path / "full.pth")
    torch.save({"module." + k: v for k, v in sd.items()}, path)                         # test_flow_off.py:52-58
    loaded, missing, ignored = CK.load_checkpoint(m, path)
    assert len(loaded) == len(want) and not missing and not ignored
    assert torch.equal(m.state_dict()["inception_4e_double_3x3_2_bn.running_var"], sd["inception_4e_double_3x3_2_bn.running_var"])
    assert torch.equal(m.off.engine.params["motion_conv_trans.weight"], sd["motion_conv_trans.weight"])
    m.load_state_dict(sd, strict=True)                                                   # and the plain strict path


@pytest.mark.parametrize("variant", ["rgb", "flow"])
def test_builtin_backbone_matches_the_reference_taps(variant):
    """The built-in BN-Inception restatement against the reference class run on the same seeded FULL state_dict and images
    (fixture tests/golden/backbone_*.npz, fp64): the nine taps that feed the OFF units and Feature_Generation_Score."""
    import torch
    import off_oracle as O
    from off_b200.backbone import BNInceptionBackbone
    fix = np.load(os.path.join(ROOT, "tests", "golden", f"backbone_{variant}_b1_l3.npz"))
    B, Lg, seed = int(fix["batch"]), int(fix["length"]), int(fix["seed"])
    cin = 10 if variant == "flow" else 3
    bb = BNInceptionBackbone(101, cin).double()
    sd = O.make_state_dict(seed, _full_keys(variant))
    own = bb.state_dict()
    bb.load_state_dict({k: sd[k] for k in own}, strict=True)
    x = O.hash_normal(seed, (B * Lg, cin, 224, 224)).double()
    taps, score, conv2 = bb(x)
    assert list(taps) == ["3a", "3b", "3c", "4a", "4b", "4c", "4d", "5a", "5b"] and conv2.shape == (B * Lg, 192, 56, 56)
    for t, v in taps.items():
        flat = v.reshape(-1)
        idx = torch.from_numpy(fix[f"tap{t}.idx"])
        np.testing.assert_allclose(flat[idx].numpy(), fix[f"tap{t}.val"], rtol=0, atol=1e-9 * max(1.0, float(np.abs(fix[f"tap{t}.val"]).max())))
        assert abs(float(flat.norm()) - float(fix[f"tap{t}.l2"])) <= 1e-9 * float(fix[f"tap{t}.l2"])
    if variant == "rgb":                                     # per-frame score (RGB_OFF.py:592-594,860)
        np.testing.assert_allclose(score.numpy(), fix["score"], rtol=0, atol=1e-9)
    else:                                                    # Flow_OFF.forward returns its segment consensus (:867-872)
        np.testing.assert_allclose(score.view(B, Lg, -1).mean(1).numpy(), fix["score"], rtol=0, atol=1e-9)


def test_launch_policies_are_wave_aware():
    """Host-side tile / split-K policies (plan.py): pure functions of the problem shape, pinned here on the shapes whose
    measurements motivated them (DESIGN.md 3.2, finding 5)."""
    import off_b200  # noqa: F401
    from off_b200 import plan as PL
    # 3xTF32 (one CTA per SM): a second N tile repeats the A tile and its residual pass -- only the 37-tile 7x7 layers narrow
    assert PL._auto_tile_n(56 * 128, 160, True, True) == 0           # unit_5a: one tile of 160 columns, not five of 32
    assert PL._auto_tile_n(147 * 128, 64, True, True) == 0           # motion_conv_trans_28: 147 x 1, not 147 x 2
    assert PL._auto_tile_n(37 * 128, 256, True, True) == 128         # 7x7 stage: 37 x 2
    assert PL._auto_tile_n(37 * 128, 1024, True, True) == 0          # 37 x 4 tiles of 256 already
    # weight gradients: CTAs = tiles x split lands on whole rounds of the resident slots
    assert PL._wgrad_split(3, 3600, 148) == 49                       # unit_3a.wgrad: 147 CTAs, one round (was 3 x 98)
    assert PL._wgrad_split(3, 3600, 296) == 98                       # tf32 mode: two CTAs per SM
    s = PL._wgrad_split(123, 294, 148, 64)                           # motion_conv_trans_28.wgrad, 64-pixel K-blocks
    assert 123 * s <= 148 * math.ceil(123 * s / 148) and (148 * math.ceil(123 * s / 148) - 123 * s) < 15
    assert PL._wgrad_split(1, 588, 148) == 147                       # a single-tile 1x1 layer still fills the machine
