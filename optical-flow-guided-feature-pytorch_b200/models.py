"""The reference's model-class surface over the B200 OFF path: ``BNInception_OFF(num_classes, batch, length)`` and the
``bninception_off(num_classes, batch, num_seg)`` factories of RGB_OFF.py:30-36,1346-1377, Flow_OFF.py:38-51,1371-1385
and RGB_OFF_v2.py:43-58,1378-1392.

Only the OFF section (RGB_OFF.py:596-860 / Flow_OFF.py:606-884) is implemented here -- it runs on liboffk through
``OFFSubNetwork``.  The frozen BN-Inception feature extractor (RGB_OFF.py:43-263,362-594; train_off.py:39-57 keeps it
in eval mode without gradients) is optional: pass ``backbone="bninception"`` for the built-in
table-driven restatement on stock torch ops (``off_b200/backbone.py``; the model is then a complete drop-in: images in,
the reference's 593 / 576 state_dict entries), ``backbone="bninception_fused"`` for the same extractor on liboffk
(``off_b200/extractor.py``: CUDA fp32 images of exactly ``batch*length`` frames, BatchNorm folded from its running
statistics, the taps written channels-last straight into the OFF engine's input buffers), or pass any module mapping the
image batch ``[batch*length, 3 | 10, 224, 224]`` to ``(taps, score)`` where ``taps`` holds the nine Inception outputs
'3a'..'5b' (``inception_3a_output_out`` ... ``inception_5b_output_out``, RGB_OFF.py:395-590) and ``score`` is
``Feature_Generation_Score`` ``[batch*length, num_classes]`` (:592-594).  Without a backbone the forward methods take
the taps themselves (what every BASELINE config does with synthetic features) and the score is ``None``.

The ``motion_*`` / ``fc_action_motion*`` sub-modules sit directly on this class under the reference's attribute names,
so ``state_dict()`` carries exactly the reference's OFF keys (plus ``sobel_edge_diagonal.conv.weight`` for Flow / v2),
and the training scripts' ``'motion' in name`` parameter filter (train_off.py:40) selects the same tensors.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import spec as S
from .basic_ops import ConsensusModule
from .modules import OFFSubNetwork


class BNInception_OFF(nn.Module):
    """variant 'rgb'  : RGB_OFF.BNInception_OFF  -- learned depth-wise 3x3 spatial gradient, per-pair outputs
                        ``RGB_OFF_forward(x) -> (fc7 [B(L-1),101], score [BL,num_classes], fc14 [B(L-1),101])`` (:860)
       variant 'flow' : Flow_OFF.BNInception_OFF -- fixed diagonal Sobel, segment consensus (``self.consensus``),
                        ``forward(x) -> (fc7 [B,101], score [B,num_classes], fc14 [B,101])`` or their sum when
                        ``self.modality_fuse`` (Flow_OFF.py:867-884)
       variant 'rgb_v2': RGB_OFF_v2.BNInception_OFF -- as 'flow' on RGB input; the non-fused return carries a 4th item,
                        ``conv2_relu_3x3_out`` (RGB_OFF_v2.py:891), taken from the backbone's optional third output."""

    def __init__(self, num_classes=1000, batch=16, length=7, variant="rgb", backbone=None, precision="tf32",
                 index_mode="reference_flat", tap_grads=False, device="cuda"):
        super().__init__()
        assert variant in ("rgb", "flow", "rgb_v2")
        self.batch, self.length, self.num_classes, self.variant = batch, length, num_classes, variant
        self.modality_fuse = False                                            # Flow_OFF.py:45, RGB_OFF_v2.py:52
        self.consensus_type = "avg"
        self.consensus = ConsensusModule(self.consensus_type, dim=1)          # Flow_OFF.py:47-48
        off_variant = "rgb" if variant == "rgb" else "flow"
        if isinstance(backbone, str) and backbone not in ("bninception", "bninception_fused"):
            raise ValueError("backbone: a module, None, 'bninception' (the built-in TSN BN-Inception extractor on stock torch "
                             "ops) or 'bninception_fused' (the same extractor on liboffk, writing channels-last taps)")
        fused = backbone == "bninception_fused"
        # not registered as a child: its parameter holders are re-registered below under the reference's names
        object.__setattr__(self, "off", OFFSubNetwork(batch, length, off_variant, precision=precision, index_mode=index_mode,
                                                      tap_grads=tap_grads, device=device,
                                                      tap_layout="channels_last" if fused else "nchw"))
        for name, mod in self.off.named_children():
            setattr(self, name, mod)                  # motion_conv_gen_3a ... fc_action_motion_14 (+ sobel_edge_diagonal)
        self._off_children = tuple(n for n, _ in self.off.named_children())
        if fused:
            from .extractor import FusedBNInception
            backbone = FusedBNInception(num_classes, 10 if variant == "flow" else 3, batch * length, precision, device,
                                        taps=self.off.engine.tap_sets[0])
        elif isinstance(backbone, str):
            from .backbone import BNInceptionBackbone
            backbone = BNInceptionBackbone(num_classes, in_channels=10 if variant == "flow" else 3).to(device)
        self._attach_backbone(backbone)

    # ------------------------------------------------------------------ helpers
    def _attach_backbone(self, backbone):
        """The reference keeps the BN-Inception layers at the TOP level of the class (``conv1_7x7_s2.weight``, ...,
        RGB_OFF.py:43-263), so its checkpoints carry top-level keys.  The feature extractor's layers (and its direct
        parameters / buffers) are therefore registered here under their own names -- ``state_dict()`` / ``load_state_dict``
        / ``.to()`` see them exactly as the reference's do -- while the extractor object itself is a plain attribute."""
        object.__setattr__(self, "backbone", backbone)
        if backbone is None:
            return
        taken = set(self._off_children) | {"consensus"}
        for name, child in backbone.named_children():
            if name in taken:
                raise ValueError(f"backbone layer name {name!r} collides with an OFF module of the same name")
            setattr(self, name, child)
        for name, p in backbone.named_parameters(recurse=False):
            self.register_parameter(name, p)
        for name, b in backbone.named_buffers(recurse=False):
            self.register_buffer(name, b)

    def train(self, mode=True):
        super().train(mode)
        self.off.train(mode)                          # dropout of the OFF section follows the model (RGB_OFF.py:356)
        if self.backbone is not None:
            self.backbone.training = mode             # its layers are children of this class and were switched above
        return self

    def _apply(self, fn, recurse=True):
        """``.cuda()`` / ``.to()`` / ``.float()`` place the feature extractor; the OFF parameters are views of the engine's
        flat CUDA buffer and must not be replaced by moved / cast copies (the kernels would keep reading the buffer):
        they are routed through ``OFFSubNetwork._apply`` (a no-op on the right device / dtype, an error otherwise)."""
        self.off._apply(fn)
        order = list(self._modules.items())
        for n in self._off_children:
            self._modules.pop(n)
        try:
            super()._apply(fn)
        finally:
            held = dict(order)
            self._modules.clear()
            for n, m in order:
                self._modules[n] = held[n]
        return self

    def _taps_and_score(self, input):
        if self.backbone is None:
            if not isinstance(input, (dict, list, tuple)):
                raise RuntimeError("BNInception_OFF was built without a backbone: pass the nine Inception taps "
                                   "('3a'..'5b'), or construct it with backbone=<module returning (taps, score)>")
            return input, None, None
        if hasattr(self.backbone, "plan"):            # FusedBNInception: its pass is replayed as a graph with the OFF passes
            self.backbone.use_graphs = self.off.use_graphs
        out = self.backbone(input)
        taps, score = out[0], out[1]
        extra = out[2] if len(out) > 2 else None
        return taps, score, extra

    # ------------------------------------------------------------------ reference entry points
    def RGB_OFF_forward(self, input):
        """RGB_OFF.py:360-860: per-pair logits, no consensus (it is commented out there, :849-858)."""
        taps, score, _ = self._taps_and_score(input)
        fc7, _fc28, fc14 = self.off(taps)
        if fc7.shape[0] == 1:
            # one frame pair (batch 1, two segments): the reference's torch.squeeze before the Linear drops the batch
            # dimension too, so its heads return [101] (RGB_OFF.py:786,792,846)
            fc7, fc14 = fc7.squeeze(0), fc14.squeeze(0)
        return fc7, score, fc14

    def forward(self, input):
        if self.variant == "rgb":
            # RGB_OFF.forward is the plain TSN backbone classifier (RGB_OFF.py:1340-1344); the OFF entry point of that
            # class is RGB_OFF_forward
            if self.backbone is None:
                raise RuntimeError("RGB_OFF.BNInception_OFF.forward is the backbone classifier; use RGB_OFF_forward "
                                   "for the OFF path or pass a backbone")
            return self.backbone(input)[1]
        taps, score, extra = self._taps_and_score(input)
        fc7, _fc28, fc14 = self.off(taps)             # consensus over the L-1 pairs happens inside (Flow_OFF.py:873-876)
        if score is not None:                         # Feature_Generation_Score: consensus over the L segments (:867,872)
            score = self.consensus(score.reshape(self.batch, self.length, -1).contiguous()).squeeze(1)
        if self.modality_fuse:                        # Flow_OFF.py:879-881
            if score is None:
                raise RuntimeError("modality_fuse needs the backbone score (Feature_Generation_Score)")
            return fc7 + score + fc14
        if self.variant == "rgb_v2":
            return fc7, score, fc14, extra            # RGB_OFF_v2.py:891
        return fc7, score, fc14                       # Flow_OFF.py:884


def bninception_off(num_classes=1000, batch=1, num_seg=25, variant="rgb", **kw):
    """RGB_OFF.py:1346-1360 (variant='rgb'), Flow_OFF.py:1371-1385 ('flow'), RGB_OFF_v2.py:1378-1392 ('rgb_v2')."""
    return BNInception_OFF(num_classes, batch, num_seg, variant=variant, **kw)


def bninception_off_sobel(num_classes=1000, batch=1, num_seg=25, **kw):
    """RGB_OFF.py:1363-1377: identical body to bninception_off in the reference."""
    return BNInception_OFF(num_classes, batch, num_seg, variant="rgb", **kw)
