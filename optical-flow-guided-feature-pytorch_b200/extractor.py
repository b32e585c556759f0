"""The frozen BN-Inception extractor on liboffk: ``FusedBNInception`` runs the forward of ``BNInceptionBackbone``
(RGB_OFF.py:43-263,362-594; 10-channel stem Flow_OFF.py:53) as a static plan of tensor-core GEMMs and channels-last pools
for a fixed number of frames.

* Every BatchNorm runs on its running statistics (train_off.py:53-57) and is folded into its conv:
  ``w' = w * g / sqrt(var + eps)``, ``b' = (b - mean) * g / sqrt(var + eps) + beta``.  The folded weights sit OHWI in one
  flat buffer (plus their tf32 residuals behind it in the fp32 mode, as in the OFF engine).  The fold is redone before a
  forward whenever a parameter or buffer of the module changed since the last one (``load_state_dict``, an optimizer, ...).
* The image batch is converted to channels-last with 4 (RGB) or 12 (flow) channels, so the 7x7 stem is a gather-fed GEMM
  with 16-byte channel groups; every other conv is one TMA-fed GEMM (``plan.TGemm``) with bias + ReLU in its epilogue,
  writing its channel slice of the module's channels-last output: the Inception concatenations cost nothing.
* The nine tap modules write straight into the tap buffers of the OFF engine the extractor is paired with (its first input
  set, channels-last), so the OFF forward reads them in place.

It is a subclass of ``BNInceptionBackbone``: same children, parameters, buffers and state_dict keys.  It is forward-only
(the extractor is frozen, train_off.py:39-46) and takes CUDA fp32 input only; ``BNInceptionBackbone`` stays the path for
CPU tensors and the reference the tests compare against.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict

import numpy as np
import torch

from . import _lib as L
from . import tables as T
from .backbone import BNInceptionBackbone, TAPS, _NORMAL, _ORDER, _REDUCE
from .plan import Gemm, LaunchPlan, Schedule, _nm, _ptr

IMG = 224                                      # input resolution of the TSN BN-Inception (RGB_OFF.py:362)


def _module_channels(tag):
    """(input channels, output channels, input size, output size) of Inception module ``tag``."""
    size = {"3a": 28, "3b": 28, "3c": 28, "4a": 14, "4b": 14, "4c": 14, "4d": 14, "4e": 14, "5a": 7, "5b": 7}[tag]
    if tag in _NORMAL:
        cin, n1, _, n3, _, d, pp, _ = _NORMAL[tag]
        return cin, n1 + n3 + d + pp, size, size
    cin, _, n3, _, d = _REDUCE[tag]
    return cin, n3 + d + cin, size, size // 2


class ExtractorPlan(LaunchPlan):
    """Buffers, folded weights and launch list of one ``FusedBNInception`` forward over ``n_frames`` images."""

    def __init__(self, net: BNInceptionBackbone, n_frames: int, in_channels: int, num_classes: int, precision: str,
                 device, taps=None):
        super().__init__(device, precision)
        self.N = n_frames
        self.cin, self.c_pad = in_channels, (in_channels + 3) // 4 * 4
        self.num_classes = num_classes
        N, dev = n_frames, self.device

        # ---- folded weights: name -> (offset, cout, kh, kw, cin of the weight rows), OHWI; biases in their own buffer
        self.convs = OrderedDict()
        off = boff = 0
        for name, conv in net.named_children():
            if not isinstance(conv, torch.nn.Conv2d):
                continue
            cin = self.c_pad if name == "conv1_7x7_s2" else conv.in_channels
            kh, kw = conv.kernel_size
            self.convs[name] = (off, boff, conv.out_channels, kh, kw, cin)
            off += (conv.out_channels * kh * kw * cin + 3) // 4 * 4
            boff += (conv.out_channels + 3) // 4 * 4
        self.fc_off, self.fc_boff = off, boff
        off += (num_classes * 1024 + 3) // 4 * 4
        boff += (num_classes + 3) // 4 * 4
        self.w_flat, self.w_lo = self._weights(off)
        self.b_flat = torch.zeros(boff, device=dev)
        self.folded_key = None

        # ---- activations, channels-last
        nhwc = lambda s, c: torch.zeros(N, s, s, c, device=dev)
        self.buf = OrderedDict()
        self.buf["image"] = nhwc(IMG, self.c_pad)
        self.buf["conv1"] = nhwc(112, 64)
        self.buf["pool1"] = nhwc(56, 64)
        self.buf["conv2_red"] = nhwc(56, 64)
        self.buf["conv2"] = nhwc(56, 192)
        self.buf["pool2"] = nhwc(28, 192)
        if taps is None:
            taps = OrderedDict((t, None) for t in TAPS)
        self.taps = OrderedDict()
        for tag in _ORDER:
            cin, ctot, s_in, s_out = _module_channels(tag)
            if tag in TAPS:
                t = taps[tag]
                if t is None:
                    t = nhwc(s_out, ctot).permute(0, 3, 1, 2)
                if (tuple(t.shape) != (N, ctot, s_out, s_out) or t.dtype != torch.float32 or t.device != dev
                        or not t.is_contiguous(memory_format=torch.channels_last)):
                    raise ValueError(f"tap {tag}: needs a channels-last fp32 [{N}, {ctot}, {s_out}, {s_out}] tensor on {dev}")
                self.taps[tag] = t
                self.buf["out_" + tag] = t.permute(0, 2, 3, 1)           # its channels-last storage, [N, S, S, C]
            else:
                self.buf["out_" + tag] = nhwc(s_out, ctot)
            p = f"inception_{tag}_"
            for br in ("3x3_reduce", "double_3x3_reduce", "double_3x3_1"):
                self.buf[p + br] = nhwc(s_in, getattr(net, p + br).out_channels)
            if tag in _NORMAL:
                self.buf[p + "pool"] = nhwc(s_in, cin)
        self.buf["pooled"] = torch.zeros(N, 1024, device=dev)
        self.buf["score"] = torch.zeros(N, num_classes, device=dev)
        self._src = None                 # image batch the conversion step reads (set per forward)
        self._net = net
        self._build()
        del self._net

    # ------------------------------------------------------------------ plan
    def _w(self, name):
        off, boff, cout, kh, kw, cin = self.convs[name]
        return self.w_flat[off:off + cout * kh * kw * cin].view(cout, kh * kw * cin), self.b_flat[boff:boff + cout]

    def _conv(self, name, x, y, s_in, *, y_ctot=0, y_coff=0):
        """conv + folded BN + ReLU as one TMA-fed GEMM into channels [y_coff, y_coff + cout) of y."""
        _, _, cout, k, _, cin = self.convs[name]
        conv = getattr(self._net, name)
        geom = T.ConvGeom(self.N, cin, s_in, s_in, cout, k, k, conv.stride[0], conv.padding[0], y_ctot=y_ctot, y_coff=y_coff)
        w, b = self._w(name)
        # split-K accumulates into a zeroed buffer of its own; a channel slice of a concatenation is written once
        self.steps += self._conv_fwd(name, x, y, geom, w, b, relu=True, no_split=geom.y_ctot != cout)
        return geom

    def _pool(self, name, x, s_in, c, stride, pad, kind, y, y_ctot, y_coff):
        lib, N = self.lib, self.N
        x_ctot = x.shape[-1]

        def run(stream):
            L.check(lib.offk_pool3_nhwc(_ptr(x), N, s_in, s_in, x_ctot, 0, c, stride, pad, kind, _ptr(y), y_ctot, y_coff,
                                        stream), name)
        self.steps.append(_nm(run, name, reads=[x], writes=[y]))

    def _build(self):
        bf, N, lib = self.buf, self.N, self.lib
        self.steps = []

        def convert(stream):
            L.check(lib.offk_image_to_nhwc(_ptr(self._src), _ptr(bf["image"]), N, self.cin, IMG * IMG, self.c_pad, stream),
                    "image_to_nhwc")
        self.steps.append(_nm(convert, "image_to_nhwc", writes=[bf["image"]]))
        # ---- stem: 7x7 / 2 over 4 or 12 channels, gather-fed (cin % 32 != 0 has no im2col tensor map)
        g1 = T.ConvGeom(N, self.c_pad, IMG, IMG, 64, 7, 7, 2, 3)
        spc = T.conv_fwd_spec(g1, "nhwc", "nhwc")
        w, b = self._w("conv1_7x7_s2")
        stem = Gemm(self, spc, ("stem", self.c_pad, N), a_src=bf["image"], b_src=w, out=bf["conv1"], bias=b,
                    relu_pre_cols=64, name="conv1_7x7_s2")
        self.steps.append(stem)
        self.flops_fwd += 2.0 * spc.M * 64 * 49 * self.cin          # the zero padding channels are not algorithmic work
        self._pool("pool1", bf["conv1"], 112, 64, 2, 0, L.POOL_MAX, bf["pool1"], 64, 0)
        self._conv("conv2_3x3_reduce", bf["pool1"], bf["conv2_red"], 56)
        self._conv("conv2_3x3", bf["conv2_red"], bf["conv2"], 56)
        self._pool("pool2", bf["conv2"], 56, 192, 2, 0, L.POOL_MAX, bf["pool2"], 192, 0)
        # ---- Inception modules: each branch writes its channel slice of the module output (the torch.cat)
        x = bf["pool2"]
        for tag in _ORDER:
            p = f"inception_{tag}_"
            cin, ctot, s, _ = _module_channels(tag)
            out = bf["out_" + tag]
            c0 = 0
            if tag in _NORMAL:
                _, n1, _, n3, _, d, pp, kind = _NORMAL[tag]
                self._conv(p + "1x1", x, out, s, y_ctot=ctot, y_coff=0)
                c0 = n1
            else:
                _, _, n3, _, d = _REDUCE[tag]
            self._conv(p + "3x3_reduce", x, bf[p + "3x3_reduce"], s)
            self._conv(p + "3x3", bf[p + "3x3_reduce"], out, s, y_ctot=ctot, y_coff=c0)
            c0 += n3
            self._conv(p + "double_3x3_reduce", x, bf[p + "double_3x3_reduce"], s)
            self._conv(p + "double_3x3_1", bf[p + "double_3x3_reduce"], bf[p + "double_3x3_1"], s)
            self._conv(p + "double_3x3_2", bf[p + "double_3x3_1"], out, s, y_ctot=ctot, y_coff=c0)
            c0 += d
            if tag in _NORMAL:
                # avg: count_include_pad=True (RGB_OFF.py:73 ...); 5b: max (:253)
                self._pool(p + "pool", x, s, cin, 1, 1, L.POOL_AVG if kind == "avg" else L.POOL_MAX, bf[p + "pool"], cin, 0)
                self._conv(p + "pool_proj", bf[p + "pool"], out, s, y_ctot=ctot, y_coff=c0)
            else:
                self._pool(p + "pool", x, s, cin, 2, 0, L.POOL_MAX, out, ctot, c0)
            x = out
        # ---- score: global 7x7 average pool, then last_linear as a GEMM (num_classes up to 1000)
        x5b, pooled = bf["out_5b"], bf["pooled"]

        def gpool(stream):
            L.check(lib.offk_avgpool_drop_fwd(_ptr(x5b), N, 1024, 49, 1024, 0, L.DROP_NONE, None, 0, None, 0.0, 1.0,
                                              _ptr(pooled), stream), "global_pool")
        self.steps.append(_nm(gpool, "global_pool", reads=[x5b], writes=[pooled]))
        gfc = T.ConvGeom(N, 1024, 1, 1, self.num_classes)
        wfc = self.w_flat[self.fc_off:self.fc_off + self.num_classes * 1024].view(self.num_classes, 1024)
        bfc = self.b_flat[self.fc_boff:self.fc_boff + self.num_classes]
        self.steps += self._conv_fwd("last_linear", pooled, bf["score"], gfc, wfc, bfc, no_split=True)
        # parameters are read-only inside a pass; the image is written by the conversion step only
        self.sched = Schedule(self.steps, ignore=[self.w_flat, self.b_flat] + ([self.w_lo] if self.presplit else []))
        self._graph = None
        self._graph_src = None

    # ------------------------------------------------------------------ weights
    @torch.no_grad()
    def fold(self, net):
        """Fold every BatchNorm (running statistics) into its conv and lay the weights out OHWI; in the fp32 mode also
        write their tf32 residuals.  Torch ops on the device, issued on the current stream."""
        for name, (off, boff, cout, kh, kw, cin) in self.convs.items():
            conv, bn = getattr(net, name), getattr(net, name + "_bn")
            scale = bn.weight.double() / torch.sqrt(bn.running_var.double() + bn.eps)
            w = (conv.weight.double() * scale[:, None, None, None]).permute(0, 2, 3, 1)      # OHWI
            dst = self.w_flat[off:off + cout * kh * kw * cin].view(cout, kh, kw, cin)
            dst.zero_()
            dst[..., :w.shape[-1]].copy_(w)
            self.b_flat[boff:boff + cout].copy_((conv.bias.double() - bn.running_mean.double()) * scale + bn.bias.double())
        fc = net.last_linear
        self.w_flat[self.fc_off:self.fc_off + fc.weight.numel()].copy_(fc.weight.reshape(-1))
        self.b_flat[self.fc_boff:self.fc_boff + fc.bias.numel()].copy_(fc.bias)
        if self.presplit:
            main = torch.cuda.current_stream(self.device)
            L.check(self.lib.offk_tf32_residual(_ptr(self.w_flat), _ptr(self.w_lo), self.w_flat.numel(),
                                                C.c_void_p(main.cuda_stream)), "extractor weight residuals")

    # ------------------------------------------------------------------ run
    def _issue(self):
        self.sched.run([torch.cuda.current_stream(self.device)])

    def run(self, x, graph=False):
        if not graph:
            self._src = x
            self._issue()
            return
        if self._graph is None:
            self._graph_src = torch.empty_like(x)
            self._src = self._graph_src
            self._graph = self._capture(self._issue)
        if x.data_ptr() != self._graph_src.data_ptr():
            self._graph_src.copy_(x)
        self._graph.replay()


class FusedBNInception(BNInceptionBackbone):
    """``BNInceptionBackbone`` whose forward runs on liboffk for a fixed ``n_frames`` (= batch * length) and
    ``precision`` ('fp32' = 3xTF32, 'tf32').  forward(images [n_frames, 3 | 10, 224, 224], CUDA fp32) -> (taps, score,
    conv2_relu_3x3_out) like the stock module; the taps and conv2 are [N, C, S, S] views in torch.channels_last memory
    format of the plan's static buffers (``taps``: the paired OFF engine's), overwritten by the next forward.

    taps: optional dict '3a'..'5b' of channels-last tensors to write the taps into (``OFFEngine.tap_sets[0]`` of the
    OFF section this extractor feeds).  use_graphs: replay the pass as one captured CUDA graph."""

    def __init__(self, num_classes=101, in_channels=3, n_frames=1, precision="tf32", device="cuda", taps=None,
                 use_graphs=False):
        super().__init__(num_classes, in_channels)
        self.to(device)
        self.n_frames, self.in_channels, self.precision = n_frames, in_channels, precision
        self.use_graphs = bool(use_graphs)
        # a plain attribute, not a child module: it owns device buffers, no parameters
        object.__setattr__(self, "plan", ExtractorPlan(self, n_frames, in_channels, num_classes, precision, device, taps))

    def _state_key(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    @torch.no_grad()
    def forward(self, x):
        plan = self.plan
        if not isinstance(x, torch.Tensor) or x.device.type != "cuda" or x.dtype != torch.float32:
            raise RuntimeError("FusedBNInception takes a CUDA float32 image batch; use BNInceptionBackbone for other input")
        if x.device != plan.device:
            raise RuntimeError(f"FusedBNInception: input on {x.device}, plan on {plan.device}")
        want = (self.n_frames, self.in_channels, IMG, IMG)
        if tuple(x.shape) != want:
            raise RuntimeError(f"FusedBNInception: the plan is built for images {list(want)}, got {list(x.shape)}")
        x = x.contiguous()
        key = self._state_key()
        if key != plan.folded_key:
            plan.fold(self)
            plan.folded_key = key
        plan.run(x, graph=self.use_graphs)
        return OrderedDict(plan.taps), plan.buf["score"].clone(), plan.buf["conv2"].permute(0, 3, 1, 2)
