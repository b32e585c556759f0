"""nn.Module surface of the OFF sub-network (drop-in for the OFF section of the reference classes).

``OFFSubNetwork`` owns the parameters under the reference's names
(``motion_conv_gen_3a.weight`` ... ``fc_action_motion_14.bias``, RGB_OFF.py:265-334; plus the frozen
``sobel_edge_diagonal.conv.weight`` for the Flow / v2 variant, util.py:66,72) as views into the engine's flat
parameter buffer, and runs forward/backward through liboffk via one ``torch.autograd.Function``.
"""
from __future__ import annotations

import os
from collections import OrderedDict

import torch
import torch.nn as nn

from . import spec as S
from .engine import OFFEngine


class _Holder(nn.Module):
    """Stands in for an nn.Conv2d / nn.Linear of the reference: only carries .weight / .bias."""

    def __init__(self, weight=None, bias=None, trainable=True):
        super().__init__()
        if weight is not None:
            self.weight = nn.Parameter(weight, requires_grad=trainable)
        if bias is not None:
            self.bias = nn.Parameter(bias, requires_grad=trainable)


class _Prefetched:
    """Handle returned by OFFSubNetwork.prefetch(): an input set that is being filled on the copy stream."""

    def __init__(self, index, event):
        self.index, self.event = index, event


_NO_GRAD = ("fc_action_motion_28.weight", "fc_action_motion_28.bias")


def _step_seed():
    """Dropout seed of one training forward: drawn from torch's default CPU generator (so torch.manual_seed reproduces a
    run and a resumed run does not replay the masks of step 1), offset per rank so data-parallel replicas differ."""
    s = int(torch.randint(0, 1 << 62, (1,)).item())
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        s = (s + 0x9E3779B97F4A7C15 * (torch.distributed.get_rank() + 1)) & ((1 << 63) - 1)
    return s


class _OFFFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, train, masks, seed, n_taps, *tensors):
        eng = net.engine
        taps = tensors[:n_taps]
        if any(t.device.type != "cuda" for t in taps):
            # host tensors: stage them into the idle input set on the copy stream, then switch to it
            idx, ev = eng.stage_taps(dict(zip(eng.taps, taps)))
            torch.cuda.current_stream(eng.device).wait_event(ev)
            eng.select_taps(idx)
        else:
            own = [i for i, ts in enumerate(eng.tap_sets)
                   if all(t.data_ptr() == b.data_ptr() for t, b in zip(taps, ts.values()))]
            if own:                                     # the engine's own input buffers need no copy
                if own[0] != eng._tap_set:
                    eng.select_taps(own[0])
            else:
                for buf, t in zip(eng.taps.values(), taps):
                    buf.copy_(t, non_blocking=True)
        fc7, fc28, fc14 = eng.forward(train=train, masks=masks, seed=seed, graph=net.use_graphs and masks is None)
        ctx.graph = net.use_graphs and masks is None
        ctx.generation = eng.generation                 # the engine keeps ONE set of activations: see backward()
        ctx.net = net
        ctx.n_taps = n_taps
        ctx.tap_needs = [t.requires_grad for t in taps]
        out = (fc7.clone(), fc28.clone(), fc14.clone())
        ctx.mark_non_differentiable(out[1])             # fc28 is never returned by the reference (RGB_OFF.py:860)
        return out

    @staticmethod
    def backward(ctx, g7, g28, g14):
        net, eng = ctx.net, ctx.net.engine
        if ctx.generation != eng.generation:
            raise RuntimeError(
                "OFFSubNetwork.backward: the module ran another forward since the one this graph belongs to. The "
                "engine keeps one set of static activation buffers (no per-call saved tensors), so each backward must "
                "follow its own forward: run forward -> backward per input, or use one module per concurrent graph.")
        if any(ctx.tap_needs) and not eng.tap_grads:
            raise RuntimeError("tap gradients requested but the module was built with tap_grads=False "
                               "(the reference freezes the backbone, train_off.py:39-46)")
        params = net._flat_params
        views = [eng.grads[n] for n in eng.grads]
        # parameters the backward plan never writes get NO gradient, as in the reference, where fc_action_motion_28 is
        # not part of any returned output (RGB_OFF.py:787,860): .grad stays None, optimizers skip them (no weight decay)
        live = [n not in _NO_GRAD for n in eng.grads]
        aliased = [p.grad is not None and p.grad.data_ptr() == v.data_ptr() for p, v, l in zip(params, views, live) if l]
        in_place = all(aliased)                          # .grad already lives in the flat buffer: accumulate there
        if any(aliased) and not in_place:
            for p, a in zip([p for p, l in zip(params, live) if l], aliased):
                if a:
                    p.grad = p.grad.clone()
        g7 = torch.zeros_like(eng.d_out7) if g7 is None else g7
        g14 = torch.zeros_like(eng.d_out14) if g14 is None else g14
        eng.backward(g7.contiguous(), g14.contiguous(), zero_grads=not in_place, graph=ctx.graph and not in_place)
        pgrads = [None] * len(params) if in_place else [eng._view(eng.grads_flat, n) if l else None
                                                        for n, l in zip(eng.grads, live)]
        tgrads = [eng.tap_grad[tag].clone() if need else None
                  for tag, need in zip(eng.taps, ctx.tap_needs)] if eng.tap_grads else [None] * ctx.n_taps
        return (None, None, None, None, None, *tgrads, *pgrads)


class OFFSubNetwork(nn.Module):
    """The OFF units + 28/14/7 residual stages + heads of ``BNInception_OFF`` (RGB_OFF.py:596-860).

    forward(taps) -> (fc7, fc28, fc14); ``taps`` maps '3a'..'5b' to the BN-Inception feature maps
    ``[batch*length, C, S, S]`` (fp32, NCHW, CUDA).  variant='rgb': learned depth-wise 3x3 spatial gradient, per-pair
    logits ``[batch*(length-1), 101]``; variant='flow' (also RGB_OFF_v2): fixed diagonal Sobel and segment consensus
    ``[batch, 101]``.  Dropout follows ``self.training`` (p = 0.8, RGB_OFF.py:356); pass ``masks`` to inject keep-masks.
    ``precision``: 'fp32' = fp32-parity arithmetic on the tensor cores (3xTF32), 'tf32' = single-MMA tf32 (the default here,
    the fast mode).  ``use_graphs``: replay each pass as one captured CUDA graph.  ``tap_layout='channels_last'``: the
    engine's tap buffers are channels-last (what ``FusedBNInception`` writes in place); other taps are copied into them.
    """

    def __init__(self, batch: int, length: int, variant: str = "rgb", precision: str = "tf32",
                 index_mode: str = "reference_flat", consensus=None, tap_grads: bool = False, device="cuda",
                 use_graphs=None, tap_layout: str = "nchw"):
        super().__init__()
        self.batch, self.length, self.variant = batch, length, variant
        # forward / backward as one captured CUDA graph each (same kernels, no per-launch host cost); OFFK_GRAPHS=1 turns it
        # on for modules that do not say
        self.use_graphs = (os.environ.get("OFFK_GRAPHS", "0") == "1") if use_graphs is None else bool(use_graphs)
        self.engine = OFFEngine(batch, length, variant, device, precision, index_mode, consensus, tap_grads, tap_layout)
        self._seed = 0
        groups = OrderedDict()
        for name in S.param_shapes(variant):
            mod, leaf = name.rsplit(".", 1)
            groups.setdefault(mod, {})[leaf] = self.engine.params[name]
        for mod, d in groups.items():
            setattr(self, mod, _Holder(d.get("weight"), d.get("bias")))
        if variant == "flow":
            self.sobel_edge_diagonal = nn.Module()
            self.sobel_edge_diagonal.conv = _Holder(self.engine.sobel_w, None, trainable=False)
        self._flat_params = [getattr(getattr(self, n.rsplit(".", 1)[0]), n.rsplit(".", 1)[1])
                             for n in S.param_shapes(variant)]
        self.reset_parameters()

    @torch.no_grad()
    def reset_parameters(self):
        """Default nn.Conv2d / nn.Linear init of the reference modules: U(-1/sqrt(fan_in), 1/sqrt(fan_in))."""
        fan = 1
        for name, p in zip(S.param_shapes(self.variant), self._flat_params):
            if name.endswith(".weight"):
                fan = p[0].numel()
            p.uniform_(-1.0 / fan ** 0.5, 1.0 / fan ** 0.5)

    def tap_buffers(self):
        """The engine's static input buffers; filling these (e.g. as the H2D copy target) avoids a device copy."""
        return self.engine.taps

    def prefetch(self, taps):
        """Start the asynchronous host->device copy of the NEXT step's taps (dict or list of host tensors, pinned
        for a truly asynchronous copy) into the idle input set while the current step still computes.  Returns a
        handle to pass to forward() in place of the taps."""
        if not isinstance(taps, dict):
            taps = dict(zip(S.LEVELS, taps))
        return _Prefetched(*self.engine.stage_taps(taps))

    def _apply(self, fn, recurse=True):
        probe = fn(self.engine.params_flat[:1])
        if probe.device == self.engine.params_flat.device and probe.dtype == torch.float32:
            return self                                   # .cuda() / .float() on the right device: nothing to do
        raise RuntimeError("OFFSubNetwork parameters are views of one flat CUDA buffer; construct the module on its "
                           "device instead of moving / casting it")

    def forward(self, taps, masks=None):
        if isinstance(taps, _Prefetched):
            eng = self.engine
            torch.cuda.current_stream(eng.device).wait_event(taps.event)
            eng.select_taps(taps.index)
            taps = eng.taps
        if isinstance(taps, dict):
            taps = [taps[t] for t in S.LEVELS]
        train = self.training
        self._seed = _step_seed() if (train and masks is None) else 0
        return _OFFFunction.apply(self, train, masks, self._seed, len(taps), *taps, *self._flat_params)
