"""OFFEngine: the OFF sub-network (RGB_OFF.py:596-860 / Flow_OFF.py:606-884) as a static plan of
liboffk kernel launches over preallocated fp32 buffers.

Layout: the taps arrive NCHW (the reference's layout); the unit's fused 1x1 GEMM reads them in place through a TMA
tensor map (MN-major operand), converts to channels-last in its epilogue, and everything downstream (reduced
features, stage-fusion buffers, residual blocks, gradients) is NHWC, so that every operand tile is a TMA box or a
16-byte cp.async gather.

Every step is one C-ABI call with a descriptor bound at plan-build time; a forward or backward pass is a flat list of
launches spread over up to three streams by a hazard-derived schedule (class Schedule).  PyTorch supplies device
memory and streams only.
"""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict

import numpy as np
import torch

from . import _lib as L
from . import spec as S
from . import tables as T
from .plan import (_OUT_TABLES, _SM_TARGET, _FreeGeom, Gemm, LaunchPlan, Schedule, TGemm, _gkey, _kernels, _nm, _on,
                   _pick_tile_n, _ptr, _wgrad_split)
from .plan import _auto_tile_n, _names  # noqa: F401  (re-exported: bench.py and the tests import them from here)


class OFFEngine(LaunchPlan):
    """Plan + buffers for one (batch, length) shape on one GPU.

    tap_layout: 'nchw' (the reference's layout) or 'channels_last': both tap sets are [N, C, S, S] tensors in
               torch.channels_last memory format (what the fused BN-Inception extractor writes), and every unit reads its
               tap through dense / im2col tensor maps in place, as the NCHW plan does for the 7x7 levels through a copy

    variant: 'rgb'  learned depth-wise 3x3 spatial gradient + bias, per-pair logits (RGB_OFF.py)
             'flow' fixed diagonal Sobel, segment consensus over the L-1 pairs (Flow_OFF.py / RGB_OFF_v2.py)
    precision: 'fp32' = fp32-parity mode ON THE TENSOR CORES (OFFK_PREC_TF32X3: error-compensated 3xTF32 tcgen05 MMAs,
               fp32 accumulate; the reference's arithmetic is fp32, RGB_OFF.py:597), 'tf32' = one kind::tf32 MMA per
               product (the fast mode, tolerance stated separately)
    """

    def __init__(self, batch: int, length: int, variant: str = "rgb", device="cuda", precision: str = "tf32",
                 index_mode: str = "reference_flat", consensus=None, tap_grads: bool = False, tap_layout: str = "nchw"):
        assert variant in ("rgb", "flow") and length >= 2 and batch >= 1
        if tap_layout not in ("nchw", "channels_last"):
            raise ValueError(f"tap_layout: 'nchw' or 'channels_last', not {tap_layout!r}")
        if tap_grads and tap_layout == "channels_last":
            # the channels-last taps come from the frozen fused extractor (train_off.py:39-46): nothing consumes their gradient
            raise ValueError("tap_grads=True needs tap_layout='nchw': channels-last taps come from the frozen extractor")
        super().__init__(device, precision)
        self.tap_layout = tap_layout
        self.B, self.Lseg, self.variant = batch, length, variant
        self.N, self.P = batch * length, batch * (length - 1)
        self.precision = precision
        self.index_mode = {"reference_flat": L.INDEX_REFERENCE_FLAT, "aligned": L.INDEX_ALIGNED}[index_mode]
        self.consensus = (variant != "rgb") if consensus is None else bool(consensus)
        self.tap_grads = tap_grads
        self.single_stream = False       # True: issue every lane on the caller's stream (profiling / debugging)
        self.generation = 0

        # ---- parameters: one flat buffer, reference-named views
        self.layout, self.n_flat = S.flat_layout(variant)
        self.params_flat, self.params_lo = self._weights(self.n_flat)
        self.grads_flat = torch.zeros(self.n_flat, device=self.device)
        self.params = OrderedDict((n, self._view(self.params_flat, n)) for n in S.param_shapes(variant))
        self.grads = OrderedDict((n, self._view(self.grads_flat, n)) for n in S.param_shapes(variant))
        if variant == "flow":
            # frozen util.SobelFilter_Diagonal taps (util.py:61), [32,1,3,3]
            k = torch.tensor([[0., 1., 0.], [-1., 0., 1.], [0., -1., 0.]], device=self.device)
            self.sobel_w = k.expand(S.DOWN_C, 1, 3, 3).contiguous()

        self._alloc()
        self._build()

    # ------------------------------------------------------------------ helpers
    def _view(self, flat, name):
        off, shape = self.layout[name]
        return flat[off:off + int(np.prod(shape))].view(shape)

    def _unit_w(self, flat, tag):
        off, _ = self.layout[f"motion_conv_gen_{tag}.weight"]
        cin = S.LEVELS[tag][0]
        return flat[off:off + S.UNIT_C * cin].view(S.UNIT_C, cin)

    def _unit_b(self, flat, tag):
        off, _ = self.layout[f"motion_conv_gen_{tag}.bias"]
        return flat[off:off + S.UNIT_C]

    def _buf(self, name, *shape):
        t = torch.zeros(*shape, device=self.device)
        self.buf[name] = t
        return t

    def load_params(self, prm: dict):
        """Copy reference-named tensors (a state_dict subset) into the flat buffer."""
        with torch.no_grad():
            for n, v in self.params.items():
                v.copy_(prm[n].to(self.device, torch.float32))

    # ------------------------------------------------------------------ buffers
    def _alloc(self):
        P, N = self.P, self.N
        self.buf = {}
        for tag, (cin, s) in S.LEVELS.items():
            self._buf("gd_" + tag, N, s, s, S.UNIT_C)
            self._buf("dgd_" + tag, N, s, s, S.UNIT_C)
        for st, (ctot, s, _) in S.STAGES.items():
            self._buf("F" + st, P, s, s, ctot)
            self._buf("dF" + st, P, s, s, ctot)
        a = lambda n, c, s: (self._buf(n, P, s, s, c), self._buf("d_" + n, P, s, s, c))
        a("t28", 64, 14)
        self._buf("t28r", P, 14, 14, 64)          # relu(t28): conv1_trans_28a consumes the activated copy (RGB_OFF.py:658-659)
        a("tmp28", 64, 14)
        for blk in "abc":
            a("h1_28" + blk, 64, 14)
            a("h2_28" + blk, 64, 14)
        a("br28", 256, 14)
        a("s28a", 256, 14)
        a("s28b", 256, 14)
        a("t14", 128, 7)
        a("tmp14", 128, 7)
        for blk in "ab":
            a("h1_14" + blk, 128, 7)
            a("h2_14" + blk, 128, 7)
        a("ex14", 512, 7)
        a("s14a", 512, 7)
        a("h3_14b", 512, 7)
        a("t7", 256, 7)
        a("tmp7", 256, 7)
        a("h1_7", 256, 7)
        a("h2_7", 256, 7)
        a("br7", 1024, 7)
        a("s7", 1024, 7)
        self._buf("p28", P, 7, 7, 256)
        for k, c in (("7", 1024), ("14", 512), ("28", 256)):
            self._buf("pool" + k, P, c)
            self._buf("fc" + k, P, S.NUM_CLASSES)
            if self.consensus:
                self._buf("cfc" + k, self.B, S.NUM_CLASSES)
        # two input sets: while one is being consumed (forward AND backward read the taps) the other can be filled by
        # an asynchronous host->device copy (stage_taps)
        if self.tap_layout == "channels_last":      # [N, C, S, S] views of [N, S, S, C] storage
            tap = lambda cin, s: torch.zeros(N, s, s, cin, device=self.device).permute(0, 3, 1, 2)
        else:
            tap = lambda cin, s: torch.zeros(N, cin, s, s, device=self.device)
        self.tap_sets = [OrderedDict((tag, tap(cin, s)) for tag, (cin, s) in S.LEVELS.items()) for _ in range(2)]
        self.taps = self.tap_sets[0]
        self._tap_set = 0
        self._tap_users = {tag: [] for tag in S.LEVELS}      # bound GEMMs whose A operand is the tap
        self._copy_stream = None
        if self.tap_grads:
            self.tap_grad = OrderedDict((tag, torch.zeros_like(t)) for tag, t in self.taps.items())
        # Per-step weight re-layouts, produced by ONE gather-copy launch (wc_flat[i] = params_flat[wc_idx[i]]):
        #   wp[name] : OHWI [cout, kh, kw, cin] copies of the KxK conv weights (K order of the channels-last implicit GEMM)
        #   wd[name] : [cin, kh, kw, cout] copies with flipped taps of every stride-1 conv = the B operand of its
        #              data-gradient GEMM (dX = dY * W^T as a forward conv over dY)
        # dwp[name]: OHWI accumulators of the KxK weight gradients (un-permuted into grads_flat after the backward)
        self.wp, self.dwp, self.wd = {}, {}, {}
        kxk = [(name, cout, cin, k) for name, cout, cin, k, _, _ in S.STAGE_CONVS if k > 1]
        total = sum(cout * cin * k * k for _, cout, cin, k in kxk)
        self.dwp_flat = torch.zeros(total, device=self.device)
        idx, off, views = [], 0, []
        for name, cout, cin, k, stride, pad in S.STAGE_CONVS:
            p_off = self.layout[name + ".weight"][0]
            oihw = p_off + np.arange(cout * cin * k * k, dtype=np.int64).reshape(cout, cin, k, k)
            if k > 1:
                idx.append(oihw.transpose(0, 2, 3, 1).reshape(-1))
                views.append(("wp", name, off, (cout, k, k, cin)))
                off += oihw.size
            if stride == 1:
                idx.append(p_off + T.dgrad_class_weight_index(cout, cin, k, 1, pad, 0, 0))
                views.append(("wd", name, off, (cin, k * k * cout)))
                off += oihw.size
            else:
                # one [cin, R, Q, cout] block per stride-parity class (a, b) of the input pixel
                for a in range(stride):
                    for b in range(stride):
                        sub = p_off + T.dgrad_class_weight_index(cout, cin, k, stride, pad, a, b)
                        idx.append(sub)
                        views.append(("wd", (name, a, b), off, (cin, sub.size // cin)))
                        off += sub.size
        self.wc_idx = torch.from_numpy(np.concatenate(idx).astype(np.int32)).to(self.device)
        self.wc_flat, self.wc_lo = self._weights((off + 3) // 4 * 4)
        for kind, name, o, shape in views:
            getattr(self, kind)[name] = self.wc_flat[o:o + int(np.prod(shape))].view(shape)
        off = 0
        for name, cout, cin, k in kxk:
            n = cout * cin * k * k
            self.dwp[name] = self.dwp_flat[off:off + n].view(cout, k, k, cin)
            off += n
        # dropout state (filled per forward call)
        self.drop_mode = L.DROP_NONE
        self.drop_seed = 0
        self.masks = None
        self.seed_state = torch.zeros(1, dtype=torch.int64, device=self.device)   # per-step dropout seed (device word)
        self._graphs = {}                # (pass, tap set, dropout mode) -> torch.cuda.CUDAGraph

    # ------------------------------------------------------------------ plan
    def _conv_wgrad(self, name, x, dy, geom, dw, db, *, x_layout="nhwc", tap_copy=False):
        """tap_copy: x is a unit's channels-last tap (or, in the NCHW plan, the channels-last copy of a 7x7 tap), which is
        TMA-fed like the NCHW tap."""
        # dW is accumulated in the k order of the implicit GEMM (OHWI: consecutive accumulator rows = consecutive
        # addresses, so the split-K reductions coalesce) and un-permuted once at the end; writing OIHW directly
        # (dw_layout="oihw") was measured slower: the strided atomics cost more than the permute pass
        spc = T.conv_wgrad_spec(geom, x_layout, "nhwc")
        x3 = self.prec == L.PREC_TF32X3
        # the units' weight gradients are TMA-fed from the tap (measured 81 -> 54 us at level 3a)
        tma = TGemm.wgrad_eligible(geom, x_layout)
        bk = 0
        if tma and x_layout == "nhwc" and not tap_copy:
            # stage convs: TMA im2col with DEEP K-blocks (bk output pixels per stage: 64 / 128 instead of 32 -> fewer, larger
            # TMA boxes) where that was measured faster than the cp.async gather kernel (config 2,
            # profiles/wgrad_sweep_r02x.txt).  tf32 mode: only motion_conv_trans_28, where 128-pixel boxes win (197 us
            # gather, 389 / 204 / 169 us TMA at bk = 32 / 64 / 128; motion_conv_trans_14: 97 vs 136, motion_conv_trans:
            # 60 vs 77).  fp32 (3xTF32) mode, where the gather kernel's producers also write the residual tiles: every
            # layer, and the TMA-fed kernel wins on every KxK one (784 -> 501, 344 -> 296, 194 -> 177 us) at bk <= 64.
            max_bk = 64 if x3 else (128 if name == "motion_conv_trans_28" else 0)
            # deepest K-block <= max_bk whose pipeline stage (A: 4 stacks of {32 rows x bk pixels}, B: one per 32 columns
            # of the N tile; twice that with the 3xTF32 residual tiles) still leaves room for two stages per SM
            bn = 256 if spc.N > 256 else (spc.N + 15) // 16 * 16
            mul = 2 if x3 else 1
            fits = [b for b in (128, 64, 32) if b <= max_bk and mul * (b * 512 + math.ceil(bn / 32) * b * 128) <= 108 * 1024]
            tma, bk = bool(fits), (fits[0] if fits else 0)
        m_tiles, kb = math.ceil(spc.M / 128), math.ceil(spc.K / (bk or 32))
        n_tiles = max(1, math.ceil(spc.N / 256))
        # split-K factor: minimise rounds x (K-blocks per CTA + fixed cost), rounds = ceil(CTAs / resident CTA slots) -- two CTAs
        # per SM in the tf32 mode, one in the 3xTF32 mode.  The fixed cost (prologue, first TMA round trip, the epilogue that
        # adds the CTA's whole tile into dW) is worth ~10 K-blocks (profiles/timeline_*_r02z.txt); an under-filled round is
        # charged as idle SMs.
        split = _wgrad_split(m_tiles * n_tiles, kb, _SM_TARGET * (1 if x3 else 2), bk or 32)
        mk = (lambda *a, **k: TGemm(*a, geom=geom, x_layout=x_layout, wgrad=True, bk=bk, **k)) if tma else Gemm
        # dW[n][m]: consecutive accumulator rows are consecutive addresses -> transposed float4 adds (offk.h: out_vec = 2)
        rows_vec = dw.data_ptr() % 16 == 0 and geom.kdim % 4 == 0
        g = mk(self, spc, ("wgrad", x_layout, _gkey(geom)), a_src=x, b_src=dy, out=dw, ones_out=db,
               atomic=True, split_k=split, name=name + ".wgrad", out_vec=2 if rows_vec else None)
        self.flops_bwd += g.flops
        return g

    def _conv_dgrad(self, name, dy, w, dx, geom, *, gate=None, gate_col0=0, gate_first=False, addend=None,
                    add_geom=None, x_layout="nhwc"):
        out = []
        for i, spc in enumerate(T.conv_dgrad_specs(geom, x_layout, "nhwc", "nhwc")):
            add_tabs = None
            if addend is not None and add_geom is not None:
                # addend lives in a differently-shaped buffer: tables of the same logical (img, c, y, x) element
                aspec = T.conv_dgrad_specs(add_geom, "nhwc", "nhwc", "nhwc")[i]
                t = self._tables(("dgrad", "nhwc", _gkey(add_geom), i), aspec, _OUT_TABLES)
                add_tabs = (t["out_row"], t["out_col"])
            kw_ = dict(a_src=dy, b_src=w, out=dx, gate=gate, gate_col0=gate_col0, gate_first=gate_first, addend=addend,
                       add_tabs=add_tabs, name=f"{name}.dgrad{i}")
            key, ex = ("dgrad", x_layout, _gkey(geom), i), spc.extra
            if x_layout == "nchw":
                # the units' tap gradients: dX is NCHW, written through the out tables by the gather-fed kernel
                g = Gemm(self, spc, key, **kw_)
            elif geom.stride == 1:
                # dX of a stride-1 conv = a forward conv over dY with flipped taps and pad' = k-1-pad: TMA-fed
                gd = T.ConvGeom(geom.n_img, geom.cout, geom.hout, geom.wout, geom.cin, geom.kh, geom.kw, 1,
                                geom.kh - 1 - geom.pad, geom.y_ctot, geom.y_coff, geom.x_ctot, geom.x_coff)
                if not (name in self.wd and geom.kh == geom.kw and TGemm.eligible(gd)
                        and (gd.hout, gd.wout) == (geom.hin, geom.win)):
                    raise ValueError(f"{name}.dgrad{i}: this data gradient has no TMA-fed form")
                kw_["b_src"] = self.wd[name]
                g = TGemm(self, spc, key, geom=gd, **kw_)
            else:
                # one stride-parity class = a stride-1 correlation over dY with the class's R x Q taps (free geometry)
                if not ((name, ex["a"], ex["b"]) in self.wd and geom.cout % 32 == 0 and geom.y_ctot % 4 == 0
                        and geom.y_coff % 4 == 0 and ex["pad_h"] >= 0 and ex["pad_w"] >= 0):
                    raise ValueError(f"{name}.dgrad{i}: this data gradient has no TMA-fed form")
                R, Q = len(ex["rs"]), len(ex["qs"])
                fg = _FreeGeom(n_img=geom.n_img, cin=geom.cout, hin=geom.hout, win=geom.wout, cout=geom.cin, kh=R, kw=Q,
                               stride=1, pad=ex["pad_h"], pad_w=ex["pad_w"], x_ctot=geom.y_ctot, x_coff=geom.y_coff,
                               hout=ex["hc"], wout=ex["wc"], kdim=R * Q * geom.cout)
                kw_["b_src"] = self.wd[(name, ex["a"], ex["b"])]
                kw_["tile_n"] = _pick_tile_n(spc.M, spc.N, _SM_TARGET * (1 if self.prec == L.PREC_TF32X3 else 2))
                g = TGemm(self, spc, key, geom=fg, **kw_)
            self.flops_bwd += g.flops
            out.append(g)
        return out

    def _build(self):
        P, N, B, Lg = self.P, self.N, self.B, self.Lseg
        bf, pr, gr = self.buf, self.params, self.grads
        fwd, bwd_stage = [], []
        lib = self.lib

        # ============ OFF units (RGB_OFF.py:596-616 and the eight copies)
        self._stencils = {}
        fwd_lane = {"28": 0, "14": 1, "7": 2}
        self.stencil_fwd_steps = OrderedDict()        # stage -> batched stencil launch (bench.py times these)
        stage_levels = OrderedDict((st, [t for t in S.LEVELS if S.LEVEL_STAGE[t] == st]) for st in S.STAGES)
        n_lv = len(S.LEVELS)
        self._st_desc = (L.OffkStencil * n_lv)()      # one contiguous array: stage batches are slices of it
        self._st_io = (L.OffkStencilIO * n_lv)()
        k4_steps = []
        for li, (tag, (cin, s)) in enumerate(S.LEVELS.items()):
            st = S.LEVEL_STAGE[tag]
            fl = fwd_lane[st]
            ctot, _, members = S.STAGES[st]
            coff = dict(members)[tag]
            geom = T.ConvGeom(N, cin, s, s, S.UNIT_C)
            gd, dgd = bf["gd_" + tag], bf["dgd_" + tag]
            # K1: gen (ReLU) and down (linear) 1x1 convs as ONE GEMM with 160 output channels
            # 7x7 taps: a 196-byte channel stride is not a legal TMA stride -> one channels-last copy of the tap per
            # step feeds both the forward GEMM (dense tensor map) and the weight gradient (im2col_t), all TMA-fed.
            # Channels-last taps take that route in place, at every level.
            cl = self.tap_layout == "channels_last"
            via_copy = (s * s) % 4 != 0 and cin % 32 == 0 and not cl
            if via_copy:
                tapT = self._buf("tapT_" + tag, N, s, s, cin)

                def kt(stream, tag=tag, tapT=tapT, cin=cin, hw=s * s):
                    L.check(lib.offk_nchw_to_nhwc(_ptr(self.taps[tag]), _ptr(tapT), N, cin, hw, stream), "tapT_" + tag)
                fwd.append(_nm(kt, "tapT_" + tag, writes=[tapT], lane=fl))
            x_cl = self.taps[tag] if cl else (tapT if via_copy else None)
            if x_cl is not None:
                k1, = self._conv_fwd("unit_" + tag, x_cl, gd, geom, self._unit_w(self.params_flat, tag),
                                     self._unit_b(self.params_flat, tag), relu_cols=S.GEN_C, x_layout="nhwc", no_split=True)
                if cl:
                    self._tap_users[tag].append(getattr(k1, "gemm", k1))
            else:
                k1, = self._conv_fwd("unit_" + tag, self.taps[tag], gd, geom, self._unit_w(self.params_flat, tag),
                                     self._unit_b(self.params_flat, tag), relu_cols=S.GEN_C, x_layout="nchw")
                self._tap_users[tag].append(getattr(k1, "gemm", k1))
            fwd.append(_on(k1, fl))
            # K2 / K3 descriptors: fused spatial stencil + temporal difference + dropout + cat, into the stage buffer
            sd = self._st_desc[li]
            sd.B, sd.L, sd.Cg, sd.Cs, sd.K, sd.H, sd.W = B, Lg, S.GEN_C, S.DOWN_C, 1, s, s
            sd.g_fs = sd.d_fs = S.UNIT_C * s * s
            sd.g_ps = sd.d_ps = S.UNIT_C
            sd.out_ctot, sd.out_coff, sd.index_mode = ctot, coff, self.index_mode
            sd.drop_mode, sd.keep_scale, sd.drop_p = L.DROP_NONE, 1.0 / (1.0 - S.DROP_P), S.DROP_P
            self._stencils[tag] = sd
            if self.variant == "rgb":
                w3, b3 = pr[f"motion_spatial_grad_{tag}.weight"], pr[f"motion_spatial_grad_{tag}.bias"]
                dw3, db3 = gr[f"motion_spatial_grad_{tag}.weight"], gr[f"motion_spatial_grad_{tag}.bias"]
            else:
                w3, b3, dw3, db3 = self.sobel_w, None, None, None
            io = self._st_io[li]
            io.g, io.d = gd.data_ptr(), gd.data_ptr() + 4 * S.GEN_C            # D = channels [128,160) of every pixel
            io.w, io.bias = w3.data_ptr(), (b3.data_ptr() if b3 is not None else None)
            io.out, io.dout = bf["F" + st].data_ptr(), bf["dF" + st].data_ptr()
            io.dg, io.dd = dgd.data_ptr(), dgd.data_ptr() + 4 * S.GEN_C
            io.dg_fs = io.dd_fs = S.UNIT_C * s * s
            io.dw = dw3.data_ptr() if dw3 is not None else None
            io.dbias = db3.data_ptr() if db3 is not None else None
            # K4: weight / bias gradient of the fused 1x1 (no dX for the frozen taps unless asked, train_off.py:39-46)
            if x_cl is not None:
                k4 = self._conv_wgrad("unit_" + tag, x_cl, dgd, geom, self._unit_w(self.grads_flat, tag),
                                      self._unit_b(self.grads_flat, tag), x_layout="nhwc", tap_copy=True)
                if cl:
                    self._tap_users[tag].append(k4)
            else:
                k4 = self._conv_wgrad("unit_" + tag, self.taps[tag], dgd, geom,
                                      self._unit_w(self.grads_flat, tag), self._unit_b(self.grads_flat, tag), x_layout="nchw")
                self._tap_users[tag].append(k4)
            k4.unit_tag = tag                       # data parallelism: this unit's gradients are final once k4 is done
            grp = [_on(k4, li % 3)]
            if self.tap_grads:
                grp += [_on(g, li % 3) for g in self._conv_dgrad("unit_" + tag, dgd, self._unit_w(self.params_flat, tag),
                                                                  self.tap_grad[tag], geom, x_layout="nchw")]
            k4_steps += grp
        # K2: the forward stencil in two batched launches: the 28-stage units on their own (they open the critical path);
        # the 14- and 7-stage units together (the 7x7 levels are 7 MB each: on their own they run at a fifth of the
        # bandwidth)
        tags = list(S.LEVELS)
        self.stencil_fwd_tags = OrderedDict()         # launch name -> level tags (bench.py: algorithmic bytes)
        for gname, sts in (("28", ["28"]), ("14+7", ["14", "7"])):
            lv_tags = [t for st in sts for t in stage_levels[st]]
            i0, n = tags.index(lv_tags[0]), len(lv_tags)
            assert tags[i0:i0 + n] == lv_tags

            def k2(stream, i0=i0, n=n, gname=gname):
                L.check(lib.offk_stencil_diff_fwd_batch(n, C.byref(self._st_desc[i0]), C.byref(self._st_io[i0]), stream),
                        "stencil_fwd_" + gname)
            step = _nm(k2, "stencil_fwd_" + gname, reads=[bf["gd_" + t] for t in lv_tags], writes=[bf["F" + st] for st in sts],
                       lane=fwd_lane[sts[0]])
            fwd.append(step)
            self.stencil_fwd_steps[gname] = step
            self.stencil_fwd_tags[gname] = lv_tags
        # K3: the backward of all nine units in ONE launch (every stage gradient dF* is complete by then), then their weight
        # gradients.  Running the 7- and 14-stage units' backward early on side lanes, under the rest of the stage chain, was
        # measured slower at config 2 (2.90 vs 2.84 ms/step): the HBM-bound unit kernels slow the chain more than the
        # overlap saves.
        grad3 = [gr[f"motion_spatial_grad_{t}.{k}"] for t in tags for k in ("weight", "bias")] if self.variant == "rgb" else []

        def k3(stream):
            L.check(lib.offk_stencil_diff_bwd_batch(n_lv, self._st_desc, self._st_io, stream), "stencil_bwd")
        k3 = _nm(k3, "stencil_bwd", reads=[bf["dF" + st] for st in S.STAGES] + [bf["gd_" + t] for t in tags],
                 writes=[bf["dgd_" + t] for t in tags] + grad3, lane=0)
        bwd_units = [k3] + k4_steps

        # ============ stage convs
        def geom_of(name, n_img, s_in, x_ctot=0, x_coff=0, y_ctot=0, y_coff=0):
            _, cout, cin, k, stride, pad = S.CONV_BY_NAME[name]
            return T.ConvGeom(n_img, cin, s_in, s_in, cout, k, k, stride, pad, x_ctot, x_coff, y_ctot, y_coff)

        def W(n): return self.wp[n] if n in self.wp else pr[n + ".weight"]     # OHWI copy for KxK convs
        def Bv(n): return pr[n + ".bias"]
        def dW(n): return self.dwp[n] if n in self.dwp else gr[n + ".weight"]
        def dB(n): return gr[n + ".bias"]

        def layer(name, x, y, s_in, *, relu=False, addend=None, relu_post=False,
                  x_ctot=0, x_coff=0, y_ctot=0, y_coff=0, lane=0, aux=None):
            """forward conv; returns geom for the gradient wiring."""
            geom = geom_of(name, P, s_in, x_ctot, x_coff, y_ctot, y_coff)
            fwd.extend(_on(st, lane) for st in self._conv_fwd(name, x, y, geom, W(name), Bv(name), relu=relu, addend=addend,
                                                              relu_post=relu_post, aux=aux))
            return geom

        # ---- resolution 28 (RGB_OFF.py:655-685)
        # pre-ReLU output kept for the branch (:665); its ReLU'd copy (:658) is the second output
        g_t28 = layer("motion_conv_trans_28", bf["F28"], bf["t28"], 28, aux=(bf["t28r"], 64, 0, None, "relu_t28"))
        g_c1a = layer("motion_conv1_trans_28a", bf["t28r"], bf["h1_28a"], 14, relu=True)
        g_c2a = layer("motion_conv2_trans_28a", bf["h1_28a"], bf["h2_28a"], 14, relu=True)
        g_bra = layer("motion_conv_branch_28a", bf["t28"], bf["br28"], 14, lane=2)
        g_c3a = layer("motion_conv3_trans_28a", bf["h2_28a"], bf["s28a"], 14, addend=bf["br28"], relu_post=True)
        g_c1b = layer("motion_conv1_trans_28b", bf["s28a"], bf["h1_28b"], 14, relu=True)
        g_c2b = layer("motion_conv2_trans_28b", bf["h1_28b"], bf["h2_28b"], 14, relu=True)
        g_c3b = layer("motion_conv3_trans_28b", bf["h2_28b"], bf["s28b"], 14, addend=bf["s28a"], relu_post=True)
        g_c1c = layer("motion_conv1_trans_28c", bf["s28b"], bf["h1_28c"], 14, relu=True)
        g_c2c = layer("motion_conv2_trans_28c", bf["h1_28c"], bf["h2_28c"], 14, relu=True)
        # sum_28c goes straight into the 14-stage fusion buffer at channel 800 (cat, :760)
        g_c3c = geom_of("motion_conv3_trans_28c", P, 14, y_ctot=1056, y_coff=800)
        g_s28b_as_f14 = T.ConvGeom(P, 256, 14, 14, 256, y_ctot=256)  # tables for the s28b addend (plain [P,14,14,256])
        spc_add = T.conv_fwd_spec(g_s28b_as_f14, "nhwc", "nhwc")
        tabs_add = self._tables(("fwd", "nhwc", _gkey(g_s28b_as_f14)), spc_add, _OUT_TABLES)
        fwd.extend(self._conv_fwd("motion_conv3_trans_28c", bf["h2_28c"], bf["F14"], g_c3c,
                                  W("motion_conv3_trans_28c"), Bv("motion_conv3_trans_28c"), addend=bf["s28b"],
                                  add_tabs=(tabs_add["out_row"], tabs_add["out_col"]), relu_post=True))

        # ---- resolution 14 (RGB_OFF.py:759-780)
        g_t14 = layer("motion_conv_trans_14", bf["F14"], bf["t14"], 14, relu=True)
        g_14a1 = layer("motion_conv1_trans_14a", bf["t14"], bf["h1_14a"], 7, relu=True)
        g_14a2 = layer("motion_conv2_trans_14a", bf["h1_14a"], bf["h2_14a"], 7, relu=True)
        g_14ex = layer("motion_conv_expand_trans_14a", bf["t14"], bf["ex14"], 7, lane=2)
        g_14a3 = layer("motion_conv3_trans_14a", bf["h2_14a"], bf["s14a"], 7, addend=bf["ex14"], relu_post=True)
        g_14b1 = layer("motion_conv1_trans_14b", bf["s14a"], bf["h1_14b"], 7, relu=True)
        g_14b2 = layer("motion_conv2_trans_14b", bf["h1_14b"], bf["h2_14b"], 7, relu=True)
        # 3x3 + ReLU (:316,:778), kept for the backward gate; sum_14b = relu(s14a + h3_14b) -> 7-stage fusion buffer channels
        # [320,832) (:779-780, cat :832) is the second output
        g_14b3 = layer("motion_conv3_trans_14b", bf["h2_14b"], bf["h3_14b"], 7, relu=True,
                       aux=(bf["F7"], 832, 320, bf["s14a"], "sum_14b"))

        # ---- heads 28 / 14 (RGB_OFF.py:783-793)
        fwd.append(_nm(lambda stream: L.check(lib.offk_pool3_nhwc(_ptr(bf["F14"]), P, 14, 14, 1056, 800, 256, 2, 0, L.POOL_MAX,
                                                                   _ptr(bf["p28"]), 256, 0, stream), "maxpool28"), "maxpool28",
                       reads=[bf["F14"]], writes=[bf["p28"]], lane=1))
        # each head = ONE launch: avgpool 7x7 -> dropout -> Linear (-> segment consensus)   (SURVEY K6)
        fwd.append(_on(self._head_fwd("28", bf["p28"], 256, 256, 0, "fc_action_motion_28"), 1))
        fwd.append(_on(self._head_fwd("14", bf["F7"], 512, 832, 320, "fc_action_motion_14"), 1))

        # ---- resolution 7 (RGB_OFF.py:831-847)
        g_t7 = layer("motion_conv_trans", bf["F7"], bf["t7"], 7, relu=True)
        g_71 = layer("motion_conv1_trans", bf["t7"], bf["h1_7"], 7, relu=True)
        g_72 = layer("motion_conv2_trans", bf["h1_7"], bf["h2_7"], 7, relu=True)
        g_7br = layer("motion_conv_branch_trans", bf["t7"], bf["br7"], 7, lane=2)
        g_73 = layer("motion_conv3_trans", bf["h2_7"], bf["s7"], 7, addend=bf["br7"])        # no final ReLU (:841)
        fwd.append(self._head_fwd("7", bf["s7"], 1024, 1024, 0, "fc_action_motion"))

        # ============ backward of the stages (reverse order); every d_* buffer holds dL/d(pre-activation)
        bs = bwd_stage
        d = lambda n: bf["d_" + n]
        # upstream gradients: [B,101] with the consensus (its backward, g.expand / T, is folded into the head kernels),
        # [P,101] without
        n_up = B if self.consensus else P
        self.d_out7 = torch.zeros(n_up, S.NUM_CLASSES, device=self.device)
        self.d_out14 = torch.zeros(n_up, S.NUM_CLASSES, device=self.device)
        # heads (fc28 receives no gradient: never returned, RGB_OFF.py:860): Linear weight / bias gradient, and
        # ds7 = avgpool'(dropout'(Linear'(d_out7))) in one pass
        bs.extend(self._head_bwd("7", self.d_out7, d("s7"), 1024, 1024, 0, "fc_action_motion", act=None, accumulate=False))

        def back(name, x, dy, geom):
            bs.append(_on(self._conv_wgrad(name, x, dy, geom, dW(name), dB(name)), 1))   # wgrad lane

        def dgrad(name, dy, dx, geom, lane=0, **kw):
            bs.extend(_on(g, lane) for g in self._conv_dgrad(name, dy, W(name), dx, geom, **kw))

        # ---- 7
        back("motion_conv3_trans", bf["h2_7"], d("s7"), g_73)
        dgrad("motion_conv3_trans", d("s7"), d("h2_7"), g_73, gate=bf["h2_7"])
        back("motion_conv_branch_trans", bf["t7"], d("s7"), g_7br)
        dgrad("motion_conv_branch_trans", d("s7"), d("tmp7"), g_7br, lane=2)
        back("motion_conv2_trans", bf["h1_7"], d("h2_7"), g_72)
        dgrad("motion_conv2_trans", d("h2_7"), d("h1_7"), g_72, gate=bf["h1_7"])
        back("motion_conv1_trans", bf["t7"], d("h1_7"), g_71)
        dgrad("motion_conv1_trans", d("h1_7"), d("t7"), g_71, gate=bf["t7"], addend=d("tmp7"))
        back("motion_conv_trans", bf["F7"], d("t7"), g_t7)
        dgrad("motion_conv_trans", d("t7"), bf["dF7"], g_t7)
        # d sum_14b = (dF7[:,320:] + head-14 pool gradient) * [sum_14b > 0]   (in place in the dF7 slice)
        bs.extend(self._head_bwd("14", self.d_out14, bf["dF7"], 512, 832, 320, "fc_action_motion_14", act=bf["F7"], accumulate=True))
        # ---- 14b:  sum_14b = relu(s14a + relu(conv3_14b(h2b)))
        bs.append(_nm(lambda stream: L.check(lib.offk_gate_copy(_ptr(bf["dF7"]), 832, 320, _ptr(bf["h3_14b"]), 512, 0,
                                                                _ptr(d("h3_14b")), 512, 0, P, 512, 49, stream), "gate_h3b"),
                      "gate_h3b", reads=[bf["dF7"], bf["h3_14b"]], writes=[d("h3_14b")]))
        back("motion_conv3_trans_14b", bf["h2_14b"], d("h3_14b"), g_14b3)
        dgrad("motion_conv3_trans_14b", d("h3_14b"), d("h2_14b"), g_14b3, gate=bf["h2_14b"])
        back("motion_conv2_trans_14b", bf["h1_14b"], d("h2_14b"), g_14b2)
        dgrad("motion_conv2_trans_14b", d("h2_14b"), d("h1_14b"), g_14b2, gate=bf["h1_14b"])
        back("motion_conv1_trans_14b", bf["s14a"], d("h1_14b"), g_14b1)
        g_slice7 = T.ConvGeom(P, 512, 7, 7, 128, x_ctot=832, x_coff=320)   # addresses dF7[:,320:832] like a conv input
        dgrad("motion_conv1_trans_14b", d("h1_14b"), d("s14a"), g_14b1, gate=bf["s14a"], addend=bf["dF7"],
              add_geom=g_slice7)
        # ---- 14a
        back("motion_conv3_trans_14a", bf["h2_14a"], d("s14a"), g_14a3)
        dgrad("motion_conv3_trans_14a", d("s14a"), d("h2_14a"), g_14a3, gate=bf["h2_14a"])
        back("motion_conv_expand_trans_14a", bf["t14"], d("s14a"), g_14ex)
        dgrad("motion_conv_expand_trans_14a", d("s14a"), d("tmp14"), g_14ex, lane=2)
        back("motion_conv2_trans_14a", bf["h1_14a"], d("h2_14a"), g_14a2)
        dgrad("motion_conv2_trans_14a", d("h2_14a"), d("h1_14a"), g_14a2, gate=bf["h1_14a"])
        back("motion_conv1_trans_14a", bf["t14"], d("h1_14a"), g_14a1)
        dgrad("motion_conv1_trans_14a", d("h1_14a"), d("t14"), g_14a1, gate=bf["t14"], addend=d("tmp14"))
        back("motion_conv_trans_14", bf["F14"], d("t14"), g_t14)
        # dF14; channels >= 800 are sum_28c = relu(.) -> gate them here (fc28 contributes nothing)
        dgrad("motion_conv_trans_14", d("t14"), bf["dF14"], g_t14, gate=bf["F14"], gate_col0=800)
        # ---- 28c / 28b (identity residuals): the incoming gradient of 28c is the dF14 slice [800,1056)
        g_dy_c3c = g_c3c
        back("motion_conv3_trans_28c", bf["h2_28c"], bf["dF14"], g_dy_c3c)
        dgrad("motion_conv3_trans_28c", bf["dF14"], d("h2_28c"), g_dy_c3c, gate=bf["h2_28c"])
        back("motion_conv2_trans_28c", bf["h1_28c"], d("h2_28c"), g_c2c)
        dgrad("motion_conv2_trans_28c", d("h2_28c"), d("h1_28c"), g_c2c, gate=bf["h1_28c"])
        back("motion_conv1_trans_28c", bf["s28b"], d("h1_28c"), g_c1c)
        g_slice14 = T.ConvGeom(P, 256, 14, 14, 64, x_ctot=1056, x_coff=800)
        dgrad("motion_conv1_trans_28c", d("h1_28c"), d("s28b"), g_c1c, gate=bf["s28b"], addend=bf["dF14"],
              add_geom=g_slice14)
        back("motion_conv3_trans_28b", bf["h2_28b"], d("s28b"), g_c3b)
        dgrad("motion_conv3_trans_28b", d("s28b"), d("h2_28b"), g_c3b, gate=bf["h2_28b"])
        back("motion_conv2_trans_28b", bf["h1_28b"], d("h2_28b"), g_c2b)
        dgrad("motion_conv2_trans_28b", d("h2_28b"), d("h1_28b"), g_c2b, gate=bf["h1_28b"])
        back("motion_conv1_trans_28b", bf["s28a"], d("h1_28b"), g_c1b)
        dgrad("motion_conv1_trans_28b", d("h1_28b"), d("s28a"), g_c1b, gate=bf["s28a"], addend=d("s28b"))
        # ---- 28a: the branch consumes the PRE-ReLU conv_trans_28 output (:665), conv1 the ReLU'd one (:659)
        back("motion_conv3_trans_28a", bf["h2_28a"], d("s28a"), g_c3a)
        dgrad("motion_conv3_trans_28a", d("s28a"), d("h2_28a"), g_c3a, gate=bf["h2_28a"])
        back("motion_conv_branch_28a", bf["t28"], d("s28a"), g_bra)
        dgrad("motion_conv_branch_28a", d("s28a"), d("tmp28"), g_bra, lane=2)
        back("motion_conv2_trans_28a", bf["h1_28a"], d("h2_28a"), g_c2a)
        dgrad("motion_conv2_trans_28a", d("h2_28a"), d("h1_28a"), g_c2a, gate=bf["h1_28a"])
        back("motion_conv1_trans_28a", bf["t28r"], d("h1_28a"), g_c1a)
        dgrad("motion_conv1_trans_28a", d("h1_28a"), d("t28"), g_c1a, gate=bf["t28"], gate_first=True,
              addend=d("tmp28"))
        back("motion_conv_trans_28", bf["F28"], d("t28"), g_t28)
        dgrad("motion_conv_trans_28", d("t28"), bf["dF28"], g_t28)

        # weight re-layouts before the forward (one launch), OHWI -> OIHW weight gradients after the backward
        wc, wci, pflat = self.wc_flat, self.wc_idx, self.params_flat
        pre = [_nm(lambda stream: L.check(lib.offk_gather_copy(_ptr(pflat), _ptr(wci), _ptr(wc), wc.numel(), stream),
                                          "weight copies"), "weight_copies", writes=[wc], lane=2)]
        if self.presplit:
            # 3xTF32 residuals of every weight, once per step (the GEMMs then get both weight tiles by TMA)
            plo, wlo = self.params_lo, self.wc_lo
            pre.append(_nm(lambda stream: L.check(lib.offk_tf32_residual(_ptr(pflat), _ptr(plo), pflat.numel(), stream),
                                                  "weight residuals"), "weight_residuals_params", writes=[plo], lane=0))
            pre.append(_nm(lambda stream: L.check(lib.offk_tf32_residual(_ptr(wc), _ptr(wlo), wc.numel(), stream),
                                                  "weight residuals"), "weight_residuals_copies", reads=[wc], writes=[wlo],
                           lane=2))
        # OHWI -> OIHW accumulation of every KxK weight gradient: one launch
        kxk = [(name, cout, cin, k) for name, cout, cin, k, _, _ in S.STAGE_CONVS if k > 1]
        self._unperm = (L.OffkPermute * len(kxk))()
        for i, (name, cout, cin, k) in enumerate(kxk):
            it = self._unperm[i]
            it.src, it.dst = self.dwp[name].data_ptr(), gr[name + ".weight"].data_ptr()
            it.cout, it.cin, it.kh, it.kw = cout, cin, k, k
        post = [_nm(lambda stream: L.check(lib.offk_permute_weight_batch(len(kxk), self._unperm, 2, stream), "unpermute"),
                    "unpermute_kxk_weight_grads", reads=[self.dwp_flat], writes=[gr[n + ".weight"] for n, _, _, _ in kxk], lane=1)]
        self.fwd_steps = pre + fwd
        # gradient accumulators start from zero (split-K / atomic accumulation); grads_flat only when asked
        self._zero_grads = True
        gflat, dwflat = self.grads_flat, self.dwp_flat
        zero = [_nm(lambda stream: self._zero_grads and L.check(lib.offk_fill_zero(_ptr(gflat), gflat.numel(), stream),
                                                                 "zero grads"), "zero grads_flat", writes=[gflat]),
                _nm(lambda stream: L.check(lib.offk_fill_zero(_ptr(dwflat), dwflat.numel(), stream), "zero dwp"),
                    "zero dwp_flat", writes=[dwflat], lane=1)]
        # the stage / head gradients are complete before the units run: their bucket can be all-reduced meanwhile
        self.bwd_stage_steps = zero + bwd_stage + post
        self.bwd_unit_steps = bwd_units
        self.bwd_steps = self.bwd_stage_steps + self.bwd_unit_steps
        self.steps = self.fwd_steps + self.bwd_steps
        self.launches_fwd = len(_kernels(self.fwd_steps))
        self.launches_bwd = len(_kernels(self.bwd_steps))
        # parameters and taps are read-only inside a pass: never a hazard
        ro = [self.params_flat] + [t for ts in self.tap_sets for t in ts.values()]
        if self.variant == "flow":
            ro.append(self.sobel_w)
        self.fwd_sched = Schedule(self.fwd_steps, ignore=ro)
        self.bwd_sched = Schedule(self.bwd_steps, ignore=ro)
        self._lanes = max(self.fwd_sched.n_lanes, self.bwd_sched.n_lanes)
        self._side = None
        unit_end = max(self.layout[f"motion_{k}_{t}.bias"][0] + (S.GEN_C if k == "conv_gen" else S.DOWN_C)
                       for t in S.LEVELS for k in (("conv_gen", "spatial_down") + (("spatial_grad",) if self.variant == "rgb" else ())))
        self.unit_range = (0, (unit_end + 3) // 4 * 4)          # flat offsets of the nine units' parameters
        # per unit: [first parameter of the level, first parameter of the next level) -- contiguous, 16-byte aligned
        starts = [self.layout[f"motion_conv_gen_{t}.weight"][0] for t in S.LEVELS] + [self.unit_range[1]]
        self.unit_ranges = OrderedDict((t, (starts[i], starts[i + 1])) for i, t in enumerate(S.LEVELS))
        self.stage_range = (self.unit_range[1], self.n_flat)    # stage convs + FC heads

    # ------------------------------------------------------------------ small step factories
    @staticmethod
    def _site_salt(site):
        """Constant 64-bit salt of dropout call site ``site`` (12 per forward, RGB_OFF.py:612..:845): splitmix64(site).
        The kernels add the step seed, which lives in device memory (``seed_state``; offk.h: seed_dev), and hash the sum
        with the element index, so every bit of both reaches every keep decision -- and a captured CUDA graph, whose
        kernel arguments are frozen, still draws new masks whenever the device word changes."""
        m = 0xFFFFFFFFFFFFFFFF
        z = ((site + 1) * 0xD1B54A32D192ED03) & m
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
        return z ^ (z >> 31)

    def _seed_dev(self):
        return _ptr(self.seed_state) if self.drop_mode == L.DROP_SEED else None

    def _head_fwd(self, k, x, c, ctot, coff, fcname):
        """global_pool -> dropout -> fc_action_motion* (-> consensus) as ONE launch (RGB_OFF.py:784-787,790-793,844-847;
        Flow_OFF.py:867-876).  Linear ops only: exact fp32 in every precision mode."""
        lib, P, bf = self.lib, self.P, self.buf
        site = {"28": 9, "14": 10, "7": 11}[k]
        w, b = self.params[fcname + ".weight"], self.params[fcname + ".bias"]
        T_ = self.Lseg - 1 if self.consensus else 1
        cons = bf["cfc" + k] if self.consensus else None

        def run(stream):
            m = self.masks["fc" + k] if self.drop_mode == L.DROP_MASK else None
            L.check(lib.offk_head_fwd(_ptr(x), P, c, 49, ctot, coff, self.drop_mode, _ptr(m), self._site_salt(site),
                                      self._seed_dev(), S.DROP_P, 1.0 / (1.0 - S.DROP_P), _ptr(w), _ptr(b), S.NUM_CLASSES, T_,
                                      _ptr(bf["pool" + k]), _ptr(bf["fc" + k]), _ptr(cons), stream), "head_fwd" + k)
        self.flops_fwd += 2.0 * P * c * S.NUM_CLASSES
        return _nm(run, "head_fwd" + k, reads=[x], writes=[bf["pool" + k], bf["fc" + k], cons])

    def _head_bwd(self, k, dout, dx, c, ctot, coff, fcname, act, accumulate):
        """Backward of _head_fwd in two launches: Linear weight / bias gradient; Linear data gradient + dropout' + average
        pool backward (+ the producer's ReLU', + accumulation into a slice that already holds a gradient)."""
        lib, P, bf = self.lib, self.P, self.buf
        site = {"28": 9, "14": 10, "7": 11}[k]
        w = self.params[fcname + ".weight"]
        dw, db = self.grads[fcname + ".weight"], self.grads[fcname + ".bias"]
        T_ = self.Lseg - 1 if self.consensus else 1

        def call(stream, dx_, dw_, db_):
            m = self.masks["fc" + k] if self.drop_mode == L.DROP_MASK else None
            L.check(lib.offk_head_bwd(_ptr(dout), P, c, 49, ctot, coff, self.drop_mode, _ptr(m), self._site_salt(site),
                                      self._seed_dev(), S.DROP_P, 1.0 / (1.0 - S.DROP_P), _ptr(w), S.NUM_CLASSES, T_,
                                      _ptr(bf["pool" + k]), _ptr(act), int(accumulate), _ptr(dx_), _ptr(dw_), _ptr(db_), stream),
                    "head_bwd" + k)
        self.flops_bwd += 4.0 * P * c * S.NUM_CLASSES
        # the data gradient opens the dgrad chain (lane 0); the weight gradient runs beside it on the weight-gradient lane
        dgrad = _nm(lambda stream: call(stream, dx, None, None), "head_bwd%s.dgrad" % k,
                    reads=[dout, act, dx if accumulate else None], writes=[dx], lane=0)
        wgrad = _nm(lambda stream: call(stream, None, dw, db), "head_bwd%s.wgrad" % k, reads=[dout, bf["pool" + k]],
                    writes=[dw, db], lane=1)
        return [dgrad, wgrad]

    # ------------------------------------------------------------------ run
    def _set_dropout(self, train, masks, seed):
        if not train:
            self.drop_mode, self.masks = L.DROP_NONE, None
        elif masks is not None:
            self.drop_mode = L.DROP_MASK
            self.masks = {k: v.to(self.device, torch.uint8).contiguous() for k, v in masks.items()}
        else:
            self.drop_mode, self.masks = L.DROP_SEED, None
            self.drop_seed = int(seed)
        for i, (tag, sd) in enumerate(self._stencils.items()):
            sd.drop_mode = self.drop_mode
            sd.seed = self._site_salt(i)
            sd.seed_dev = self.seed_state.data_ptr() if self.drop_mode == L.DROP_SEED else None
            sd.keep_mask = self.masks[tag].data_ptr() if self.drop_mode == L.DROP_MASK else None

    def set_taps(self, taps: dict):
        for tag, t in self.taps.items():
            t.copy_(taps[tag], non_blocking=True)

    def select_taps(self, idx: int):
        """Make input set ``idx`` the one forward() and backward() read (re-binds the A operand of the unit GEMMs)."""
        self._tap_set = idx
        self.taps = self.tap_sets[idx]
        for tag, users in self._tap_users.items():
            ptr = self.taps[tag].data_ptr()
            for g in users:
                g.set_a_src(ptr)

    def stage_taps(self, taps: dict):
        """Asynchronously copy ``taps`` (host -- ideally pinned -- or device tensors) into the IDLE input set on a
        side stream, so the transfer overlaps the forward/backward still running on the other set.  Returns
        (set index, event); pass the index to select_taps() after making the compute stream wait on the event."""
        idx = 1 - self._tap_set
        main = torch.cuda.current_stream(self.device)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        # everything enqueued so far (incl. the last backward that read set idx) must finish before it is overwritten
        self._copy_stream.wait_stream(main)
        with torch.cuda.stream(self._copy_stream):
            for tag, t in self.tap_sets[idx].items():
                t.copy_(taps[tag], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        return idx, ev

    def forward(self, taps: dict = None, train: bool = False, masks: dict = None, seed: int = 0, graph: bool = False):
        """Run the forward plan.  Returns (fc7, fc28, fc14): [P,101] each, or [B,101] with consensus.
        graph=True replays the plan as ONE captured CUDA graph (captured on first use per input set and dropout mode):
        the same kernels, bit for bit, without the ~60 host-side launches."""
        if taps is not None:
            self.set_taps(taps)
        self._set_dropout(train, masks, seed)
        self.generation += 1            # backward() consumes the activations of THIS forward (one set of static buffers)
        if self.drop_mode == L.DROP_SEED:
            main = torch.cuda.current_stream(self.device)
            L.check(self.lib.offk_seed_set(_ptr(self.seed_state), self.drop_seed & 0xFFFFFFFFFFFFFFFF,
                                           C.c_void_p(main.cuda_stream)), "seed_set")
        if graph:
            self._replay("fwd")
        else:
            self._issue("fwd")
        pre = "cfc" if self.consensus else "fc"
        return self.buf[pre + "7"], self.buf[pre + "28"], self.buf[pre + "14"]

    # ------------------------------------------------------------------ CUDA graphs (SURVEY 8f-1)
    def _issue(self, which):
        streams = self._fork()
        (self.fwd_sched if which == "fwd" else self.bwd_sched).run(streams)
        self._join(streams)

    def _replay(self, which):
        if self.drop_mode == L.DROP_MASK:
            raise RuntimeError("graph replay supports eval mode and seeded dropout; injected masks are an eager-only test facility")
        key = (which, self._tap_set, self.drop_mode)
        g = self._graphs.get(key)
        if g is None:
            g = self._graphs[key] = self._capture(lambda: self._issue(which))
        g.replay()

    def backward(self, g7: torch.Tensor, g14: torch.Tensor, zero_grads: bool = True, after_stage=None, after_unit=None,
                 graph: bool = False):
        """Run the backward plan for dL/dfc7 and dL/dfc14; fills grads_flat (views in self.grads).
        ``after_stage()`` is called once the stage/head gradients (flat range ``stage_range``) are final and
        before the unit gradients are computed (used to overlap their all-reduce); ``after_unit(tag, stream)`` right
        after the last kernel that writes unit ``tag``'s gradients (flat range ``unit_ranges[tag]``) was issued on
        ``stream``."""
        self.d_out7.copy_(g7.reshape(self.d_out7.shape))
        self.d_out14.copy_(g14.reshape(self.d_out14.shape))
        if graph:
            if not zero_grads or after_stage is not None or after_unit is not None:
                raise RuntimeError("graph replay of the backward pass zeroes the gradient buffers and takes no hooks")
            self._zero_grads = True
            self._replay("bwd")
            return self.grads
        self._zero_grads = bool(zero_grads)
        streams = self._fork()
        n_stage = len(self.bwd_stage_steps)
        self.bwd_sched.run(streams, 0, n_stage)
        if after_stage is not None:
            self._join(streams)                      # the caller's stream now trails every stage-gradient kernel
            after_stage()
        on_step = None
        if after_unit is not None:
            def on_step(step, stream):
                tag = getattr(step, "unit_tag", None)
                if tag is not None:
                    after_unit(tag, stream)
        self.bwd_sched.run(streams, n_stage, on_step=on_step)
        self._join(streams)
        return self.grads

    def _fork(self):
        """[caller's stream, side streams...]; the side lanes start behind everything already enqueued by the caller."""
        main = torch.cuda.current_stream(self.device)
        if self.single_stream or self._lanes == 1:
            return [main] * self._lanes
        if self._side is None:
            self._side = [torch.cuda.Stream(device=self.device) for _ in range(self._lanes - 1)]
        for s_ in self._side:
            s_.wait_stream(main)
        return [main] + self._side

    def _join(self, streams):
        for s_ in streams[1:]:
            if s_ is not streams[0]:
                streams[0].wait_stream(s_)
