"""What the static launch plans (the OFF engine, engine.py; the BN-Inception extractor, extractor.py) are built from:
``LaunchPlan``, bound GEMM launches (gather-fed ``Gemm``, TMA-fed ``TGemm``), the tile / split-K policies and the
multi-stream ``Schedule`` of plan steps (callables taking a stream handle, annotated by ``_nm``)."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L
from . import tables as T

_SM_TARGET = 148
_PICK_A = 128           # _pick_tile_n: per-CTA cost ~ _PICK_A + bn (A rows + B rows of a K-block)
_WGRAD_FIXED_KB = 10    # _wgrad_split: fixed cost of a weight-gradient CTA, in K-blocks of 32 pixels
_TF32_WANT_CTAS = _SM_TARGET    # _auto_tile_n: CTAs a TMA-fed GEMM without split-K aims for in the tf32 mode
_X3_WANT_CTAS = 40      # ... and in the 3xTF32 mode
_FINISH_MIN_TILES = 100     # output tiles from which a split-K conv finishes in-kernel (_conv_fwd)

_OUT_TABLES = ("out_row", "out_col")
_ALL_TABLES = ("a_row", "a_col", "b_row", "b_col") + _OUT_TABLES


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class _FreeGeom:
    """im2col geometry with a caller-given output grid and separate top / left padding (OFFK_TGEMM_FREE_GEOM)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def _pick_tile_n(M: int, N: int, slots: int = 2 * _SM_TARGET) -> int:
    """N tile (multiple of 16, <= 256; the last tile may be partial) of a GEMM without split-K: the one that minimises
    rounds x per-CTA cost, rounds = ceil(CTAs / resident CTA slots) and cost ~ 128 + bn (rows of A and B a K-block moves
    through shared memory).  Wave quantisation matters: 37 x 11 tiles of 96 columns are 1.4 rounds, 37 x 8 of 144 are one."""
    mt = math.ceil(M / 128)
    best, best_cost = 0, None
    for bn in range(256, 15, -16):
        if bn > (N + 15) // 16 * 16:
            continue
        nt = math.ceil(N / bn)
        cost = math.ceil(mt * nt / slots) * (_PICK_A + bn) * (1.0 if mt * nt >= _SM_TARGET else _SM_TARGET / (mt * nt)) ** 0.5
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = bn, cost
    return best


def _wgrad_split(tiles: int, kb: int, slots: int, bk: int = 32) -> int:
    """Split-K factor of a weight-gradient GEMM with `tiles` output tiles and `kb` K-blocks of `bk` pixels: the one that
    minimises rounds x (K-blocks per CTA + fixed cost), rounds = ceil(CTAs / resident CTA slots); an under-filled round is
    charged as idle SMs.  The fixed cost (prologue, first TMA round trip, adding the tile into dW) is worth ~10 K-blocks of
    32 pixels (profiles/timeline_*_r02z.txt); the result is insensitive to it between 5 and 20 (profiles/env_r03j.log)."""
    fixed = _WGRAD_FIXED_KB * 32 / bk
    cost = lambda s_: math.ceil(tiles * s_ / slots) * (math.ceil(kb / s_) + fixed) * max(1.0, _SM_TARGET / (tiles * s_))
    return min(range(1, max(1, kb // 4) + 1), key=lambda s_: (cost(s_), s_))


def _auto_tile_n(M: int, N: int, tma: bool = False, x3: bool = False) -> int:
    """N tile of a GEMM launched without split-K; 0 = the kernel's default (widest legal tile).
    TMA-fed: two CTAs fit an SM and one CTA's epilogue should overlap another's main loop, so aim for >= 2 x 148 CTAs
    with the widest tile that gets there (re-reading A per N tile is one cheap TMA instruction).
    Gather-fed: the A gather is the expensive part and is repeated per N tile, so only narrow the tile when the grid
    would otherwise leave most SMs idle (the 7x7-resolution layers: 37 M tiles)."""
    mt = math.ceil(M / 128)
    bn0 = (N + 15) // 16 * 16 if N <= 256 else 256
    want, enough = (120, 140)
    if tma:         # (2 x 148 before the MMA issue path was fixed: narrow tiles were issue-bound then; profiles/env_r03t.log)
        want = enough = _TF32_WANT_CTAS
    if tma and x3:
        # 3xTF32: one CTA per SM, and every extra N tile repeats the A tile AND its residual pass (motion_conv_trans_28,
        # 147 x 1 tiles of 64: two tiles of 32 took 586 us against 371 us; unit_5a, 56 M tiles: five tiles of 32 columns
        # 38 us against ~20 for one of 160).  Only the 37-tile 7x7 layers are narrowed (sweep: profiles/env_r03s.log)
        want = enough = _X3_WANT_CTAS
    if mt * math.ceil(N / bn0) >= want:
        return 0
    best = 0
    for bn in (128, 64, 32):
        if bn < bn0 and N % bn == 0:
            best = bn
            if mt * (N // bn) >= enough:
                break
    return best


def _bind_epilogue(step, plan, spc: T.GemmSpec, d, tabs, *, tma, a_src, b_src, out, bias=None, relu_pre_cols=0,
                   gate=None, gate_col0=0, gate_first=False, addend=None, add_tabs=None, relu_post=False,
                   atomic=False, ones_out=None, split_k=1, tile_n=0, name="", finish=False, aux=None, out_vec=None):
    """Fill the fields of offk_gemm_t ``d`` that the gather-fed and the TMA-fed kernel read alike (problem size, operand
    sources, output tables, epilogue, split-K), and annotate ``step`` as a plan step."""
    d.M, d.N, d.K = spc.M, spc.N, spc.K
    d.a_src, d.b_src, d.a_ones_row = a_src.data_ptr(), b_src.data_ptr(), spc.a_ones_row
    d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
    d.bias = bias.data_ptr() if bias is not None else None
    d.relu_pre_cols = relu_pre_cols
    d.gate = gate.data_ptr() if gate is not None else None
    d.gate_col0, d.gate_first = gate_col0, int(gate_first)
    d.addend = addend.data_ptr() if addend is not None else None
    d.add_row = add_tabs[0].data_ptr() if add_tabs else None
    d.add_col = add_tabs[1].data_ptr() if add_tabs else None
    d.relu_post, d.atomic_out = int(relu_post), int(atomic)
    d.ones_row_out = ones_out.data_ptr() if ones_out is not None else None
    if tile_n == 0 and split_k == 1:
        tile_n = _auto_tile_n(spc.M, spc.N, tma, plan.prec == L.PREC_TF32X3)
    d.split_k, d.tile_n = split_k, tile_n
    d.out_vec = spc.out_vec if out_vec is None else out_vec
    counter = None
    if finish:                         # split-K finished in-kernel by the last CTA of each output tile (offk.h)
        bn = tile_n if tile_n else (256 if spc.N > 256 else (spc.N + 15) // 16 * 16)
        counter = torch.zeros(math.ceil(spc.M / 128) * math.ceil(spc.N / bn), dtype=torch.int32, device=plan.device)
        d.finish_counter = counter.data_ptr()
    if aux is not None:                # (aux_out, aux_row table or None, aux_addend or None)
        d.aux_out = aux[0].data_ptr()
        d.aux_row = aux[1].data_ptr() if aux[1] is not None else None
        d.aux_addend = aux[2].data_ptr() if aux[2] is not None else None
    step.plan, step.name, step.spec = plan, name, spc
    step._keep = (tabs, a_src, b_src, out, bias, gate, addend, add_tabs, ones_out, counter, aux)
    step.flops = 2.0 * spc.M * spc.N * spc.K
    step.launches = [name]
    step.reads = [a_src, b_src, addend, gate, bias, aux[2] if aux else None]
    step.writes = [out, ones_out, aux[0] if aux else None]
    step.lane = 0


class Gemm:
    """One bound gather-GEMM launch (offk_gather_gemm: descriptor + device tables kept alive)."""

    def __init__(self, plan: "LaunchPlan", spc: T.GemmSpec, key, name="", **kw):
        if spc.a_mode is None or spc.b_mode is None:
            raise ValueError(f"{name}: an operand of this {spc.kind} GEMM has no 16-byte load form (tables.GemmSpec)")
        tabs = plan._tables(key, spc, _ALL_TABLES)
        d = self.desc = L.OffkGemm()
        _bind_epilogue(self, plan, spc, d, tabs, tma=False, name=name, **kw)
        d.a_row, d.a_col = tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
        d.a_h, d.a_w = (spc.a_h, spc.a_w) if spc.a_h else (T.NO_BOX, T.NO_BOX)
        d.a_mode = spc.a_mode
        d.b_row, d.b_col, d.b_mode = tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
        T.check_modes(spc)

    def __call__(self, stream):
        L.check(self.plan.lib.offk_gather_gemm(C.byref(self.desc), self.plan.prec, stream), self.name)


class TGemm:
    """A conv / FC on a channels-last input (or an NCHW tap) as ONE TMA-fed launch (offk_tma_gemm): A through a dense
    2-D tensor map (1x1, stride 1) or TMA im2col mode (KxK), B = the [cout, K] weight matrix; or the weight gradient with
    A = im2col(x)^T / the NCHW tap and B = dY.  The epilogue reads the output tables (and the addend / aux tables a caller
    passes); the gather tables and load modes of offk_gemm_t stay 0."""

    @staticmethod
    def eligible(geom: T.ConvGeom, x_layout="nhwc") -> bool:
        if x_layout == "nchw":      # the taps, read in place as an MN-major operand: 1x1 conv over whole frames
            return (T._is1x1(geom) and geom.cin % 32 == 0 and geom.x_coff == 0 and geom.x_ctot == geom.cin
                    and (geom.hin * geom.win) % 4 == 0)
        return geom.cin % 32 == 0 and geom.x_ctot % 4 == 0 and geom.x_coff % 4 == 0 and geom.kdim % 4 == 0

    @staticmethod
    def wgrad_eligible(geom: T.ConvGeom, x_layout="nhwc") -> bool:
        """Weight gradient with both operands TMA-fed: A = im2col(x)^T (channels-last) or the NCHW tap, B = dY."""
        y_ok = geom.y_ctot % 4 == 0 and geom.y_coff % 4 == 0 and geom.cout % 4 == 0
        if x_layout == "nchw":
            return (y_ok and T._is1x1(geom) and geom.x_coff == 0 and geom.x_ctot == geom.cin
                    and (geom.hin * geom.win) % 4 == 0)
        return y_ok and geom.cin % 32 == 0 and geom.x_ctot % 4 == 0 and geom.x_coff % 4 == 0

    def __init__(self, plan: "LaunchPlan", spc: T.GemmSpec, key, geom: T.ConvGeom, x_layout="nhwc", wgrad=False, bk=0,
                 **kw):
        t = self.tdesc = L.OffkTGemm()
        _bind_epilogue(self, plan, spc, t.g, plan._tables(key, spc, _OUT_TABLES), tma=True, **kw)
        T.check_modes(spc, gather=False)
        one = geom.kh == 1 and geom.kw == 1 and geom.stride == 1 and geom.pad == 0
        if wgrad:
            t.a_kind = L.TMA_A_NCHW_T if x_layout == "nchw" else L.TMA_A_IM2COL_T
        elif x_layout == "nchw":
            t.a_kind = L.TMA_A_NCHW
        elif one:
            t.a_kind, t.lda = L.TMA_A_DENSE, geom.x_ctot
            t.g.a_src = kw["a_src"].data_ptr() + 4 * geom.x_coff
        else:
            t.a_kind = L.TMA_A_IM2COL
        t.a_coff = geom.x_coff
        if not wgrad and spc.out_vec == 1 and spc.M > 1:
            # linear output rows: a plain epilogue may leave through TMA tile stores (offk.h: out_ld)
            r = np.asarray(spc.out_row, dtype=np.int64)
            ld = int(r[1] - r[0])
            if ld > 0 and r[0] == 0 and np.array_equal(r, np.arange(spc.M, dtype=np.int64) * ld):
                t.out_ld, t.out_c0 = ld, int(spc.out_col[0])
        t.precision = plan.prec
        t.bk = bk if (wgrad and x_layout != "nchw") else 0
        if plan.presplit and not wgrad:
            # B is a weight matrix inside one of the plan's weight buffers: its residuals sit at the same offset of the
            # twin buffer
            bp = kw["b_src"].data_ptr()
            for hi, lo in plan.lo_twins:
                if hi.data_ptr() <= bp < hi.data_ptr() + hi.numel() * 4:
                    t.b_lo_delta = (lo.data_ptr() - hi.data_ptr()) // 4
                    self.reads.append(lo)
        t.n_img, t.hin, t.win, t.ctot, t.cin = geom.n_img, geom.hin, geom.win, geom.x_ctot, geom.cin
        t.kh, t.kw, t.stride, t.pad, t.hout, t.wout = geom.kh, geom.kw, geom.stride, geom.pad, geom.hout, geom.wout
        if isinstance(geom, _FreeGeom):
            t.geom_flags, t.pad_w = L.TGEMM_FREE_GEOM, geom.pad_w
        if wgrad:                         # B = dY[pixel, cout slice], row-major
            t.b_kind, t.ldb = L.TMA_B_DENSE_T, geom.y_ctot
            t.g.b_src = kw["b_src"].data_ptr() + 4 * geom.y_coff
        else:
            t.b_kind, t.ldb = L.TMA_B_DENSE, geom.kdim
        self._by_src = {}                 # a_src pointer -> prepared descriptor (the two tap sets alternate)

    @property
    def desc(self):
        """The offk_gemm_t inside the current descriptor."""
        return self.tdesc.g

    def set_a_src(self, ptr):
        if self.tdesc.g.a_src == ptr:
            return
        self._by_src[self.tdesc.g.a_src] = self.tdesc
        t = self._by_src.get(ptr)
        if t is None:
            t = L.OffkTGemm()
            C.memmove(C.byref(t), C.byref(self.tdesc), C.sizeof(L.OffkTGemm))
            t.g.a_src, t.prepared = ptr, 0
        self.tdesc = t

    def __call__(self, stream):
        lib = self.plan.lib
        if not self.tdesc.prepared:                                  # tensor maps are encoded on first use (needs a driver)
            L.check(lib.offk_tma_gemm_prepare(C.byref(self.tdesc)), self.name + " (prepare)")
        L.check(lib.offk_tma_gemm(C.byref(self.tdesc), stream), self.name)


class LaunchPlan:
    """State and policy shared by the static launch plans: the library, the device (a bare "cuda" is the current device),
    the precision mode (``prec``; ``presplit``: 3xTF32 with the weights' tf32 residuals in twin buffers, ``lo_twins``),
    the GEMM table cache, the algorithmic FLOP counts and the forward-conv launch policy (``_conv_fwd``).  An unknown
    precision raises KeyError."""

    def __init__(self, device, precision: str):
        self.lib = L.lib()
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            # "cuda" means the current device; tensors report it with its index ("cuda:0"), which the checks compare against
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.prec = {"fp32": L.PREC_TF32X3, "tf32": L.PREC_TF32}[precision]
        self.presplit = self.prec == L.PREC_TF32X3
        self.lo_twins = []               # [(weights, residuals)] buffer pairs allocated by _weights
        self._tab_cache = {}
        self.flops_fwd = self.flops_bwd = 0.0
        self._cap_stream = None

    def _weights(self, n):
        """A zeroed buffer of ``n`` weights and, in the fp32 (3xTF32) mode, the twin buffer of their tf32 residuals directly
        behind it (registered in ``lo_twins``), so that the GEMMs receive both weight tiles by TMA (offk.h: b_lo_delta) instead
        of splitting them in shared memory in every CTA and K-block.  Returns (weights, residuals or None)."""
        buf = torch.zeros(n * (2 if self.presplit else 1), device=self.device)
        if not self.presplit:
            return buf, None
        self.lo_twins.append((buf[:n], buf[n:]))
        return self.lo_twins[-1]

    def _tables(self, key, spc: T.GemmSpec, names):
        """Device copies of the padded tables ``names`` of ``spc`` (tables.padded_tables), cached per (key, names)."""
        ck = (key, names)
        if ck not in self._tab_cache:
            tabs = T.padded_tables(spc)
            self._tab_cache[ck] = {k: torch.from_numpy(tabs[k]).to(self.device) for k in names}
        return self._tab_cache[ck]

    def _conv_fwd(self, name, x, y, geom, w, b, *, relu=False, relu_cols=None, addend=None,
                  add_tabs=None, relu_post=False, x_layout="nhwc", no_split=False, aux=None):
        """One TMA-fed launch (TGemm); a geometry without a TMA-fed form is an error.  Returns the plan steps: the GEMM
        step and, when its epilogue cannot write ``aux``, the elementwise step that does.
        aux = (buffer, channel total, channel offset, addend | None, launch name): a second output
        max(v + addend, 0) of the conv's output v into channels [offset, offset + cout) of a channels-last buffer."""
        spc = T.conv_fwd_spec(geom, x_layout, "nhwc")
        m_tiles, kb = math.ceil(spc.M / 128), math.ceil(spc.K / 32)
        n_tiles = max(1, math.ceil(spc.N / 256))
        split = 1
        if addend is None and m_tiles * n_tiles < 200 and kb >= 32:
            # split-K factor: minimise rounds x K-blocks per CTA, rounds = ceil(CTAs / resident CTA slots) (two CTAs per SM in
            # the tf32 mode, one in the 3xTF32 mode whose stages are twice as large); ties go to the smaller factor.
            # 147 tiles: 2 splits = 294 CTAs = one round (3 splits were 1.49 rounds at 31 % tensor-pipe activity).
            slots = _SM_TARGET * (1 if self.prec == L.PREC_TF32X3 else 2)
            tiles = m_tiles * n_tiles
            split = min(range(1, max(1, kb // 8) + 1),
                        key=lambda s_: (math.ceil(tiles * s_ / slots) * math.ceil(kb / s_) * (1 if tiles * s_ >= 0.9 * _SM_TARGET else 4), s_))
        cols = (geom.cout if relu else 0) if relu_cols is None else relu_cols
        if not TGemm.eligible(geom, x_layout):
            raise ValueError(f"{name}: this conv geometry has no TMA-fed form (TGemm.eligible)")
        if x_layout == "nchw" or no_split:
            split = 1                     # per-frame M tiles already fill the machine (N * ceil(hw/128) CTAs)
        # in-kernel finishing pays when there are enough output tiles for the finishing CTAs to keep the machine busy
        # (motion_conv_trans_28: 147 tiles, same time as the bare split-K GEMM, bias_act and ReLU copy for free); with the
        # 37-tile 7x7 layers the fences + a finishing pass by 37 CTAs cost 9-27 us more than a separate full-grid bias_act
        # pass (measured, profiles/launches_tf32_r02g*.txt), so those keep the two-kernel form
        finish = split > 1 and spc.out_vec and m_tiles * n_tiles >= _FINISH_MIN_TILES
        # the second output is written by the epilogue wherever it produces final values, with the float4 epilogue (out_vec)
        aux_fused = aux is not None and spc.out_vec and (split == 1 or finish)
        aux_d = None
        if aux_fused:
            buf, ctot, coff, aux_add, _ = aux
            row = None                    # NULL: the output's own row table
            if (ctot, coff) != (geom.y_ctot, geom.y_coff):
                ga = T.ConvGeom(geom.n_img, geom.cout, geom.hout, geom.wout, geom.cout, y_ctot=ctot, y_coff=coff)
                row = self._tables(("fwd", "nhwc", _gkey(ga)), T.conv_fwd_spec(ga, "nhwc", "nhwc"), _OUT_TABLES)["out_row"]
            aux_d = (buf, row, aux_add)
        key, hw = ("fwd", x_layout, _gkey(geom)), geom.hout * geom.wout
        if split > 1:
            # split-K partial tiles are added into the zeroed output; either the last CTA of each tile applies bias / ReLU
            # (and writes the second output) in place, or a separate bias_act pass does
            assert geom.y_coff == 0 and geom.y_ctot == geom.cout
            epi = dict(bias=b, relu_pre_cols=cols, finish=True, aux=aux_d) if finish else {}
            g = TGemm(self, spc, key, geom, x_layout, a_src=x, b_src=w, out=y, split_k=split, name=name, **epi)

            def step(stream):
                L.check(self.lib.offk_fill_zero(_ptr(y), y.numel(), stream), name + ".zero")
                g(stream)
                if not finish:
                    L.check(self.lib.offk_bias_act(_ptr(y), _ptr(b), geom.n_img, geom.cout, hw, geom.y_ctot, geom.y_coff,
                                                   cols, stream), name + ".bias_act")
            step.name, step.flops, step.gemm = name, g.flops, g
            step.launches = [name + ".zero", name + ".splitk"] + ([] if finish else [name + ".bias_act"])
            step.reads, step.writes, step.lane = g.reads, g.writes, 0
        else:
            # nchw TMA: one N tile (re-reading the tap per N tile would multiply the HBM traffic of an HBM-bound GEMM)
            tn = (spc.N + 15) // 16 * 16 if (x_layout == "nchw" and spc.N <= 256) else 0
            g = step = TGemm(self, spc, key, geom, x_layout, a_src=x, b_src=w, out=y, bias=b, relu_pre_cols=cols,
                             addend=addend, add_tabs=add_tabs, relu_post=relu_post, tile_n=tn, name=name, aux=aux_d)
        self.flops_fwd += g.flops
        if aux is None or aux_fused:
            return [step]
        buf, ctot, coff, aux_add, aux_name = aux
        lib = self.lib
        if aux_add is None:               # the ReLU'd copy of the whole output
            assert (ctot, coff) == (geom.y_ctot, geom.y_coff)
            return [step, _nm(lambda stream: L.check(lib.offk_relu_gate(_ptr(y), _ptr(y), y.numel(), _ptr(buf), stream),
                                                     aux_name), aux_name, reads=[y], writes=[buf])]
        return [step, _nm(lambda stream: L.check(lib.offk_add_relu_slice(_ptr(aux_add), _ptr(y), _ptr(buf), ctot, coff,
                                                                          geom.n_img, geom.cout, hw, 1, stream), aux_name),
                          aux_name, reads=[aux_add, y], writes=[buf])]

    def _capture(self, issue):
        """Capture the pass that ``issue()`` enqueues on the current stream into a CUDA graph (side lanes fork from and join
        the capturing stream through the schedule's events, so the graph keeps the plan's multi-stream concurrency)."""
        main = torch.cuda.current_stream(self.device)
        if self._cap_stream is None:
            self._cap_stream = torch.cuda.Stream(device=self.device)
        cap = self._cap_stream
        cap.wait_stream(main)
        with torch.cuda.stream(cap):
            issue()                      # eager once on this stream: tensor maps encoded, kernel attributes set
        cap.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=cap):
            issue()
        main.wait_stream(cap)
        return g

    def launch_names(self):
        """One name per kernel launch of the plan's passes (``steps``), in issue order (for annotating launch lists)."""
        return _kernels(self.steps)


def _is_memset(name):
    return name.endswith(".zero") or name.startswith("zero ")


def _kernels(steps):
    """Launch names of ``steps`` that are liboffk kernels (cudaMemsetAsync zero-fills are not)."""
    return [n for st in steps for n in _names(st) if not _is_memset(n)]


def _nm(fn, name, reads=(), writes=(), lane=0):
    """Annotate a plan step: launch name, the buffers it reads / writes (for cross-stream hazard analysis), its lane."""
    fn.launches = [name]
    fn.reads, fn.writes, fn.lane = list(reads), list(writes), lane
    return fn


def _on(step, lane):
    step.lane = lane
    return step


def _span(t):
    return (t.data_ptr(), t.data_ptr() + t.numel() * t.element_size())


class Schedule:
    """A fixed list of steps spread over a few CUDA streams ("lanes").  Steps on one lane run in issue order; a step
    that touches a buffer last written (or still being read) by a step on another lane waits on an event recorded
    behind that step.  The hazards (RAW / WAW / WAR on byte ranges) are derived from the steps' declared reads and
    writes, so lane assignment is purely a performance choice: any assignment is correct."""

    def __init__(self, steps, ignore=()):
        self.steps = list(steps)
        n = len(self.steps)
        self.n_lanes = 1 + max((getattr(st, "lane", 0) for st in self.steps), default=0)
        ign = [_span(t) for t in ignore]

        def spans(ts):
            out = []
            for t in ts:
                if t is None:
                    continue
                sp = _span(t)
                if any(lo <= sp[0] and sp[1] <= hi for lo, hi in ign):
                    continue                      # read-only inputs (parameters, taps): never a hazard
                out.append(sp)
            return out

        rd = [spans(getattr(st, "reads", ())) for st in self.steps]
        wr = [spans(getattr(st, "writes", ())) for st in self.steps]
        hit = lambda A, B: any(a[0] < b[1] and b[0] < a[1] for a in A for b in B)
        lanes = [getattr(st, "lane", 0) for st in self.steps]
        self.lanes = lanes
        covered = [[-1] * self.n_lanes for _ in range(self.n_lanes)]   # covered[a][b]: latest step of lane b that a awaited
        self.waits = [[] for _ in range(n)]
        record = set()
        for i in range(n):
            need = {}
            for j in range(i):
                if lanes[j] == lanes[i] or j <= covered[lanes[i]][lanes[j]]:
                    continue
                if hit(wr[j], rd[i]) or hit(wr[j], wr[i]) or hit(rd[j], wr[i]):
                    need[lanes[j]] = j
            for lane_j, j in need.items():
                self.waits[i].append(j)
                covered[lanes[i]][lane_j] = j
                record.add(j)
        self.record = record
        self.events = {j: torch.cuda.Event() for j in record}

    def run(self, streams, lo=0, hi=None, on_step=None):
        """Issue steps [lo, hi) on ``streams`` (torch.cuda.Stream per lane; lane 0 = the caller's stream).
        ``on_step(step, stream)`` is called after each step has been issued."""
        hi = len(self.steps) if hi is None else hi
        handles = [C.c_void_p(st.cuda_stream) for st in streams]
        for i in range(lo, hi):
            lane = self.lanes[i]
            for j in self.waits[i]:
                streams[lane].wait_event(self.events[j])
            self.steps[i](handles[lane])
            if i in self.record:
                self.events[i].record(streams[lane])
            if on_step is not None:
                on_step(self.steps[i], streams[lane])


def _names(step):
    ls = getattr(step, "launches", None)
    if ls is not None:
        return list(ls)
    return [getattr(step, "name", None) or getattr(step, "__name__", "step")]


def _gkey(g: T.ConvGeom):
    return (g.n_img, g.cin, g.hin, g.win, g.cout, g.kh, g.kw, g.stride, g.pad, g.x_ctot, g.x_coff, g.y_ctot, g.y_coff)
