"""Index tables that turn every dense op of the OFF path into one gather-GEMM.

``D[m,n] = sum_k A(m,k) * B(n,k)`` with
``A(m,k) = a_src[a_row[m].off + a_col[k].off]`` (zero outside the validity box),
``B(n,k) = b_src[b_row[n] + b_col[k]]`` and ``out[out_row[m] + out_col[n]]``
(see include/offk.h).  The tables depend only on the layer geometry, so they are
built once per (batch, length) plan on the host with numpy and uploaded; the
kernels contain no div/mod and no layout knowledge.

Forward  (nn.Conv2d call sites RGB_OFF.py:597..:847):  m = output pixel, k = (c,r,q), n = cout
Wgrad    (autograd of the same):  m = (c,r,q) [+ one "ones" row -> bias grad], k = output pixel, n = cout
Dgrad    : m = input pixel of one stride-parity class, k = (cout,r',q'), n = cin

``emulate()`` evaluates a spec with numpy so the tables can be verified on a CPU
against plain conv2d / autograd (tests/test_tables.py).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import numpy as np

IDX_DTYPE = np.dtype([("off", "<i4"), ("y", "<i2"), ("x", "<i2")])


@dataclass
class ConvGeom:
    """y[n_img, cout, hout, wout] = conv2d(x[n_img, cin, hin, win], w[cout, cin, kh, kw], stride, pad);
    x / y may be channel slices [coff, coff+c) of wider NCHW buffers with ctot channels."""
    n_img: int
    cin: int
    hin: int
    win: int
    cout: int
    kh: int = 1
    kw: int = 1
    stride: int = 1
    pad: int = 0
    x_ctot: int = 0
    x_coff: int = 0
    y_ctot: int = 0
    y_coff: int = 0

    def __post_init__(self):
        self.x_ctot = self.x_ctot or self.cin
        self.y_ctot = self.y_ctot or self.cout
        self.hout = (self.hin + 2 * self.pad - self.kh) // self.stride + 1
        self.wout = (self.win + 2 * self.pad - self.kw) // self.stride + 1
        assert self.x_coff + self.cin <= self.x_ctot and self.y_coff + self.cout <= self.y_ctot
        lim = 2 ** 31 - 1
        assert self.n_img * self.x_ctot * self.hin * self.win < lim, "tensor too large for int32 offsets"
        assert self.n_img * self.y_ctot * self.hout * self.wout < lim, "tensor too large for int32 offsets"

    @property
    def kdim(self):
        return self.cin * self.kh * self.kw


@dataclass
class GemmSpec:
    """Host-side description of one gather-GEMM (numpy tables; pointers are bound later).  a_mode / b_mode: the
    16-byte load form the operand's layout allows (LOAD_VEC_K / LOAD_VEC_ROW), or None when it has none -- such a spec
    can be emulated on the CPU but not launched."""
    M: int
    N: int
    K: int
    a_row: np.ndarray
    a_col: np.ndarray
    b_row: np.ndarray
    b_col: np.ndarray
    out_row: np.ndarray
    out_col: np.ndarray
    a_h: int = 0
    a_w: int = 0
    a_ones_row: int = -1
    a_mode: Optional[int] = None
    b_mode: Optional[int] = None
    out_vec: int = 0
    kind: str = ""
    extra: dict = field(default_factory=dict)


LOAD_VEC_K, LOAD_VEC_ROW = 2, 3          # offk.h OFFK_LOAD_*


def _idx(off, y, x):
    off, y, x = np.broadcast_arrays(off, y, x)
    t = np.empty(off.shape, IDX_DTYPE)
    t["off"] = off
    t["y"] = y
    t["x"] = x
    return np.ascontiguousarray(t.reshape(-1))


def _i32(a):
    return np.ascontiguousarray(np.asarray(a).reshape(-1).astype(np.int32))


def _pixel_tables(g: ConvGeom, x_layout: str, y_layout: str):
    """Per output pixel m=(img,oh,ow): where its receptive field starts in x, and where it lives in y."""
    img, oh, ow = np.meshgrid(np.arange(g.n_img), np.arange(g.hout), np.arange(g.wout), indexing="ij")
    y0 = oh * g.stride - g.pad
    x0 = ow * g.stride - g.pad
    if x_layout == "nchw":
        off = (img * g.x_ctot + g.x_coff) * (g.hin * g.win) + y0 * g.win + x0
    else:
        off = ((img * g.hin + y0) * g.win + x0) * g.x_ctot + g.x_coff
    pix = oh * g.wout + ow
    if y_layout == "nchw":
        y_off = (img * g.y_ctot + g.y_coff) * (g.hout * g.wout) + pix
    else:
        y_off = (img * (g.hout * g.wout) + pix) * g.y_ctot + g.y_coff
    return _idx(off, y0, x0), _i32(y_off)


def _filter_tables(g: ConvGeom, x_layout: str):
    """Per filter tap: offset inside the receptive field.  k order is (c,r,q) for NCHW inputs (the canonical
    weight layout [cout,cin,kh,kw]) and (r,q,c) for NHWC inputs (weights permuted to [cout,kh,kw,cin])."""
    if x_layout == "nchw":
        c, r, q = np.meshgrid(np.arange(g.cin), np.arange(g.kh), np.arange(g.kw), indexing="ij")
        return _idx(c * (g.hin * g.win) + r * g.win + q, r, q)
    r, q, c = np.meshgrid(np.arange(g.kh), np.arange(g.kw), np.arange(g.cin), indexing="ij")
    return _idx((r * g.win + q) * g.x_ctot + c, r, q)


def _is1x1(g):
    return g.kh == 1 and g.kw == 1 and g.pad == 0 and g.stride == 1


def conv_fwd_spec(g: ConvGeom, x_layout: str = "nchw", y_layout: str = "nchw") -> GemmSpec:
    """y = conv2d(x, w) + epilogue.  A = im2col(x) gathered on the fly, B = w viewed as [cout, K]
    (K ordered like the x layout, see _filter_tables)."""
    a_row, y_off = _pixel_tables(g, x_layout, y_layout)
    K = g.kdim
    hw, hwo = g.hin * g.win, g.hout * g.wout
    box = not (g.kh == 1 and g.kw == 1 and g.pad == 0)
    if x_layout == "nhwc":
        a_mode = LOAD_VEC_K if (g.cin % 4 == 0 and g.x_ctot % 4 == 0 and g.x_coff % 4 == 0) else None
    else:
        a_mode = LOAD_VEC_ROW if (_is1x1(g) and hw % 4 == 0) else None
    if y_layout == "nhwc":
        out_col = np.arange(g.cout)
        out_vec = int(g.cout % 4 == 0 and g.y_ctot % 4 == 0 and g.y_coff % 4 == 0)
    else:
        out_col, out_vec = np.arange(g.cout) * hwo, 0
    return GemmSpec(
        M=g.n_img * hwo, N=g.cout, K=K, a_row=a_row, a_col=_filter_tables(g, x_layout),
        b_row=_i32(np.arange(g.cout) * K), b_col=_i32(np.arange(K)), out_row=y_off, out_col=_i32(out_col),
        a_h=g.hin if box else 0, a_w=g.win if box else 0, a_mode=a_mode,
        b_mode=LOAD_VEC_K if K % 4 == 0 else None, out_vec=out_vec, kind="fwd")


def conv_wgrad_spec(g: ConvGeom, x_layout: str = "nchw", y_layout: str = "nchw", dw_layout: str = None) -> GemmSpec:
    """dW[cout, K_w] += sum_pixels dY * im2col(x);  the extra all-ones A row yields db[cout].
    Rows are the filter taps in the x-layout k order, k walks output pixels.  dw_layout: where row (c,r,q) lands in
    dW -- default = the x-layout k order (OHWI for channels-last inputs); 'oihw' = the reference's canonical
    [cout,cin,kh,kw] whatever the input layout (the gradient then needs no un-permute pass)."""
    pix, _ = _pixel_tables(g, x_layout, y_layout)
    K_w = g.kdim
    hw, hwo = g.hin * g.win, g.hout * g.wout
    box = not (g.kh == 1 and g.kw == 1 and g.pad == 0)
    a_row = np.concatenate([_filter_tables(g, x_layout), np.zeros(1, IDX_DTYPE)])
    img = np.repeat(np.arange(g.n_img), hwo)
    p = np.tile(np.arange(hwo), g.n_img)
    if x_layout == "nhwc":
        a_mode = LOAD_VEC_ROW if (g.cin % 4 == 0 and g.x_ctot % 4 == 0 and g.x_coff % 4 == 0) else None
    else:
        a_mode = LOAD_VEC_K if (_is1x1(g) and hw % 4 == 0) else None
    if y_layout == "nhwc":
        b_row, b_col = np.arange(g.cout) + g.y_coff, (img * hwo + p) * g.y_ctot
        b_mode = LOAD_VEC_ROW if (g.cout % 4 == 0 and g.y_ctot % 4 == 0 and g.y_coff % 4 == 0) else None
    else:
        b_row, b_col = (np.arange(g.cout) + g.y_coff) * hwo, img * g.y_ctot * hwo + p
        b_mode = LOAD_VEC_K if hwo % 4 == 0 else None
    out_row = np.arange(K_w + 1)
    if dw_layout == "oihw" and x_layout == "nhwc":
        r, q, c = np.meshgrid(np.arange(g.kh), np.arange(g.kw), np.arange(g.cin), indexing="ij")
        out_row = np.concatenate([(c * (g.kh * g.kw) + r * g.kw + q).reshape(-1), [0]])
    return GemmSpec(
        M=K_w + 1, N=g.cout, K=g.n_img * hwo, a_row=a_row, a_col=pix, b_row=_i32(b_row), b_col=_i32(b_col),
        out_row=_i32(out_row), out_col=_i32(np.arange(g.cout) * K_w),
        a_h=g.hin if box else 0, a_w=g.win if box else 0, a_ones_row=K_w, a_mode=a_mode, b_mode=b_mode, kind="wgrad")


def conv_dgrad_specs(g: ConvGeom, x_layout: str = "nchw", y_layout: str = "nchw", w_layout: str = None):
    """dX = conv_transpose(dY, w), one GEMM per stride-parity class (a,b) of the input pixel
    (ih = s*ih' + a):  only filter rows r = r0 + s*r' with r0 = (a+pad) % s reach that class, so the
    zero-stuffed taps of a strided transposed conv are never multiplied.
    w_layout: 'nchw' = canonical [cout,cin,kh,kw], 'nhwc' = permuted [cout,kh,kw,cin] (default: x_layout)."""
    w_layout = w_layout or x_layout
    s, p = g.stride, g.pad
    hwo, hwi = g.hout * g.wout, g.hin * g.win
    kw_tot = g.cin * g.kh * g.kw
    specs = []
    for a in range(s):
        for b in range(s):
            r0, q0 = (a + p) % s, (b + p) % s
            rs, qs = np.arange(r0, g.kh, s), np.arange(q0, g.kw, s)
            hc, wc = len(range(a, g.hin, s)), len(range(b, g.win, s))
            if hc == 0 or wc == 0:
                continue
            assert len(rs) > 0 and len(qs) > 0, "stride larger than kernel is not on the OFF path"
            dh, dw = (a + p - r0) // s, (b + p - q0) // s
            img, ih, iw = np.meshgrid(np.arange(g.n_img), np.arange(hc), np.arange(wc), indexing="ij")
            oy, ox = ih + dh, iw + dw
            if y_layout == "nchw":
                a_row = _idx((img * g.y_ctot + g.y_coff) * hwo + oy * g.wout + ox, oy, ox)
                co, rr, qq = np.meshgrid(np.arange(g.cout), np.arange(len(rs)), np.arange(len(qs)), indexing="ij")
                a_col = _idx(co * hwo - rr * g.wout - qq, -rr, -qq)
                a_mode = None
            else:
                a_row = _idx(((img * g.hout + oy) * g.wout + ox) * g.y_ctot + g.y_coff, oy, ox)
                rr, qq, co = np.meshgrid(np.arange(len(rs)), np.arange(len(qs)), np.arange(g.cout), indexing="ij")
                a_col = _idx((-rr * g.wout - qq) * g.y_ctot + co, -rr, -qq)
                a_mode = LOAD_VEC_K if (g.cout % 4 == 0 and g.y_ctot % 4 == 0 and g.y_coff % 4 == 0) else None
            r_full, q_full = r0 + s * rr, q0 + s * qq
            if w_layout == "nchw":
                b_row = np.arange(g.cin) * (g.kh * g.kw)
                b_col = co * kw_tot + r_full * g.kw + q_full
                b_mode = None
            else:
                b_row = np.arange(g.cin)
                b_col = co * kw_tot + (r_full * g.kw + q_full) * g.cin
                b_mode = LOAD_VEC_ROW if g.cin % 4 == 0 else None
            iy, ix = s * ih + a, s * iw + b
            if x_layout == "nchw":
                out_row = (img * g.x_ctot + g.x_coff) * hwi + iy * g.win + ix
                out_col, out_vec = np.arange(g.cin) * hwi, 0
            else:
                out_row = ((img * g.hin + iy) * g.win + ix) * g.x_ctot + g.x_coff
                out_col = np.arange(g.cin)
                out_vec = int(g.cin % 4 == 0 and g.x_ctot % 4 == 0 and g.x_coff % 4 == 0)
            specs.append(GemmSpec(
                M=g.n_img * hc * wc, N=g.cin, K=g.cout * len(rs) * len(qs), a_row=a_row, a_col=a_col,
                b_row=_i32(b_row), b_col=_i32(b_col), out_row=_i32(out_row), out_col=_i32(out_col),
                a_h=g.hout, a_w=g.wout, a_mode=a_mode, b_mode=b_mode, out_vec=out_vec, kind=f"dgrad[{a},{b}]",
                # the same class as a stride-1 correlation over dY (TMA im2col form): output grid hc x wc, filter
                # len(rs) x len(qs) with taps walked in reverse, top / left padding len(rs)-1-dh / len(qs)-1-dw
                extra=dict(a=a, b=b, rs=rs, qs=qs, hc=hc, wc=wc, pad_h=len(rs) - 1 - dh, pad_w=len(qs) - 1 - dw)))
    return specs


def dgrad_class_weight_index(cout: int, cin: int, k: int, stride: int, pad: int, a: int, b: int) -> np.ndarray:
    """Element indices into an OIHW weight [cout, cin, k, k] that lay out the B operand of the data-gradient GEMM of
    stride-parity class (a, b) as [cin, R, Q, cout]: only the taps r = r0 + stride*i (r0 = (a + pad) % stride) reach
    input rows of parity a, and the im2col form of that class walks them in reverse (``conv_dgrad_specs`` ``extra``).
    For stride 1 this is the whole filter flipped: dX = conv(dY, flip(W)^T)."""
    oihw = np.arange(cout * cin * k * k, dtype=np.int64).reshape(cout, cin, k, k)
    rs = np.arange((a + pad) % stride, k, stride)[::-1]
    qs = np.arange((b + pad) % stride, k, stride)[::-1]
    return oihw[:, :, rs][:, :, :, qs].transpose(1, 2, 3, 0).reshape(-1)


def emulate_dgrad_class(g: ConvGeom, spec: GemmSpec, dy_nhwc: np.ndarray, w_oihw: np.ndarray) -> np.ndarray:
    """numpy mirror of what the TMA-im2col kernel computes for one stride-parity class of the data gradient
    (OFFK_TGEMM_FREE_GEOM): a stride-1 correlation over dY [n, hout, wout, cout] with the class's R x Q taps, output
    grid hc x wc, zero padding pad_h rows above / pad_w columns left.  Returns D[M = n*hc*wc, N = cin] (float64)."""
    ex = spec.extra
    R, Q, hc, wc = len(ex["rs"]), len(ex["qs"]), ex["hc"], ex["wc"]
    idx = dgrad_class_weight_index(g.cout, g.cin, g.kh, g.stride, g.pad, ex["a"], ex["b"])
    wcls = w_oihw.reshape(-1).astype(np.float64)[idx].reshape(g.cin, R, Q, g.cout)
    dy = dy_nhwc.astype(np.float64)
    pad = np.zeros((g.n_img, hc + R - 1 + g.hout, wc + Q - 1 + g.wout, g.cout))
    pad[:, ex["pad_h"]:ex["pad_h"] + g.hout, ex["pad_w"]:ex["pad_w"] + g.wout] = dy
    out = np.zeros((g.n_img, hc, wc, g.cin))
    for r in range(R):
        for q in range(Q):
            out += pad[:, r:r + hc, q:q + wc] @ wcls[:, r, q].T
    return out.reshape(-1, g.cin)


def check_modes(spec: GemmSpec, gather: bool = True):
    """Assert the promises behind the vector store mode and, for a gather-fed launch (``gather``), behind the vector load
    modes (contiguity, alignment, shared validity)."""
    def quads(tab, n):
        t = tab[: n - n % 4].reshape(-1, 4)
        return t

    if spec.out_vec:
        assert spec.N % 4 == 0 and (spec.out_col == spec.out_col[0] + np.arange(spec.N)).all()
        assert spec.out_col[0] % 4 == 0 and (spec.out_row % 4 == 0).all()
    if not gather:
        return
    if spec.a_mode == LOAD_VEC_K:
        assert spec.K % 4 == 0
        q = quads(spec.a_col, spec.K)
        assert (q["off"] == q["off"][:, :1] + np.arange(4)).all() and (q["off"][:, 0] % 4 == 0).all()
        assert spec.a_h == 0 or ((q["y"] == q["y"][:, :1]).all() and (q["x"] == q["x"][:, :1]).all())
        rows = spec.a_row if spec.a_ones_row < 0 else np.delete(spec.a_row, spec.a_ones_row)
        assert (rows["off"] % 4 == 0).all()
    if spec.a_mode == LOAD_VEC_ROW:
        m_real = spec.M - (1 if spec.a_ones_row >= 0 else 0)
        assert m_real % 4 == 0 and spec.a_ones_row in (-1, m_real)
        q = quads(spec.a_row[:m_real], m_real)
        assert (q["off"] == q["off"][:, :1] + np.arange(4)).all() and (q["off"][:, 0] % 4 == 0).all()
        assert spec.a_h == 0 or ((q["y"] == q["y"][:, :1]).all() and (q["x"] == q["x"][:, :1]).all())
        assert (spec.a_col["off"] % 4 == 0).all()
    if spec.b_mode == LOAD_VEC_K:
        assert spec.K % 4 == 0
        q = quads(spec.b_col, spec.K)
        assert (q == q[:, :1] + np.arange(4)).all() and (q[:, 0] % 4 == 0).all() and (spec.b_row % 4 == 0).all()
    if spec.b_mode == LOAD_VEC_ROW:
        assert spec.N % 4 == 0
        q = quads(spec.b_row, spec.N)
        assert (q == q[:, :1] + np.arange(4)).all() and (q[:, 0] % 4 == 0).all() and (spec.b_col % 4 == 0).all()


NO_BOX = 32767          # a_h / a_w value meaning "every real element is valid"
PAD_Y = -16384          # y of padding entries: never inside any box


def padded_tables(spec: GemmSpec):
    """Device-ready int32 arrays obeying the padding contract of the tensor-core kernel (include/offk.h):
    a_row -> ceil(M/128)*128 entries, a_col / b_col -> ceil(K/32)*32 + 64, b_row -> ceil(N/256)*256;
    A padding entries have y = PAD_Y (rejected by the always-on box test), B padding entries are 0."""
    def pad_idx(t, n):
        out = np.zeros(n, IDX_DTYPE)
        out["y"] = PAD_Y
        out[: len(t)] = t
        return out

    def pad_i32(t, n):
        out = np.zeros(n, np.int32)
        out[: len(t)] = t
        return out

    kp = (spec.K + 31) // 32 * 32 + 64
    a_row = pad_idx(spec.a_row, (spec.M + 127) // 128 * 128)
    if spec.a_ones_row >= 0:
        a_row[spec.a_ones_row]["y"] = PAD_Y          # never gathered; the kernel synthesises the ones
    tabs = {
        "a_row": a_row, "a_col": pad_idx(spec.a_col, kp),
        "b_row": pad_i32(spec.b_row, (spec.N + 255) // 256 * 256), "b_col": pad_i32(spec.b_col, kp),
        "out_row": spec.out_row, "out_col": spec.out_col,
    }
    return {k: np.ascontiguousarray(v).view(np.int32).reshape(-1) for k, v in tabs.items()}


def emulate(spec: GemmSpec, a_src: np.ndarray, b_src: np.ndarray) -> np.ndarray:
    """Dense D[M,N] of a spec, evaluated with numpy (float64).  CPU-side check of the tables only."""
    a_src = a_src.reshape(-1).astype(np.float64)
    b_src = b_src.reshape(-1).astype(np.float64)
    ar, ac = spec.a_row, spec.a_col
    D = np.zeros((spec.M, spec.N))
    B = b_src[spec.b_row.astype(np.int64)[:, None] + spec.b_col.astype(np.int64)[None, :]]  # [N,K]
    step = max(1, (1 << 22) // max(spec.K, 1))
    for m0 in range(0, spec.M, step):
        r = ar[m0:m0 + step]
        off = r["off"].astype(np.int64)[:, None] + ac["off"].astype(np.int64)[None, :]
        if spec.a_h:
            y = r["y"].astype(np.int32)[:, None] + ac["y"].astype(np.int32)[None, :]
            x = r["x"].astype(np.int32)[:, None] + ac["x"].astype(np.int32)[None, :]
            ok = (y >= 0) & (y < spec.a_h) & (x >= 0) & (x < spec.a_w)
        else:
            ok = np.ones(off.shape, bool)
        A = np.where(ok, a_src[np.where(ok, off, 0)], 0.0)
        if spec.a_ones_row >= 0 and m0 <= spec.a_ones_row < m0 + step:
            A[spec.a_ones_row - m0] = 1.0
        D[m0:m0 + step] = A @ B.T
    return D


def scatter(spec: GemmSpec, D: np.ndarray, out: np.ndarray, ones_out: Optional[np.ndarray] = None, accumulate=False):
    """Write / accumulate D through the output tables into the flat buffer ``out`` (numpy mirror of the epilogue
    without bias / activation)."""
    o = out.reshape(-1)
    rows = np.arange(spec.M)
    if spec.a_ones_row >= 0:
        if ones_out is not None:
            ones_out += D[spec.a_ones_row]
        rows = rows[rows != spec.a_ones_row]
    idx = spec.out_row.astype(np.int64)[rows][:, None] + spec.out_col.astype(np.int64)[None, :]
    if accumulate:
        np.add.at(o, idx, D[rows])
    else:
        o[idx] = D[rows]
    return out
