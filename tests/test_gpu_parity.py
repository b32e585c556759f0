"""GPU: parity of the sm_100a path with the CPU oracle, through the C ABI (liboffk.so).

Tolerances (stated per mode, as BASELINE.json's north_star asks):
  fp32 mode (3xTF32 tcgen05, fp32 accumulate): <= 2e-5 max-abs relative to the tensor's max, per level / head;
  tf32 mode (tcgen05 kind::tf32, fp32 accumulate): <= 5e-3 on the stage-fusion tensors, <= 1e-2 on the logits;
  gradients are compared in relative L2 norm (a single ReLU whose pre-activation sits within round-off of 0 may flip
  between fp32 and the fp64 oracle, which moves individual entries but not the norm): fp32 <= 2e-3, tf32 <= 0.2.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import off_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def dev():
    import off_b200  # noqa: F401
    from off_b200 import _lib
    _lib.lib()            # raises if the extension is missing: no fallback
    return torch.device("cuda")


def _rel(a, b):
    b = b.double()
    return (a.detach().double().cpu() - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _rel_l2(a, b):
    b = b.double()
    return (a.detach().double().cpu() - b).norm().item() / max(b.norm().item(), 1e-30)


def _run_spec(spc, a_src, b_src, out_shape, prec, dev, bias=None, ones=None, split_k=1, atomic=False):
    from off_b200 import _lib as L, tables as T
    tabs = {k: torch.from_numpy(v).to(dev) for k, v in T.padded_tables(spc).items()}
    out = torch.zeros(out_shape, device=dev)
    d = L.OffkGemm()
    d.M, d.N, d.K = spc.M, spc.N, spc.K
    d.a_src, d.a_row, d.a_col = a_src.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
    d.a_h, d.a_w = (spc.a_h, spc.a_w) if spc.a_h else (T.NO_BOX, T.NO_BOX)
    d.a_ones_row, d.a_mode = spc.a_ones_row, spc.a_mode
    d.b_src, d.b_row, d.b_col, d.b_mode = b_src.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
    d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
    d.bias = bias.data_ptr() if bias is not None else None
    d.ones_row_out = ones.data_ptr() if ones is not None else None
    d.split_k, d.atomic_out, d.out_vec = split_k, int(atomic), spc.out_vec
    L.check(L.lib().offk_gather_gemm(C.byref(d), prec, None), "gemm")
    torch.cuda.synchronize()
    return out


GEMM_CASES = [
    # n, cin, h, w, cout, k, s, p, x_ctot, x_coff, y_ctot, y_coff, x_layout, y_layout
    (3, 8, 7, 7, 8, 1, 1, 0, 8, 0, 8, 0, "nchw", "nhwc"),          # unit conv, 7x7 taps: data gradient only
    (5, 64, 14, 14, 160, 1, 1, 0, 64, 0, 160, 0, "nchw", "nhwc"),  # unit conv, vectorised transposing loader
    (4, 64, 14, 14, 64, 3, 1, 1, 64, 0, 64, 0, "nhwc", "nhwc"),
    (2, 32, 28, 28, 64, 7, 2, 3, 32, 0, 64, 0, "nhwc", "nhwc"),  # motion_conv_trans_28 geometry
    (2, 24, 14, 14, 128, 5, 2, 2, 40, 8, 160, 32, "nhwc", "nhwc"),  # 5x5 s2 on channel slices
    (3, 128, 7, 7, 512, 3, 1, 1, 128, 0, 512, 0, "nhwc", "nhwc"),  # N > 256: two N tiles
    (8, 1024, 1, 1, 101, 1, 1, 0, 1024, 0, 101, 0, "nhwc", "nhwc"),  # FC head, N not a multiple of 4: forward only
]


@pytest.mark.parametrize("prec,tol", [(1, 3e-3), (2, 1e-5)], ids=["tf32", "tf32x3"])
@pytest.mark.parametrize("case", GEMM_CASES, ids=[f"{c[1]}x{c[2]}k{c[5]}s{c[6]}{c[12]}" for c in GEMM_CASES])
def test_gather_gemm_conv_parity(dev, case, prec, tol):
    """Forward, weight gradient and data gradient of a conv through offk_gather_gemm against autograd of conv2d; a GEMM
    whose operand layout has no 16-byte load form (tables.GemmSpec mode None) cannot be launched and is skipped."""
    from off_b200 import tables as T
    n, cin, h, w, cout, k, s, p, xct, xco, yct, yco, xl, yl = case
    g = T.ConvGeom(n, cin, h, w, cout, k, k, s, p, xct, xco, yct, yco)
    torch.manual_seed(0)
    x = torch.randn(n, xct, h, w, device=dev)
    wt = torch.randn(cout, cin, k, k, device=dev) / (g.kdim ** 0.5)
    b = torch.randn(cout, device=dev)
    dy = torch.randn(n, yct, g.hout, g.wout, device=dev)
    xs = x[:, xco:xco + cin].double().requires_grad_(True)
    wd = wt.double().requires_grad_(True)
    y = torch.nn.functional.conv2d(xs, wd, b.double(), s, p)
    y.backward(dy[:, yco:yco + cout].double())
    to = lambda a, lay: a.permute(0, 2, 3, 1).contiguous() if lay == "nhwc" else a
    back = lambda a, lay: a.permute(0, 3, 1, 2) if lay == "nhwc" else a
    xb, dyb = to(x, xl), to(dy, yl)
    wl = wt.permute(0, 2, 3, 1).contiguous() if xl == "nhwc" else wt
    launchable = lambda spc: spc.a_mode is not None and spc.b_mode is not None
    ran = 0
    fwd = T.conv_fwd_spec(g, xl, yl)
    if launchable(fwd):
        out = back(_run_spec(fwd, xb, wl, tuple(dyb.shape), prec, dev, bias=b), yl)
        assert _rel(out[:, yco:yco + cout], y.detach().cpu()) < tol
        other = torch.cat([out[:, :yco], out[:, yco + cout:]], 1)
        assert other.abs().max().item() == 0 if other.numel() else True           # channel slice only
        out2 = back(_run_spec(fwd, xb, wl, tuple(dyb.shape), prec, dev, split_k=3), yl)
        assert _rel(out2[:, yco:yco + cout], (y - b.double().view(1, -1, 1, 1)).detach().cpu()) < tol
        ran += 1
    wgrad = T.conv_wgrad_spec(g, xl, yl)
    if launchable(wgrad):
        db = torch.zeros(cout, device=dev)
        dw = _run_spec(wgrad, xb, dyb, tuple(wl.shape), prec, dev, ones=db, split_k=4, atomic=True)
        dwc = dw.permute(0, 3, 1, 2) if xl == "nhwc" else dw
        assert _rel(dwc, wd.grad.cpu()) < tol
        assert _rel(db, dy[:, yco:yco + cout].double().sum((0, 2, 3)).cpu()) < tol
        ran += 1
    # a 1x1 weight is the same memory in OIHW and OHWI: the NCHW cases take the weight layout of the engine's tap gradients
    dgrads = T.conv_dgrad_specs(g, xl, yl, "nhwc" if k == 1 else xl)
    if all(launchable(spc) for spc in dgrads):
        dx = torch.zeros_like(xb)
        for spc in dgrads:
            dx += _run_spec(spc, dyb, wl, tuple(xb.shape), prec, dev)
        assert _rel(back(dx, xl)[:, xco:xco + cin], xs.grad.cpu()) < tol
        ran += 1
    assert ran > 0


TMA_CASES = [
    # n, cin, h, w, cout, k, s, p, x_ctot, x_coff, y_ctot, y_coff, split_k
    (4, 64, 14, 14, 256, 1, 1, 0, 64, 0, 256, 0, 1),        # dense A (1x1), one N tile
    (3, 128, 7, 7, 512, 1, 1, 0, 160, 32, 512, 0, 1),       # dense A on a channel slice, two N tiles, M = 147
    (5, 64, 14, 14, 64, 3, 1, 1, 64, 0, 64, 0, 1),          # im2col 3x3, tiles straddle rows and images
    (3, 32, 28, 28, 64, 7, 2, 3, 32, 0, 64, 0, 1),          # motion_conv_trans_28 geometry (7x7 stride 2)
    (2, 96, 14, 14, 128, 5, 2, 2, 160, 32, 160, 32, 1),     # 5x5 stride 2 on channel slices, M = 98
    (3, 128, 7, 7, 128, 3, 1, 1, 128, 0, 128, 0, 4),        # split-K accumulation
    (8, 1024, 1, 1, 101, 1, 1, 0, 1024, 0, 101, 0, 1),      # FC head, N = 101
]


PRECS = pytest.mark.parametrize("prec,tol", [(1, 3e-3), (2, 1e-5)], ids=["tf32", "tf32x3"])


@PRECS
@pytest.mark.parametrize("case", TMA_CASES, ids=[f"{c[1]}x{c[2]}k{c[5]}s{c[6]}n{c[4]}" for c in TMA_CASES])
def test_tma_gemm_conv_parity(dev, case, prec, tol):
    """offk_tma_gemm (TMA dense / im2col operand fetch + tcgen05) against conv2d, and against the gather-fed tensor-core
    kernel on the same operands: bit for bit in the tf32 mode (same products, same fp32 accumulation order per K-block)."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, h, w, cout, k, st, p, xct, xco, yct, yco, split = case
    g = T.ConvGeom(n, cin, h, w, cout, k, k, st, p, xct, xco, yct, yco)
    torch.manual_seed(0)
    x = torch.randn(n, xct, h, w, device=dev)
    wt = torch.randn(cout, cin, k, k, device=dev) / (g.kdim ** 0.5)
    bias = torch.randn(cout, device=dev)
    xl = x.permute(0, 2, 3, 1).contiguous()
    wl = wt.permute(0, 2, 3, 1).contiguous()                        # OHWI
    spc = T.conv_fwd_spec(g, "nhwc", "nhwc")
    tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
    outs = []
    for use_tma, tma_store in ((True, False), (False, False), (True, True)):
        out = torch.zeros(n, g.hout, g.wout, yct, device=dev)
        t = L.OffkTGemm()
        d = t.g
        d.M, d.N, d.K = spc.M, spc.N, spc.K
        d.a_src, d.a_row, d.a_col = xl.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
        d.a_h, d.a_w = (spc.a_h, spc.a_w) if spc.a_h else (T.NO_BOX, T.NO_BOX)
        d.a_ones_row, d.a_mode = -1, spc.a_mode
        d.b_src, d.b_row, d.b_col, d.b_mode = wl.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
        d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
        d.bias = bias.data_ptr() if split == 1 else None
        d.split_k, d.out_vec = split, spc.out_vec
        if tma_store:                      # linear output rows: the epilogue may leave through TMA tile stores (offk.h: out_ld)
            t.out_ld, t.out_c0 = yct, yco
        if use_tma:
            one = k == 1 and st == 1 and p == 0
            t.a_kind, t.lda, t.a_coff = (L.TMA_A_DENSE if one else L.TMA_A_IM2COL), xct, xco
            if one:
                d.a_src = xl.data_ptr() + 4 * xco
            t.n_img, t.hin, t.win, t.ctot, t.cin = n, h, w, xct, cin
            t.kh, t.kw, t.stride, t.pad, t.hout, t.wout = k, k, st, p, g.hout, g.wout
            t.b_kind, t.ldb, t.precision = L.TMA_B_DENSE, g.kdim, prec
            L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
            L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
        else:
            L.check(lib.offk_gather_gemm(C.byref(d), prec, None), "gather_gemm")
        torch.cuda.synchronize()
        outs.append(out)
    ref = torch.nn.functional.conv2d(x[:, xco:xco + cin].double(), wt.double(), bias.double() if split == 1 else None, st, p)
    got = outs[0].permute(0, 3, 1, 2)[:, yco:yco + cout]
    assert _rel(got, ref.cpu()) < tol
    if yco:
        assert outs[0][..., :yco].abs().max().item() == 0
    # TMA tile stores / adds against st.global / red.global of the same kernel: the same values (the same arithmetic per element)
    if split == 1:
        assert torch.equal(outs[0], outs[2])
    else:
        assert _rel(outs[0], outs[2].cpu()) < 1e-5
    if split == 1 and prec == 1:
        assert torch.equal(outs[0], outs[1])
    elif split == 1:
        # 3xTF32: the TMA-fed kernel may keep A in tensor memory with another number of partial accumulators than the
        # gather-fed one (same products, different fp32 grouping of the K-blocks)
        assert _rel(outs[0], outs[1].cpu()) < 5e-6
    else:
        assert _rel(outs[0], outs[1].cpu()) < 1e-5                   # atomics: summation order differs


NCHW_CASES = [
    # n_img, cin, s, cout, relu_cols
    (3, 256, 28, 160, 128),     # level 3a: 784 pixels = 6 full M tiles + a 16-pixel one per frame
    (4, 320, 14, 160, 128),     # 196 pixels: 128 + 68 (the second tile skips one 32-pixel atom)
    (2, 608, 14, 160, 128),     # 19 K-blocks: the pipeline wraps several times
    (5, 64, 6, 48, 0),          # 36 pixels: one partial tile, partial atom, N = 48
]


@PRECS
@pytest.mark.parametrize("case", NCHW_CASES, ids=[f"n{c[0]}c{c[1]}s{c[2]}" for c in NCHW_CASES])
def test_tma_gemm_nchw_taps(dev, case, prec, tol):
    """The OFF units' fused 1x1 conv (RGB_OFF.py:597-598,610) with the NCHW tap fetched in place by TMA as the MN-major
    tcgen05 operand (OFFK_TMA_A_NCHW): against conv2d, and bit-for-bit against the gather-fed kernel."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, s_, cout, relu_cols = case
    g = T.ConvGeom(n, cin, s_, s_, cout)
    torch.manual_seed(1)
    x = torch.relu(torch.randn(n, cin, s_, s_, device=dev))
    wt = torch.randn(cout, cin, device=dev) / cin ** 0.5
    bias = torch.randn(cout, device=dev)
    spc = T.conv_fwd_spec(g, "nchw", "nhwc")
    tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
    outs = []
    for use_tma, tma_store in ((True, False), (False, False), (True, True)):
        out = torch.zeros(n, s_, s_, cout, device=dev)
        t = L.OffkTGemm()
        d = t.g
        d.M, d.N, d.K = spc.M, spc.N, spc.K
        d.a_src, d.a_row, d.a_col = x.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
        d.a_h, d.a_w = T.NO_BOX, T.NO_BOX
        d.a_ones_row, d.a_mode = -1, spc.a_mode
        d.b_src, d.b_row, d.b_col, d.b_mode = wt.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
        d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
        d.bias, d.relu_pre_cols = bias.data_ptr(), relu_cols
        d.split_k, d.out_vec, d.tile_n = 1, spc.out_vec, (cout + 15) // 16 * 16
        if tma_store:                      # per-frame M tiles: 3-D output map, rows clip at the frame end
            t.out_ld, t.out_c0 = cout, 0
        if use_tma:
            t.a_kind = L.TMA_A_NCHW
            t.n_img, t.hin, t.win, t.ctot, t.cin = n, s_, s_, cin, cin
            t.kh = t.kw = t.stride = 1
            t.hout, t.wout = s_, s_
            t.b_kind, t.ldb, t.precision = L.TMA_B_DENSE, cin, prec
            L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
            L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
        else:
            L.check(lib.offk_gather_gemm(C.byref(d), prec, None), "gather_gemm")
        torch.cuda.synchronize()
        outs.append(out)
    ref = torch.nn.functional.conv2d(x.double(), wt.double()[:, :, None, None], bias.double())
    ref[:, :relu_cols] = torch.relu(ref[:, :relu_cols])
    assert _rel(outs[0].permute(0, 3, 1, 2), ref.cpu()) < tol
    assert torch.equal(outs[0], outs[2])                             # TMA tile stores: the same values as st.global
    if prec == 1:
        assert torch.equal(outs[0], outs[1])
    else:
        assert _rel(outs[0], outs[1].cpu()) < 5e-6                   # 3xTF32: partial-accumulator grouping may differ


WGRAD_CASES = [
    # n, cin, h, w, cout, k, s, p, x_ctot, x_coff, y_ctot, y_coff, x_layout, split_k
    (5, 64, 14, 14, 64, 3, 1, 1, 64, 0, 64, 0, "nhwc", 1),        # 3x3; K = 980 pixels (tail K-block), M = 577
    (3, 32, 28, 28, 64, 7, 2, 3, 32, 0, 64, 0, "nhwc", 3),        # motion_conv_trans_28 geometry, split-K
    (4, 64, 14, 14, 256, 1, 1, 0, 96, 32, 288, 32, "nhwc", 2),    # 1x1 on channel slices, N tile 256
    (2, 96, 14, 14, 128, 5, 2, 2, 160, 32, 160, 32, "nhwc", 1),   # 5x5 stride 2, K = 98 pixels
    (3, 256, 28, 28, 160, 1, 1, 0, 256, 0, 160, 0, "nchw", 4),    # unit 3a: ones row opens a third M tile
    (4, 320, 14, 14, 160, 1, 1, 0, 320, 0, 160, 0, "nchw", 1),    # 196 pixels per frame: 7 K-blocks, the last one partial
]


@PRECS
@pytest.mark.parametrize("ovec", [0, 2], ids=["red_scalar", "red_v4_rows"])
@pytest.mark.parametrize("bk", [0, 64, 128])
@pytest.mark.parametrize("case", WGRAD_CASES, ids=[f"{c[12]}{c[1]}x{c[2]}k{c[5]}s{c[6]}n{c[4]}" for c in WGRAD_CASES])
def test_tma_gemm_weight_gradient(dev, case, prec, tol, bk, ovec):
    """Weight + bias gradient GEMMs with both operands TMA-fed (OFFK_TMA_A_IM2COL_T / _NCHW_T x OFFK_TMA_B_DENSE_T,
    the ones row patched into the landed tile) against autograd of conv2d and against the gather-fed kernel."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, h, w, cout, k, st, p, xct, xco, yct, yco, xl, split = case
    stage = (2 if prec == 2 else 1) * ((bk or 32) * 512 + -(-min(cout, 256) // 32) * (bk or 32) * 128)
    if bk and (xl == "nchw" or stage > 108 * 1024):
        pytest.skip("deep K-blocks: channels-last operands only, and two pipeline stages must fit the SM")
    g = T.ConvGeom(n, cin, h, w, cout, k, k, st, p, xct, xco, yct, yco)
    torch.manual_seed(2)
    x = torch.randn(n, xct, h, w, device=dev)
    dy = torch.randn(n, yct, g.hout, g.wout, device=dev)
    xs = x[:, xco:xco + cin].double().requires_grad_(False)
    wt = torch.zeros(cout, cin, k, k, device=dev, dtype=torch.float64, requires_grad=True)
    y = torch.nn.functional.conv2d(xs, wt, torch.zeros(cout, device=dev, dtype=torch.float64), st, p)
    (y * dy[:, yco:yco + cout].double()).sum().backward()
    ref_w = wt.grad.permute(0, 2, 3, 1) if xl == "nhwc" else wt.grad          # OHWI for channels-last inputs
    ref_b = dy[:, yco:yco + cout].double().sum((0, 2, 3))
    xb = x.permute(0, 2, 3, 1).contiguous() if xl == "nhwc" else x
    dyb = dy.permute(0, 2, 3, 1).contiguous()
    spc = T.conv_wgrad_spec(g, xl, "nhwc")
    tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
    outs = []
    for use_tma in (True, False):
        dw = torch.zeros(cout, g.kdim, device=dev)
        db = torch.zeros(cout, device=dev)
        t = L.OffkTGemm()
        d = t.g
        d.M, d.N, d.K = spc.M, spc.N, spc.K
        d.a_src, d.a_row, d.a_col = xb.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
        d.a_h, d.a_w = (spc.a_h, spc.a_w) if spc.a_h else (T.NO_BOX, T.NO_BOX)
        d.a_ones_row, d.a_mode = spc.a_ones_row, spc.a_mode
        d.b_src, d.b_row, d.b_col, d.b_mode = dyb.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
        d.out, d.out_row, d.out_col = dw.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
        d.ones_row_out = db.data_ptr()
        d.split_k, d.atomic_out, d.out_vec = split, 1, ovec          # 2: rows of dW contiguous -> transposed float4 adds
        if use_tma:
            t.a_kind = L.TMA_A_NCHW_T if xl == "nchw" else L.TMA_A_IM2COL_T
            t.a_coff = xco
            t.n_img, t.hin, t.win, t.ctot, t.cin = n, h, w, xct, cin
            t.kh, t.kw, t.stride, t.pad, t.hout, t.wout = k, k, st, p, g.hout, g.wout
            t.b_kind, t.ldb, t.precision, t.bk = L.TMA_B_DENSE_T, yct, prec, bk
            d.b_src = dyb.data_ptr() + 4 * yco
            L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
            L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
        else:
            L.check(lib.offk_gather_gemm(C.byref(d), prec, None), "gather_gemm")
        torch.cuda.synchronize()
        outs.append((dw, db))
    (dw_t, db_t), (dw_g, db_g) = outs
    assert _rel(dw_t.view(ref_w.shape), ref_w.cpu()) < tol
    assert _rel(db_t, ref_b.cpu()) < tol
    assert _rel(dw_t, dw_g.cpu()) < 1e-4 and _rel(db_t, db_g.cpu()) < 1e-4      # same tf32 products, other summation order


SDGRAD_CASES = [
    # n, cin, h, w, cout, k, s, p, x_ctot, x_coff
    (3, 64, 28, 28, 64, 7, 2, 3, 64, 0),          # motion_conv_trans_28 geometry: classes with 3 or 4 taps per axis
    (4, 96, 14, 14, 128, 5, 2, 2, 128, 32),       # motion_conv_trans_14 geometry, dX into a channel slice
]


@PRECS
@pytest.mark.parametrize("case", SDGRAD_CASES, ids=[f"{c[1]}x{c[2]}k{c[5]}s{c[6]}" for c in SDGRAD_CASES])
def test_tma_gemm_strided_data_gradient(dev, case, prec, tol):
    """Data gradient of a stride-2 conv, one stride-parity class at a time, as a TMA-im2col stride-1 correlation over dY
    (OFFK_TGEMM_FREE_GEOM) against autograd of conv2d and bit-for-bit against the gather-fed kernel."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, h, w, cout, k, st, p, xct, xco = case
    g = T.ConvGeom(n, cin, h, w, cout, k, k, st, p, xct, xco)
    torch.manual_seed(3)
    x = torch.zeros(n, cin, h, w, device=dev, dtype=torch.float64, requires_grad=True)
    wt = torch.randn(cout, cin, k, k, device=dev) / (g.kdim ** 0.5)
    dy = torch.randn(n, cout, g.hout, g.wout, device=dev)
    (torch.nn.functional.conv2d(x, wt.double(), None, st, p) * dy.double()).sum().backward()
    dyb = dy.permute(0, 2, 3, 1).contiguous()
    w_ohwi = wt.permute(0, 2, 3, 1).contiguous()
    outs = []
    for use_tma in (True, False):
        dx = torch.zeros(n, h, w, xct, device=dev)
        for spc in T.conv_dgrad_specs(g, "nhwc", "nhwc", "nhwc"):
            ex = spc.extra
            tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
            t = L.OffkTGemm()
            d = t.g
            d.M, d.N, d.K = spc.M, spc.N, spc.K
            d.a_src, d.a_row, d.a_col = dyb.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
            d.a_h, d.a_w, d.a_ones_row, d.a_mode = spc.a_h, spc.a_w, -1, spc.a_mode
            d.b_src, d.b_row, d.b_col, d.b_mode = w_ohwi.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
            d.out, d.out_row, d.out_col = dx.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
            d.split_k, d.out_vec, d.tile_n = 1, spc.out_vec, 32
            if use_tma:
                rs, qs = ex["rs"][::-1].copy(), ex["qs"][::-1].copy()
                wsub = wt[:, :, torch.as_tensor(rs, device=dev)][:, :, :, torch.as_tensor(qs, device=dev)]
                wcls = wsub.permute(1, 2, 3, 0).contiguous()                   # [cin, R, Q, cout]
                t.a_kind, t.a_coff = L.TMA_A_IM2COL, 0
                t.n_img, t.hin, t.win, t.ctot, t.cin = n, g.hout, g.wout, cout, cout
                t.kh, t.kw, t.stride, t.pad, t.pad_w = len(rs), len(qs), 1, ex["pad_h"], ex["pad_w"]
                t.hout, t.wout, t.geom_flags = ex["hc"], ex["wc"], L.TGEMM_FREE_GEOM
                t.b_kind, t.ldb, t.precision = L.TMA_B_DENSE, len(rs) * len(qs) * cout, prec
                d.b_src = wcls.data_ptr()
                L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
                L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
            else:
                L.check(lib.offk_gather_gemm(C.byref(d), prec, None), "gather_gemm")
            torch.cuda.synchronize()
        outs.append(dx)
    got = outs[0].permute(0, 3, 1, 2)[:, xco:xco + cin]
    assert _rel(got, x.grad.cpu()) < tol
    assert _rel(outs[0], outs[1].cpu()) < 1e-5           # same products; the K order (tap walk) differs
    if xco:
        assert outs[0][..., :xco].abs().max().item() == 0


STENCIL_CASES = [
    # B, L, S, K, index_mode, drop_mode
    (2, 3, 28, 1, 0, 0), (3, 4, 14, 1, 1, 1), (2, 2, 7, 1, 0, 2), (2, 3, 7, 2, 0, 0), (1, 7, 14, 1, 0, 1), (1, 2, 5, 1, 1, 0),
]


@pytest.mark.parametrize("case", STENCIL_CASES, ids=[f"B{c[0]}L{c[1]}S{c[2]}K{c[3]}m{c[4]}d{c[5]}" for c in STENCIL_CASES])
def test_stencil_diff_fwd_bwd(dev, case):
    """Fused stencil (RGB_OFF.py:599-616): spatial gradient + temporal difference + dropout + cat, and its backward."""
    from off_b200 import _lib as L
    lib = L.lib()
    B, Lg, S, K, mode, drop = case
    N, P, Cg, Cs = B * Lg, B * (Lg - 1), 128, 32
    torch.manual_seed(1)
    gd_c = torch.randn(N, Cg + Cs, S, S, device=dev)
    gd_c[:, :Cg].relu_()
    gd = gd_c.permute(0, 2, 3, 1).contiguous()
    w = torch.randn(Cs, K, 3, 3, device=dev)
    bias = torch.randn(Cs * K, device=dev)
    ctot, coff = 400, 64
    out_l = torch.zeros(P, S, S, ctot, device=dev)
    sd = L.OffkStencil()
    sd.B, sd.L, sd.Cg, sd.Cs, sd.K, sd.H, sd.W = B, Lg, Cg, Cs, K, S, S
    sd.g_fs = sd.d_fs = (Cg + Cs) * S * S
    sd.g_ps = sd.d_ps = Cg + Cs
    sd.out_ctot, sd.out_coff, sd.index_mode = ctot, coff, mode
    sd.drop_mode, sd.keep_scale, sd.drop_p, sd.seed = drop, 5.0, 0.8, 1234
    mask = (torch.rand(P, K * Cs, S, S, device=dev) > 0.8).to(torch.uint8)
    sd.keep_mask = mask.data_ptr()
    L.check(lib.offk_stencil_diff_fwd(C.byref(sd), gd.data_ptr(), gd.data_ptr() + 4 * Cg, w.data_ptr(), bias.data_ptr(),
                                      out_l.data_ptr(), None), "fwd")
    torch.cuda.synchronize()
    out = out_l.permute(0, 3, 1, 2)
    G, D = gd_c[:, :Cg].double(), gd_c[:, Cg:].double()
    Gv = G.view(B, Lg, Cg, S, S)
    Tref = (Gv[:, 1:] - Gv[:, :-1]).reshape(P, Cg, S, S)
    Ds = (D[:P] if mode == 0 else D.view(B, Lg, Cs, S, S)[:, :-1].reshape(P, Cs, S, S)).clone().requires_grad_(True)
    wd, bd = w.double().clone().requires_grad_(True), bias.double().clone().requires_grad_(True)
    Sg = torch.nn.functional.conv2d(Ds.repeat(1, K, 1, 1), wd.permute(1, 0, 2, 3).reshape(K * Cs, 1, 3, 3), bd, 1, 1, 1, K * Cs)
    if drop == 1:
        keep = mask.double() * 5.0
    elif drop == 2:      # counter-hash dropout: regenerate on the host with the library's own hash (host mirror)
        # element index = channels-last ((p*HW + pix)*K*Cs + ch); 4 consecutive elements share one hash
        n_el = P * K * Cs * S * S
        k16 = np.array([lib.offk_drop_keep_host(1234, i, 0.8) for i in range(n_el)], dtype=np.float64)
        assert 0.15 < k16.mean() < 0.25
        keep = torch.from_numpy(k16).to(dev).view(P, S, S, K * Cs).permute(0, 3, 1, 2) * 5.0
    else:
        keep = torch.ones(P, K * Cs, S, S, device=dev, dtype=torch.float64)
    Sg = Sg * keep
    ref = torch.cat([Sg, Tref], 1)
    assert (out[:, coff:coff + K * Cs + Cg].double() - ref.detach()).abs().max().item() < 2e-5
    assert out[:, :coff].abs().max().item() == 0 and out[:, coff + K * Cs + Cg:].abs().max().item() == 0
    # temporal rows are exact fp32 differences: bit-exact against torch on the GPU
    Gf = gd_c[:, :Cg].view(B, Lg, Cg, S, S)
    assert torch.equal(out[:, coff + K * Cs:coff + K * Cs + Cg], (Gf[:, 1:] - Gf[:, :-1]).reshape(P, Cg, S, S))
    # telescoping: sum_t T[b,t] == G[b,L-1] - G[b,0]
    tel = out[:, coff + K * Cs:coff + K * Cs + Cg].reshape(B, Lg - 1, Cg, S, S).double().sum(1)
    assert (tel - (Gv[:, -1] - Gv[:, 0])).abs().max().item() < 1e-5

    dout_l = torch.randn(P, S, S, ctot, device=dev)
    dout = dout_l.permute(0, 3, 1, 2)
    dgd_l = torch.full((N, S, S, Cg + Cs), float("nan"), device=dev)
    dw, dbias = torch.zeros_like(w), torch.zeros_like(bias)
    fs = (Cg + Cs) * S * S
    L.check(lib.offk_stencil_diff_bwd(C.byref(sd), dout_l.data_ptr(), gd.data_ptr(), gd.data_ptr() + 4 * Cg, w.data_ptr(),
                                      dgd_l.data_ptr(), fs, dgd_l.data_ptr() + 4 * Cg, fs, dw.data_ptr(), dbias.data_ptr(),
                                      None), "bwd")
    torch.cuda.synchronize()
    dgd = dgd_l.permute(0, 3, 1, 2)
    assert not torch.isnan(dgd).any()
    dT = dout[:, coff + K * Cs:coff + K * Cs + Cg].double().reshape(B, Lg - 1, Cg, S, S)
    dG = torch.zeros(B, Lg, Cg, S, S, device=dev, dtype=torch.float64)
    dG[:, 1:] += dT
    dG[:, :-1] -= dT
    dG = dG.view(N, Cg, S, S) * (G > 0)
    Sg.backward(dout[:, coff:coff + K * Cs].double())
    dD = torch.zeros(N, Cs, S, S, device=dev, dtype=torch.float64)
    if mode == 0:
        dD[:P] = Ds.grad
    else:
        dD.view(B, Lg, Cs, S, S)[:, :-1] = Ds.grad.view(B, Lg - 1, Cs, S, S)
    assert (dgd[:, :Cg].double() - dG).abs().max().item() < 1e-5
    assert (dgd[:, Cg:].double() - dD).abs().max().item() < 5e-5
    assert _rel(dw, wd.grad.cpu()) < 1e-5 and _rel(dbias, bd.grad.cpu()) < 1e-5


def test_stencil_batch_equals_single_launches(dev):
    """offk_stencil_diff_fwd_batch / _bwd_batch (one launch for several OFF units) write exactly what the per-unit
    calls write: same arithmetic per element, only the block -> work mapping differs."""
    from off_b200 import _lib as L
    lib = L.lib()
    B, Lg, Cg, Cs = 3, 4, 128, 32
    N, P = B * Lg, B * (Lg - 1)
    torch.manual_seed(3)
    geoms = [(14, 480, 0), (14, 480, 160), (14, 480, 320)]
    n = len(geoms)
    descs, ios = (L.OffkStencil * n)(), (L.OffkStencilIO * n)()
    keep = []
    F_b, F_s = torch.zeros(P, 14, 14, 480, device=dev), torch.zeros(P, 14, 14, 480, device=dev)
    dF = torch.randn(P, 14, 14, 480, device=dev)
    for i, (S, ctot, coff) in enumerate(geoms):
        gd = torch.randn(N, S, S, Cg + Cs, device=dev)
        gd[..., :Cg].relu_()
        w, bias = torch.randn(Cs, 1, 3, 3, device=dev), torch.randn(Cs, device=dev)
        bufs = {k: (torch.full_like(gd, float("nan")), torch.zeros_like(w), torch.zeros_like(bias)) for k in "bs"}
        sd = descs[i]
        sd.B, sd.L, sd.Cg, sd.Cs, sd.K, sd.H, sd.W = B, Lg, Cg, Cs, 1, S, S
        sd.g_fs = sd.d_fs = (Cg + Cs) * S * S
        sd.g_ps = sd.d_ps = Cg + Cs
        sd.out_ctot, sd.out_coff, sd.index_mode = ctot, coff, i % 2
        sd.drop_mode, sd.keep_scale, sd.drop_p, sd.seed = 2, 5.0, 0.8, 40 + i
        io = ios[i]
        io.g, io.d, io.w, io.bias = gd.data_ptr(), gd.data_ptr() + 4 * Cg, w.data_ptr(), bias.data_ptr()
        io.out, io.dout = F_b.data_ptr(), dF.data_ptr()
        dgd, dw, db = bufs["b"]
        io.dg, io.dd, io.dg_fs, io.dd_fs = dgd.data_ptr(), dgd.data_ptr() + 4 * Cg, sd.g_fs, sd.g_fs
        io.dw, io.dbias = dw.data_ptr(), db.data_ptr()
        keep.append((gd, w, bias, bufs))
    L.check(lib.offk_stencil_diff_fwd_batch(n, descs, ios, None), "fwd_batch")
    L.check(lib.offk_stencil_diff_bwd_batch(n, descs, ios, None), "bwd_batch")
    for i in range(n):
        gd, w, bias, bufs = keep[i]
        dgd, dw, db = bufs["s"]
        L.check(lib.offk_stencil_diff_fwd(C.byref(descs[i]), ios[i].g, ios[i].d, ios[i].w, ios[i].bias, F_s.data_ptr(), None), "fwd")
        L.check(lib.offk_stencil_diff_bwd(C.byref(descs[i]), dF.data_ptr(), ios[i].g, ios[i].d, ios[i].w, dgd.data_ptr(),
                                          descs[i].g_fs, dgd.data_ptr() + 4 * Cg, descs[i].g_fs, dw.data_ptr(), db.data_ptr(),
                                          None), "bwd")
    torch.cuda.synchronize()
    assert torch.equal(F_b, F_s) and F_b.abs().sum().item() > 0
    for gd, w, bias, bufs in keep:
        assert torch.equal(bufs["b"][0], bufs["s"][0])                                   # dG, dD: bit-exact
        assert _rel(bufs["b"][1], bufs["s"][1].cpu()) < 1e-5 and _rel(bufs["b"][2], bufs["s"][2].cpu()) < 1e-5  # atomics: order


def test_layout_helpers(dev):
    """offk_nchw_to_nhwc (the 7x7 tap copy) and offk_permute_weight_batch (all KxK weight-gradient un-permutes in one
    launch) against torch permutes: pure data movement, bit-exact."""
    from off_b200 import _lib as L
    lib = L.lib()
    torch.manual_seed(5)
    for n, c, hw in ((5, 1024, 49), (3, 70, 36), (2, 33, 1)):
        x = torch.randn(n, c, hw, device=dev)
        y = torch.full((n, hw, c), float("nan"), device=dev)
        L.check(lib.offk_nchw_to_nhwc(x.data_ptr(), y.data_ptr(), n, c, hw, None), "nchw_to_nhwc")
        torch.cuda.synchronize()
        assert torch.equal(y, x.permute(0, 2, 1).contiguous())
    shapes = [(64, 320, 7), (128, 96, 5), (40, 33, 3), (16, 64, 1)]
    items = (L.OffkPermute * len(shapes))()
    keep = []
    for it, (co, ci, k) in zip(items, shapes):
        src = torch.randn(co, k, k, ci, device=dev)                 # OHWI accumulator
        dst = torch.randn(co, ci, k, k, device=dev)                 # OIHW gradient, accumulated into
        want = dst + src.permute(0, 3, 1, 2)
        it.src, it.dst, it.cout, it.cin, it.kh, it.kw = src.data_ptr(), dst.data_ptr(), co, ci, k, k
        keep.append((src, dst, want))
    L.check(lib.offk_permute_weight_batch(len(shapes), items, 2, None), "permute_weight_batch")
    torch.cuda.synchronize()
    for src, dst, want in keep:
        assert torch.equal(dst, want)


import functools

# ---- tolerances of the whole-section comparisons: (stage-fusion tensors, logits: max-abs / tensor max; gradients: worst
# relative L2 over the parameters).
# fp32 mode vs the fp64 oracle.  Forward: fp32 level.  Gradients against the oracle's OWN ReLU gates are dominated by
# gate flips, not arithmetic: an element whose pre-activation sits within round-off of zero takes either sign, and each
# flipped gate moves a weight gradient by O(1/sqrt(#elements)).  The reference's own fp32 CPU arithmetic shows the same
# against fp64 (B=1, L=3: worst relative L2 1.4e-2; 1.8e-6 once the gates are matched -- measured with oracle/off_oracle.py),
# so the exact-oracle gate only bounds the flip rate and the arithmetic is pinned by the gate-matched run.
# Measured on the B200 (profiles/parity_r02b.txt): fp32 mode forward 4e-7 .. 2.5e-6, gate-matched gradients 3.5e-6 .. 5.1e-6,
# exact-oracle gradients 3.5e-6 (no flip) .. 3.7e-3 (B = 48).
TOL_FP32 = (5e-6, 1e-5, 5e-2)
TOL_FP32_GATED = (5e-6, 1e-5, 2e-5)


@functools.lru_cache(maxsize=2)
def _taps_cached(seed, B, Lg):
    return O.make_taps(seed, B, Lg)


@functools.lru_cache(maxsize=4)
def _oracle_cached(variant, B, Lg, train, mm):
    """fp64 oracle forward+backward for the seeded case (cached: several precision modes compare against one run).
    mm='tf32_trunc': every contraction consumes operands truncated to tf32 like tcgen05 kind::tf32 does."""
    seed = 5
    taps, prm = _taps_cached(seed, B, Lg), O.make_params(seed, variant)
    masks = O.make_dropout_masks(seed, B, Lg) if train else None
    n_out = B * (Lg - 1) if variant == "rgb" else B
    r7, r14 = O.hash_normal(77, (n_out, 101)).double(), O.hash_normal(78, (n_out, 101)).double()
    lossf = lambda o: (o["fc7"].reshape(r7.shape) * r7).sum() + (o["fc14"].reshape(r14.shape) * r14).sum()
    ref, gref = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float64, loss=lossf, mm=mm)
    keep = {k: ref[k] for k in ("fusion28", "fusion14", "fusion7", "fc7", "fc28", "fc14")}
    return taps, prm, masks, r7, r14, keep, gref


from helpers import engine_gates as _engine_gates  # noqa: E402


def _engine_vs_oracle(dev, precision, variant, B, Lg, train, tol_fuse, tol_logit, tol_grad, mm="exact", gate_matched=False):
    """gate_matched: the oracle is re-run with the ENGINE's ReLU sign patterns (off_oracle._act), so that the gradient
    comparison measures arithmetic only -- a pre-activation within round-off of zero may take either sign, and one
    flipped gate moves a weight gradient by ~1/sqrt(#elements) in relative L2, far above fp32 round-off."""
    from off_b200 import engine as E
    taps, prm, masks, r7, r14, ref, gref = _oracle_cached(variant, B, Lg, train, mm)
    eng = E.OFFEngine(B, Lg, variant, dev, precision)
    eng.load_params(prm)
    fc7, fc28, fc14 = eng.forward({k: v.to(dev) for k, v in taps.items()}, train=train, masks=masks)
    torch.cuda.synchronize()
    if gate_matched:
        lossf = lambda o: (o["fc7"].reshape(r7.shape) * r7).sum() + (o["fc14"].reshape(r14.shape) * r14).sum()
        ref, gref = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float64, loss=lossf, mm=mm,
                                           gates=_engine_gates(eng))
    report, bad = {}, []
    for k, st in (("fusion28", "F28"), ("fusion14", "F14"), ("fusion7", "F7")):      # per-level error (channels-last -> NCHW)
        report[k] = _rel(eng.buf[st].permute(0, 3, 1, 2), ref[k])
        if not report[k] < tol_fuse:
            bad.append((k, report[k], tol_fuse))
    for name, got in (("fc7", fc7), ("fc28", fc28), ("fc14", fc14)):
        report[name] = _rel(got, ref[name].reshape(got.shape))
        if not report[name] < tol_logit:
            bad.append((name, report[name], tol_logit))
    grads = eng.backward(r7.float().to(dev), r14.float().to(dev))
    torch.cuda.synchronize()
    worst, worst_name = 0.0, ""
    for n, g in grads.items():
        if gref[n].abs().max().item() == 0:
            if g.abs().max().item() != 0:
                bad.append((n, "expected an all-zero gradient", 0))   # fc_action_motion_28.* never gets a gradient
            continue
        e = _rel_l2(g, gref[n])
        if e > worst:
            worst, worst_name = e, n
    if not worst < tol_grad:
        bad.append(("grad " + worst_name, worst, tol_grad))
    print(f"[parity {precision} vs {mm}{'+gates' if gate_matched else ''} oracle, {variant} B{B} L{Lg} train={train}] " +
          " ".join(f"{k}={v:.2e}" for k, v in report.items()) + f" grad_rel_l2_worst={worst:.2e} ({worst_name})")
    assert not bad, bad
    return report, worst


@pytest.mark.parametrize("variant,B,Lg,train", [("rgb", 2, 3, False), ("flow", 2, 3, False), ("rgb", 2, 2, True),
                                                ("flow", 1, 4, False), ("rgb", 1, 3, False),
                                                ("rgb", 2, 7, False), ("flow", 1, 7, True),   # config 4 geometry: 7 segments
                                                ("flow", 1, 4, True)])
def test_engine_fp32_mode_matches_oracle(dev, variant, B, Lg, train):
    """precision='fp32' = the fp32-parity mode on the tensor cores (3xTF32 tcgen05, OFFK_PREC_TF32X3)."""
    _engine_vs_oracle(dev, "fp32", variant, B, Lg, train, *TOL_FP32)
    _engine_vs_oracle(dev, "fp32", variant, B, Lg, train, *TOL_FP32_GATED, gate_matched=True)


TF32_CASES = [("rgb", 2, 3, False), ("flow", 2, 3, False), ("rgb", 2, 2, True), ("rgb", 2, 7, True)]


@pytest.mark.parametrize("variant,B,Lg,train", TF32_CASES)
def test_engine_tf32_mode_matches_oracle(dev, variant, B, Lg, train):
    """tf32 mode against the EXACT oracle: the stated tf32 tolerance (operand truncation to 10 mantissa bits)."""
    _engine_vs_oracle(dev, "tf32", variant, B, Lg, train, 5e-3, 1e-2, 0.2)


# tf32 mode against an oracle whose contractions consume tf32-TRUNCATED operands (oracle mm='tf32_trunc'): what is left
# is fp32 accumulation order plus the rare operand whose fp32 value (GPU) and fp64 value (oracle) straddle a tf32
# truncation boundary.  This pins the tensor-core path itself: a wrong tap, stride-parity class or table entry moves a
# gradient by O(1), two orders of magnitude above these gates.
# Measured (profiles/parity_r02b.txt): stage-fusion tensors 7e-7 (first stage: accumulation order only) .. 5.4e-5, logits
# <= 1.6e-4, gradients 5e-4 .. 1.1e-3 -- against 8e-4 / 2e-3 / 6e-2 for the same mode vs the exact oracle.
TOL_TF32_EMU = (2e-4, 5e-4, 3e-3)      # + the oracle follows the engine's ReLU gates (gate_matched)


@pytest.mark.parametrize("variant,B,Lg,train", TF32_CASES)
def test_engine_tf32_mode_matches_truncated_operand_oracle(dev, variant, B, Lg, train):
    _engine_vs_oracle(dev, "tf32", variant, B, Lg, train, *TOL_TF32_EMU, mm="tf32_trunc", gate_matched=True)


# BASELINE.json's own shapes (config 2: RGB 48 x 3, config 3: Flow 48 x 3, config 4 per GPU at 8 ranks: RGB 16 x 7):
# split-K factors, N tiles and grids depend on the batch, so the plans that bench.py times are checked here, in both
# precision modes, against the fp64 oracle (and the tf32 mode against the truncated-operand oracle as well).
BENCH_SHAPES = [("rgb", 48, 3, True), ("flow", 48, 3, False), ("rgb", 16, 7, False)]


@pytest.mark.parametrize("variant,B,Lg,train", BENCH_SHAPES, ids=["cfg2_rgb48x3_train", "cfg3_flow48x3", "cfg4_rgb16x7"])
def test_benchmark_shapes_match_oracle(dev, variant, B, Lg, train):
    _engine_vs_oracle(dev, "fp32", variant, B, Lg, train, *TOL_FP32)
    _engine_vs_oracle(dev, "fp32", variant, B, Lg, train, *TOL_FP32_GATED, gate_matched=True)
    _engine_vs_oracle(dev, "tf32", variant, B, Lg, train, 5e-3, 1e-2, 0.2)
    _engine_vs_oracle(dev, "tf32", variant, B, Lg, train, *TOL_TF32_EMU, mm="tf32_trunc", gate_matched=True)


@pytest.mark.parametrize("name", ["rgb_b1_l3", "rgb_b2_l3", "flow_b2_l3", "rgb_b2_l2_train", "flow_b1_l4", "v2_b2_l3", "rgb_b1_l2"])
def test_module_matches_reference_golden(dev, name):
    """The nn.Module surface against vectors produced by the reference itself (tests/golden, make_golden.py)."""
    from off_b200.modules import OFFSubNetwork
    fix = np.load(os.path.join(GOLD, f"off_{name}.npz"))
    variant, B, Lg, seed, train = str(fix["variant"]), int(fix["batch"]), int(fix["length"]), int(fix["seed"]), int(fix["train"])
    variant = "rgb" if variant == "rgb" else "flow"         # RGB_OFF_v2 runs Flow_OFF's OFF graph (fixed diagonal Sobel + consensus)
    net = OFFSubNetwork(B, Lg, variant, precision="fp32", device=dev)
    net.train(bool(train))
    net.load_state_dict(O.make_params(seed, variant), strict=(variant == "rgb"))
    masks = O.make_dropout_masks(seed, B, Lg) if train else None
    fc7, fc28, fc14 = net({k: v.to(dev) for k, v in O.make_taps(seed, B, Lg).items()}, masks=masks)
    for k, got in (("fc7", fc7), ("fc28", fc28), ("fc14", fc14)):
        want = torch.from_numpy(fix[k]).reshape(got.shape)
        assert _rel(got, want) < 1e-5, k
    (fc7.sum() + fc14.sum()).backward()
    for n, p in net.named_parameters():
        if not p.requires_grad:
            continue
        l2 = float(fix[f"grad.{n}.l2"])
        if l2 == 0:
            assert p.grad is None or p.grad.abs().max().item() == 0
            continue
        idx, val = torch.from_numpy(fix[f"grad.{n}.idx"]), torch.from_numpy(fix[f"grad.{n}.val"])
        got = p.grad.reshape(-1)[idx.to(dev)].double().cpu()
        # gradients: flip-level tolerance (TOL_FP32 above says why); the arithmetic itself is pinned by the gate-matched
        # oracle tests, the fixture pins that the oracle is the reference
        assert abs(p.grad.double().norm().item() - l2) / l2 < 5e-2, n
        assert (got - val).norm().item() <= 5e-2 * max(val.norm().item(), 1e-2 * l2), n


@pytest.mark.parametrize("P,C,T,drop,acc", [(6, 1024, 1, 0, False), (8, 512, 2, 1, True), (6, 256, 3, 2, False), (1, 512, 1, 0, True)])
def test_fused_head_fwd_bwd(dev, P, C, T, drop, acc):
    """offk_head_fwd / offk_head_bwd (SURVEY K6): global_pool -> dropout -> Linear (-> consensus over T pairs) in one launch and
    its backward (Linear', dropout', avg-pool', producer ReLU', accumulation into a channel slice) against torch in fp64.
    RGB_OFF.py:784-793,844-847; Flow_OFF.py:867-876; basic_ops.py:21-31."""
    from off_b200 import _lib as L
    lib = L.lib()
    torch.manual_seed(7)
    HW, NC, ctot, coff = 49, 101, C + 64, 32
    x = torch.randn(P, HW, ctot, device=dev)
    W, b = torch.randn(NC, C, device=dev) / C ** 0.5, torch.randn(NC, device=dev)
    seed = 1234
    if drop == 1:
        keep = (torch.rand(P, C, device=dev) >= 0.8).to(torch.uint8)
    elif drop == 2:
        keep = torch.tensor([lib.offk_drop_keep_host(seed, i, 0.8) for i in range(P * C)], dtype=torch.uint8, device=dev).view(P, C)
    else:
        keep = torch.ones(P, C, dtype=torch.uint8, device=dev)
    scale = 5.0 if drop else 1.0
    pooled = torch.zeros(P, C, device=dev)
    out = torch.zeros(P, NC, device=dev)
    cons = torch.zeros(P // T, NC, device=dev) if T > 1 else None
    mask_ptr = keep.data_ptr() if drop == 1 else None
    L.check(lib.offk_head_fwd(x.data_ptr(), P, C, HW, ctot, coff, drop, mask_ptr, seed, None, 0.8, scale, W.data_ptr(), b.data_ptr(),
                              NC, T, pooled.data_ptr(), out.data_ptr(), cons.data_ptr() if cons is not None else None, None), "head_fwd")
    xs = x[..., coff:coff + C].double().requires_grad_(True)
    Wd, bd = W.double().requires_grad_(True), b.double().requires_grad_(True)
    pr = xs.mean(1) * keep.double() * scale
    o = pr @ Wd.t() + bd
    final = o.view(P // T, T, NC).mean(1) if T > 1 else o
    assert _rel(pooled, pr.detach().cpu()) < 2e-6 and _rel(out, o.detach().cpu()) < 2e-6
    if T > 1:
        assert _rel(cons, final.detach().cpu()) < 2e-6
    dout = torch.randn(P // T, NC, device=dev)
    final.backward(dout.double())
    act = torch.randn(P, HW, ctot, device=dev)
    dx0 = torch.randn(P, HW, ctot, device=dev)
    dx = dx0.clone()
    dW, db = torch.zeros_like(W), torch.zeros_like(b)
    L.check(lib.offk_head_bwd(dout.data_ptr(), P, C, HW, ctot, coff, drop, mask_ptr, seed, None, 0.8, scale, W.data_ptr(), NC, T,
                              pooled.data_ptr(), act.data_ptr() if acc else None, int(acc), dx.data_ptr(), dW.data_ptr(),
                              db.data_ptr(), None), "head_bwd")
    torch.cuda.synchronize()
    assert _rel(dW, Wd.grad.cpu()) < 5e-6 and _rel(db, bd.grad.cpu()) < 5e-6
    want = xs.grad
    if acc:
        want = (want + dx0[..., coff:coff + C].double()) * (act[..., coff:coff + C] > 0)
    assert _rel(dx[..., coff:coff + C], want.cpu()) < 5e-6
    assert torch.equal(dx[..., :coff], dx0[..., :coff]) and torch.equal(dx[..., coff + C:], dx0[..., coff + C:])   # slice only


@PRECS
@pytest.mark.parametrize("split,with_aux", [(4, True), (3, False), (1, True)])
def test_tma_gemm_split_k_finisher_and_second_output(dev, prec, tol, split, with_aux):
    """offk_tma_gemm split-K finished in-kernel (finish_counter: the last CTA of a tile applies bias + ReLU in place) and the
    epilogue's second output aux_out = relu(v + aux_addend) in another tensor layout; launched twice on the same counters
    (they must be left at zero).  Against conv2d + the element-wise ops in fp64."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, h, cout, k = 3, 128, 7, 256, 3
    g = T.ConvGeom(n, cin, h, h, cout, k, k, 1, 1)
    torch.manual_seed(4)
    x = torch.randn(n, h, h, cin, device=dev)
    wt = torch.randn(cout, cin, k, k, device=dev) / (g.kdim ** 0.5)
    wl = wt.permute(0, 2, 3, 1).contiguous()
    bias = torch.randn(cout, device=dev)
    addend = torch.randn(n, h, h, cout, device=dev)
    spc = T.conv_fwd_spec(g, "nhwc", "nhwc")
    tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
    gaux = T.ConvGeom(n, cout, h, h, cout, y_ctot=cout + 96, y_coff=64)           # aux lands in a channel slice of a wider tensor
    aux_row = torch.from_numpy(T.padded_tables(T.conv_fwd_spec(gaux, "nhwc", "nhwc"))["out_row"]).to(dev)
    out = torch.zeros(n, h, h, cout, device=dev)
    aux = torch.zeros(n, h, h, cout + 96, device=dev)
    counter = torch.zeros(64, dtype=torch.int32, device=dev)
    t = L.OffkTGemm()
    d = t.g
    d.M, d.N, d.K = spc.M, spc.N, spc.K
    d.a_src, d.b_src = x.data_ptr(), wl.data_ptr()
    d.a_ones_row = -1
    d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
    d.bias, d.relu_pre_cols, d.split_k, d.out_vec = bias.data_ptr(), cout, split, 1
    if split > 1:
        d.finish_counter = counter.data_ptr()
    if with_aux:
        # the row table of a channel-slice geometry carries the slice offset (64)
        d.aux_out, d.aux_row, d.aux_addend = aux.data_ptr(), aux_row.data_ptr(), addend.data_ptr()
    t.a_kind = L.TMA_A_IM2COL
    t.n_img, t.hin, t.win, t.ctot, t.cin = n, h, h, cin, cin
    t.kh, t.kw, t.stride, t.pad, t.hout, t.wout = k, k, 1, 1, h, h
    t.b_kind, t.ldb, t.precision = L.TMA_B_DENSE, g.kdim, prec
    L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
    ref = torch.relu(torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).double(), wt.double(), bias.double(), 1, 1)).permute(0, 2, 3, 1)
    for rep_ in range(2):
        out.zero_()
        aux.fill_(-7.0)
        L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
        torch.cuda.synchronize()
        assert _rel(out, ref.cpu()) < tol, rep_
        assert counter.abs().max().item() == 0
        if with_aux:
            want = torch.relu(ref + addend.double())
            assert _rel(aux[..., 64:64 + cout], want.cpu()) < tol
            assert (aux[..., :64] == -7.0).all() and (aux[..., 64 + cout:] == -7.0).all()


@pytest.mark.parametrize("k,split", [(1, 1), (3, 1), (3, 4)])
def test_tma_gemm_presplit_weights_equal_in_kernel_split(dev, k, split):
    """3xTF32 with the weight residuals produced ahead of the GEMM (offk_tf32_residual + offk_tgemm_t.b_lo_delta: both weight
    tiles arrive by TMA) performs the very same MMAs on the very same operand bits as the in-kernel split: bit-identical."""
    from off_b200 import _lib as L, tables as T
    lib = L.lib()
    n, cin, h, cout = 3, 64, 14, 256
    g = T.ConvGeom(n, cin, h, h, cout, k, k, 1, k // 2)
    torch.manual_seed(8)
    x = torch.randn(n, h, h, cin, device=dev)
    nw = cout * g.kdim
    wall = torch.zeros(2 * nw, device=dev)                       # [weights | their tf32 residuals]
    wall[:nw] = (torch.randn(cout, g.kdim, device=dev) / g.kdim ** 0.5).flatten()
    L.check(lib.offk_tf32_residual(wall.data_ptr(), wall.data_ptr() + 4 * nw, nw, None), "residual")
    w = wall[:nw].view(cout, g.kdim)
    hi = (w.view(torch.int32) & -8192).view(torch.float32)
    assert (wall[nw:].view(cout, g.kdim) - (w - hi)).abs().max().item() <= 2.0 ** -11 * (w - hi).abs().max().item()
    bias = torch.randn(cout, device=dev)
    spc = T.conv_fwd_spec(g, "nhwc", "nhwc")
    tabs = {kk: torch.from_numpy(v).to(dev) for kk, v in T.padded_tables(spc).items()}
    outs = []
    for delta in (0, nw):
        out = torch.zeros(n, h, h, cout, device=dev)
        t = L.OffkTGemm()
        d = t.g
        d.M, d.N, d.K = spc.M, spc.N, spc.K
        d.a_src, d.b_src, d.a_ones_row = x.data_ptr(), wall.data_ptr(), -1
        d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
        d.bias, d.split_k, d.out_vec = (bias.data_ptr() if split == 1 else None), split, 1
        one = k == 1
        t.a_kind, t.lda = (L.TMA_A_DENSE if one else L.TMA_A_IM2COL), cin
        t.n_img, t.hin, t.win, t.ctot, t.cin = n, h, h, cin, cin
        t.kh, t.kw, t.stride, t.pad, t.hout, t.wout = k, k, 1, k // 2, h, h
        t.b_kind, t.ldb, t.precision, t.b_lo_delta = L.TMA_B_DENSE, g.kdim, 2, delta
        L.check(lib.offk_tma_gemm_prepare(C.byref(t)), "prepare")
        L.check(lib.offk_tma_gemm(C.byref(t), None), "tma_gemm")
        torch.cuda.synchronize()
        outs.append(out)
    if split == 1:
        assert torch.equal(outs[0], outs[1])
    else:
        assert _rel(outs[0], outs[1].cpu()) < 1e-6               # split-K partial tiles meet through fp32 atomics
    wd = w.view(cout, k, k, cin).permute(0, 3, 1, 2).double()
    ref = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).double(), wd, bias.double() if split == 1 else None, 1, k // 2)
    assert _rel(outs[1].permute(0, 3, 1, 2), ref.cpu()) < 1e-5
