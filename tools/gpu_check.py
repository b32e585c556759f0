"""Developer harness run on the GPU box: isolates kernel families and prints error tables.
    python tools/gpu_check.py [gemm_tc] [stencil] [engine_fp32] [engine_tf32] ...
Not a test (tests/ holds those); this prints per-case diagnostics for bring-up."""
import ctypes as C
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import off_b200  # noqa
from off_b200 import _lib as L, tables as T, engine as E
import off_oracle as O

dev = torch.device("cuda")


def run_spec(spc, a_src, b_src, out_shape, prec, bias=None, ones=None, split_k=1, atomic=False, tile_n=0):
    lib = L.lib()
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
    d.split_k, d.atomic_out, d.tile_n, d.out_vec = split_k, int(atomic), tile_n, spc.out_vec
    T.check_modes(spc)
    L.check(lib.offk_gather_gemm(C.byref(d), prec, None), "gemm")
    torch.cuda.synchronize()
    return out


def gemm_cases():
    return [
        ("1x1 tiny", T.ConvGeom(3, 8, 7, 7, 5)),
        ("1x1 unit-like", T.ConvGeom(6, 256, 28, 28, 160)),
        ("1x1 7x7 C1024", T.ConvGeom(6, 1024, 7, 7, 160)),
        ("3x3 p1", T.ConvGeom(4, 64, 14, 14, 64, 3, 3, 1, 1)),
        ("7x7 s2", T.ConvGeom(2, 32, 28, 28, 64, 7, 7, 2, 3)),
        ("5x5 s2 slice", T.ConvGeom(2, 24, 14, 14, 128, 5, 5, 2, 2, 40, 8, 128, 0)),
        ("fc", T.ConvGeom(8, 1024, 1, 1, 101)),
        ("1x1 N=1024", T.ConvGeom(4, 256, 7, 7, 1024)),
    ]


def check_gemm(prec, label):
    torch.manual_seed(0)
    worst = 0.0
    nhwc_cases = [
        ("1x1 unit-like", T.ConvGeom(6, 256, 28, 28, 160)),
        ("1x1 7x7 C1024", T.ConvGeom(6, 1024, 7, 7, 160)),
        ("3x3 p1", T.ConvGeom(4, 64, 14, 14, 64, 3, 3, 1, 1)),
        ("7x7 s2", T.ConvGeom(2, 32, 28, 28, 64, 7, 7, 2, 3)),
        ("5x5 s2 slice", T.ConvGeom(2, 24, 14, 14, 128, 5, 5, 2, 2, 40, 8, 160, 32)),
        ("fc", T.ConvGeom(8, 1024, 1, 1, 101)),
        ("1x1 N=1024", T.ConvGeom(4, 256, 7, 7, 1024)),
        ("3x3 N=512", T.ConvGeom(3, 128, 7, 7, 512, 3, 3, 1, 1)),
    ]
    runs = [(n, g, "nchw", "nchw") for n, g in gemm_cases()] + [(n, g, "nhwc", "nhwc") for n, g in nhwc_cases] + \
           [(n, g, "nchw", "nhwc") for n, g in nhwc_cases[:2]]
    to = lambda a, lay: a.permute(0, 2, 3, 1).contiguous() if lay == "nhwc" else a
    back = lambda a, lay: a.permute(0, 3, 1, 2) if lay == "nhwc" else a
    for name, g, xl, yl in runs:
        x = torch.randn(g.n_img, g.x_ctot, g.hin, g.win, device=dev)
        w = torch.randn(g.cout, g.cin, g.kh, g.kw, device=dev) / (g.kdim ** 0.5)
        b = torch.randn(g.cout, device=dev)
        dy = torch.randn(g.n_img, g.y_ctot, g.hout, g.wout, device=dev)
        xs = x[:, g.x_coff:g.x_coff + g.cin].double().requires_grad_(True)
        wd = w.double().requires_grad_(True)
        y = torch.nn.functional.conv2d(xs, wd, b.double(), g.stride, g.pad)
        y.backward(dy[:, g.y_coff:g.y_coff + g.cout].double())
        xb, dyb = to(x, xl), to(dy, yl)
        wl = w.permute(0, 2, 3, 1).contiguous() if xl == "nhwc" else w
        oshape = tuple(dyb.shape)
        t0 = time.time()
        launchable = lambda spc: spc.a_mode is not None and spc.b_mode is not None
        e_f = e_s = e_w = e_b = e_d = float("nan")                 # nan: the layout has no 16-byte load form
        fwd, wgrad = T.conv_fwd_spec(g, xl, yl), T.conv_wgrad_spec(g, xl, yl)
        dgrads = T.conv_dgrad_specs(g, xl, yl, "nhwc" if g.kh == 1 else xl)   # 1x1: OIHW and OHWI are the same memory
        if launchable(fwd):
            out = back(run_spec(fwd, xb, wl, oshape, prec, bias=b), yl)
            e_f = (out[:, g.y_coff:g.y_coff + g.cout].double() - y).abs().max().item() / y.abs().max().item()
            out2 = back(run_spec(fwd, xb, wl, oshape, prec, split_k=3), yl)
            y_nb = y - b.double().view(1, -1, 1, 1)
            e_s = (out2[:, g.y_coff:g.y_coff + g.cout].double() - y_nb).abs().max().item() / y.abs().max().item()
        if launchable(wgrad):
            db = torch.zeros(g.cout, device=dev)
            dw = run_spec(wgrad, xb, dyb, tuple(wl.shape), prec, ones=db, split_k=4, atomic=True)
            dwc = dw.permute(0, 3, 1, 2) if xl == "nhwc" else dw
            e_w = (dwc.double() - wd.grad).abs().max().item() / wd.grad.abs().max().item()
            e_b = (db.double() - dy[:, g.y_coff:g.y_coff + g.cout].double().sum((0, 2, 3))).abs().max().item() / db.abs().max().item()
        if all(launchable(spc) for spc in dgrads):
            dx = torch.zeros_like(xb)
            for spc in dgrads:
                dx += run_spec(spc, dyb, wl, tuple(xb.shape), prec)
            dxc = back(dx, xl)
            e_d = (dxc[:, g.x_coff:g.x_coff + g.cin].double() - xs.grad).abs().max().item() / xs.grad.abs().max().item()
        worst = max([worst] + [e for e in (e_f, e_s, e_w, e_b, e_d) if e == e])
        print(f"[{label}] {xl}->{yl} {name:16s} rel-err fwd {e_f:.2e} splitK {e_s:.2e} wgrad {e_w:.2e} bgrad {e_b:.2e} dgrad {e_d:.2e}  ({time.time()-t0:.2f}s)", flush=True)
    print(f"[{label}] worst {worst:.3e}", flush=True)


def check_stencil():
    lib = L.lib()
    torch.manual_seed(1)
    for (B, Lg, S, K, mode, drop) in [(2, 3, 28, 1, 0, 0), (3, 4, 14, 1, 1, 1), (2, 2, 7, 1, 0, 2), (2, 3, 7, 2, 0, 0), (1, 3, 28, 1, 0, 1)]:
        N, P, Cg, Cs = B * Lg, B * (Lg - 1), 128, 32
        gd_c = torch.randn(N, Cg + Cs, S, S, device=dev)
        gd_c[:, :Cg].relu_()
        gd = gd_c.permute(0, 2, 3, 1).contiguous()            # channels-last [N,S,S,160]
        w = torch.randn(Cs, K, 3, 3, device=dev)
        bias = torch.randn(Cs * K, device=dev)
        ctot, coff = 400, 64
        out = torch.zeros(P, S, S, ctot, device=dev)
        sd = L.OffkStencil()
        sd.B, sd.L, sd.Cg, sd.Cs, sd.K, sd.H, sd.W = B, Lg, Cg, Cs, K, S, S
        sd.g_fs = sd.d_fs = (Cg + Cs) * S * S
        sd.g_ps = sd.d_ps = Cg + Cs
        sd.out_ctot, sd.out_coff, sd.index_mode = ctot, coff, mode
        sd.drop_mode, sd.keep_scale, sd.drop_p, sd.seed = drop, 5.0, 0.8, 1234
        mask = (torch.rand(P, K * Cs, S, S, device=dev) > 0.8).to(torch.uint8)
        sd.keep_mask = mask.data_ptr()
        L.check(lib.offk_stencil_diff_fwd(C.byref(sd), gd.data_ptr(), gd.data_ptr() + 4 * Cg, w.data_ptr(),
                                          bias.data_ptr(), out.data_ptr(), None), "stencil_fwd")
        torch.cuda.synchronize()
        # reference
        G = gd_c[:, :Cg].double()
        D = gd_c[:, Cg:].double()
        out = out.permute(0, 3, 1, 2)
        Gv = G.view(B, Lg, Cg, S, S)
        Tref = (Gv[:, 1:] - Gv[:, :-1]).reshape(P, Cg, S, S)
        if mode == 0:
            Ds = D[:P]
        else:
            Ds = D.view(B, Lg, Cs, S, S)[:, :-1].reshape(P, Cs, S, S)
        Ds = Ds.clone().requires_grad_(True)
        wd = w.double().clone().requires_grad_(True)
        bd = bias.double().clone().requires_grad_(True)
        # out channel kk*Cs + c uses w[c,kk]
        wk = wd.permute(1, 0, 2, 3).reshape(K * Cs, 1, 3, 3)
        Sg = torch.nn.functional.conv2d(Ds.repeat(1, K, 1, 1), wk, bd, 1, 1, 1, K * Cs)
        if drop == 1:
            keep = mask.double() * 5.0
        elif drop == 2:
            idx = np.arange(P * K * Cs * S * S, dtype=np.uint64)
            keep_np = np.array([lib.offk_drop_keep_host(1234, int(i), 0.8) for i in idx[:4096]])
            # full host hash in numpy (same formula as drop_hash24)
            x = (np.uint64(1234) + idx * np.uint64(0x9E3779B97F4A7C15))
            x ^= x >> np.uint64(30); x *= np.uint64(0xBF58476D1CE4E5B9); x ^= x >> np.uint64(27)
            x *= np.uint64(0x94D049BB133111EB); x ^= x >> np.uint64(31)
            k24 = (x >> np.uint64(40)).astype(np.int64) >= int(0.8 * 16777216.0)
            assert (k24[:4096].astype(int) == keep_np).all()
            keep = torch.from_numpy(k24.astype(np.float64)).to(dev).view(P, K * Cs, S, S) * 5.0
            print("   seeded keep fraction", float(k24.mean()))
        else:
            keep = torch.ones(P, K * Cs, S, S, device=dev, dtype=torch.float64)
        Sg = Sg * keep
        ref = torch.cat([Sg, Tref], 1)
        got = out[:, coff:coff + K * Cs + Cg].double()
        e = (got - ref.detach()).abs().max().item()
        untouched = out[:, :coff].abs().max().item() + out[:, coff + K * Cs + Cg:].abs().max().item()
        # backward
        dout_l = torch.randn(P, S, S, ctot, device=dev)
        dout = dout_l.permute(0, 3, 1, 2)
        dgd_l = torch.full((N, S, S, Cg + Cs), float("nan"), device=dev)
        dgd = dgd_l.permute(0, 3, 1, 2)
        dw = torch.zeros_like(w)
        dbias = torch.zeros_like(bias)
        fs = (Cg + Cs) * S * S
        L.check(lib.offk_stencil_diff_bwd(C.byref(sd), dout_l.data_ptr(), gd.data_ptr(), gd.data_ptr() + 4 * Cg,
                                          w.data_ptr(), dgd_l.data_ptr(), fs, dgd_l.data_ptr() + 4 * Cg, fs,
                                          dw.data_ptr(), dbias.data_ptr(), None), "stencil_bwd")
        torch.cuda.synchronize()
        dS = dout[:, coff:coff + K * Cs].double()
        dT = dout[:, coff + K * Cs:coff + K * Cs + Cg].double().view(B, Lg - 1, Cg, S, S)
        dG = torch.zeros(B, Lg, Cg, S, S, device=dev, dtype=torch.float64)
        dG[:, 1:] += dT
        dG[:, :-1] -= dT
        dG = dG.view(N, Cg, S, S) * (G > 0)
        Sg.backward(dS)
        dD = torch.zeros(N, Cs, S, S, device=dev, dtype=torch.float64)
        if mode == 0:
            dD[:P] = Ds.grad
        else:
            dD.view(B, Lg, Cs, S, S)[:, :-1] = Ds.grad.view(B, Lg - 1, Cs, S, S)
        e_g = (dgd[:, :Cg].double() - dG).abs().max().item()
        e_d = (dgd[:, Cg:].double() - dD).abs().max().item()
        e_w = (dw.double() - wd.grad).abs().max().item() / wd.grad.abs().max().item()
        e_b = (dbias.double() - bd.grad).abs().max().item() / bd.grad.abs().max().item()
        print(f"[stencil] B{B} L{Lg} S{S} K{K} mode{mode} drop{drop}: fwd {e:.2e} untouched {untouched:.1e} dG {e_g:.2e} dD {e_d:.2e} dw(rel) {e_w:.2e} db(rel) {e_b:.2e}", flush=True)


def check_engine(precision, variant="rgb", B=2, Lg=3, train=False):
    seed = 5
    taps = O.make_taps(seed, B, Lg)
    prm = O.make_params(seed, variant)
    masks = O.make_dropout_masks(seed, B, Lg) if train else None
    r7 = O.hash_normal(77, (B * (Lg - 1) if variant == "rgb" else B, 101)).double()
    r14 = O.hash_normal(78, (B * (Lg - 1) if variant == "rgb" else B, 101)).double()
    lossf = lambda o: (o["fc7"].reshape(r7.shape) * r7).sum() + (o["fc14"].reshape(r14.shape) * r14).sum()
    ref, gref = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float64, loss=lossf)
    _, g32 = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float32, loss=lambda o: (o["fc7"].reshape(r7.shape) * r7.float()).sum() + (o["fc14"].reshape(r14.shape) * r14.float()).sum())
    eng = E.OFFEngine(B, Lg, variant, dev, precision)
    eng.load_params(prm)
    fc7, fc28, fc14 = eng.forward({k: v.to(dev) for k, v in taps.items()}, train=train, masks=masks)
    torch.cuda.synchronize()
    rel = lambda a, b: (a.double().cpu() - b).abs().max().item() / max(b.abs().max().item(), 1e-30)
    print(f"[engine {precision} {variant} B{B} L{Lg} train={train}]")
    for k, st in (("fusion28", "F28"), ("fusion14", "F14"), ("fusion7", "F7")):
        a, b = eng.buf[st].permute(0, 3, 1, 2).double().cpu(), ref[k]
        print(f"   {k}: max-abs {(a-b).abs().max().item():.3e} rel {rel(eng.buf[st].permute(0, 3, 1, 2), b):.3e} (|ref|max {b.abs().max().item():.3f})")
    print(f"   sum7: rel {rel(eng.buf['s7'].permute(0, 3, 1, 2), ref['sum7']):.3e}")
    for nme, got, key in (("fc7", fc7, "fc7"), ("fc28", fc28, "fc28"), ("fc14", fc14, "fc14")):
        b = ref[key].reshape(got.shape)
        print(f"   {nme}: max-abs {(got.double().cpu()-b).abs().max().item():.3e} rel {rel(got, b):.3e}")
    g7 = r7.float().to(dev).reshape(fc7.shape)
    g14 = r14.float().to(dev).reshape(fc14.shape)
    grads = eng.backward(g7, g14)
    torch.cuda.synchronize()
    worst = ("", 0.0)
    for n, g in grads.items():
        b = gref[n]
        if b.abs().max().item() == 0:
            assert g.abs().max().item() == 0, n
            continue
        r = rel(g, b)
        if r > worst[1]:
            worst = (n, r)
        if r > (1e-4 if precision == "fp32" else 3e-2):
            print(f"   grad {n}: rel {r:.3e}  <-- large")
    floor = max((g32[n].double() - gref[n]).abs().max().item() / max(gref[n].abs().max().item(), 1e-30) for n in gref if gref[n].abs().max().item() > 0)
    print(f"   worst grad rel err: {worst[0]} {worst[1]:.3e}   (fp32 CPU oracle vs fp64: {floor:.3e})", flush=True)


if __name__ == "__main__":
    what = sys.argv[1:] or ["gemm_tc", "stencil", "engine_fp32"]
    if what[0].startswith("perf"):
        what = []
    for w in what:
        if w == "gemm_tc":
            check_gemm(L.PREC_TF32, "tc")
        elif w == "stencil":
            check_stencil()
        elif w.startswith("engine_"):
            prec = w.split("_")[1]
            check_engine(prec, "rgb", 2, 3)
            check_engine(prec, "flow", 2, 3)
            check_engine(prec, "rgb", 2, 2, train=True)


def perf(precision="tf32", B=48, Lg=3, variant="rgb", detail=True):
    eng = E.OFFEngine(B, Lg, variant, dev, precision)
    prm = O.make_params(3, variant)
    eng.load_params(prm)
    for t in eng.taps.values():
        t.copy_(torch.relu(torch.randn_like(t)))
    g7 = torch.randn(eng.P, 101, device=dev) if not eng.consensus else torch.randn(B, 101, device=dev)
    g14 = torch.randn_like(g7)
    for _ in range(2):
        eng.forward(train=True, seed=1)
        eng.backward(g7, g14)
    torch.cuda.synchronize()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for label, fn in (("fwd", lambda: eng.forward(train=True, seed=2)), ("bwd", lambda: eng.backward(g7, g14))):
        s, e = ev(), ev()
        s.record()
        for _ in range(5):
            fn()
        e.record()
        torch.cuda.synchronize()
        print(f"[perf {precision} B{B} L{Lg}] {label}: {s.elapsed_time(e)/5:.3f} ms", flush=True)
    if detail:
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for label, steps in (("fwd", eng.fwd_steps), ("bwd", eng.bwd_steps)):
            rows = []
            for i, st in enumerate(steps):
                s, e = ev(), ev()
                st(stream)
                torch.cuda.synchronize()
                s.record()
                for _ in range(3):
                    st(stream)
                e.record()
                torch.cuda.synchronize()
                nm = getattr(st, "name", None) or getattr(st, "__name__", "step")
                fl = getattr(st, "flops", 0.0)
                rows.append((s.elapsed_time(e) / 3, nm, fl))
            tot = sum(r[0] for r in rows)
            print(f"--- {label} per-step (sum {tot:.3f} ms)")
            for t, nm, fl in sorted(rows, reverse=True)[:28]:
                print(f"   {t*1e3:9.1f} us  {nm:40s} {fl/t/1e9 if fl else 0:8.1f} TFLOP/s")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1].startswith("perf"):
    for p in sys.argv[2:] or ["tf32"]:
        perf(p)
