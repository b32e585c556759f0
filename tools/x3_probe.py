"""What does tcgen05 kind::tf32 do with the low 13 mantissa bits, and how exact is the 3xTF32 mode?
Dense GEMMs through the gather-fed kernel in OFFK_PREC_TF32 and OFFK_PREC_TF32X3 against fp64 references computed from
(a) the raw fp32 operands, (b) operands truncated to tf32, (c) operands rounded to nearest tf32.
python tools/x3_probe.py   (bring-up tool; not a test)"""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import off_b200  # noqa
from off_b200 import _lib as L, tables as T

dev = torch.device("cuda")


def run(A, B, prec, a_mn=False, b_mn=False, tile_n=0):
    M, K = A.shape
    N = B.shape[0]
    a_store = A.t().contiguous() if a_mn else A.contiguous()
    b_store = B.t().contiguous() if b_mn else B.contiguous()
    idx = lambda off: np.array([(o, 0, 0) for o in off], dtype=T.IDX_DTYPE)
    spc = T.GemmSpec(
        M=M, N=N, K=K,
        a_row=idx(np.arange(M) * (1 if a_mn else K)), a_col=idx(np.arange(K) * (M if a_mn else 1)),
        b_row=(np.arange(N) * (1 if b_mn else K)).astype(np.int32), b_col=(np.arange(K) * (N if b_mn else 1)).astype(np.int32),
        out_row=(np.arange(M) * N).astype(np.int32), out_col=np.arange(N).astype(np.int32),
        a_mode=T.LOAD_VEC_ROW if a_mn else T.LOAD_VEC_K, b_mode=T.LOAD_VEC_ROW if b_mn else T.LOAD_VEC_K, out_vec=0)
    tabs = {k: torch.from_numpy(v).to(dev) for k, v in T.padded_tables(spc).items()}
    out = torch.zeros(M, N, device=dev)
    d = L.OffkGemm()
    d.M, d.N, d.K = M, N, K
    d.a_src, d.a_row, d.a_col = a_store.data_ptr(), tabs["a_row"].data_ptr(), tabs["a_col"].data_ptr()
    d.a_h, d.a_w, d.a_ones_row, d.a_mode = T.NO_BOX, T.NO_BOX, -1, spc.a_mode
    d.b_src, d.b_row, d.b_col, d.b_mode = b_store.data_ptr(), tabs["b_row"].data_ptr(), tabs["b_col"].data_ptr(), spc.b_mode
    d.out, d.out_row, d.out_col = out.data_ptr(), tabs["out_row"].data_ptr(), tabs["out_col"].data_ptr()
    d.split_k, d.tile_n = 1, tile_n
    L.check(L.lib().offk_gather_gemm(C.byref(d), prec, None), "gemm")
    torch.cuda.synchronize()
    return out


def trunc(x):
    return (x.view(torch.int32) & -8192).view(torch.float32)


def rna(x):                                   # round to nearest, ties away: add half an ulp of tf32 to the magnitude
    return ((x.view(torch.int32) + 0x1000) & -8192).view(torch.float32)


for (M, N, K, a_mn, b_mn, pos) in [(256, 128, 512, False, False, False), (256, 128, 512, False, False, True),
                                   (384, 256, 2048, True, True, False), (128, 64, 96, True, False, True)]:
    torch.manual_seed(1)
    A = torch.randn(M, K, device=dev)
    B = torch.randn(N, K, device=dev)
    if pos:
        A, B = A.abs(), B.abs()
    exact = A.double() @ B.double().t()
    ref_t = trunc(A).double() @ trunc(B).double().t()
    ref_r = rna(A).double() @ rna(B).double().t()
    scale = exact.abs().max().item()
    e = lambda got, ref: (got.double() - ref).abs().max().item() / scale
    y1 = run(A, B, L.PREC_TF32, a_mn, b_mn)
    y3 = run(A, B, L.PREC_TF32X3, a_mn, b_mn)
    print(f"M{M} N{N} K{K} a_mn={a_mn} b_mn={b_mn} positive={pos}")
    print(f"   tf32   vs exact {e(y1, exact):.2e} | vs truncated operands {e(y1, ref_t):.2e} | vs rounded operands {e(y1, ref_r):.2e}")
    print(f"   tf32x3 vs exact {e(y3, exact):.2e}   torch fp32 matmul {e((A @ B.t()), exact):.2e}", flush=True)
