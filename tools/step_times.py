"""Per-step device time of one OFF forward+backward (CUDA events around every plan step, single stream, warm, mean of
`iters` passes) -- the quick alternative to an ncu launch list.  python tools/step_times.py [B] [L] [prec] [iters] [filter]"""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import off_b200  # noqa
from off_b200 import engine as E, plan as PL

B = int(sys.argv[1]) if len(sys.argv) > 1 else 48
Lg = int(sys.argv[2]) if len(sys.argv) > 2 else 3
prec = sys.argv[3] if len(sys.argv) > 3 else "tf32"
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 5
flt = sys.argv[5] if len(sys.argv) > 5 else ""
eng = E.OFFEngine(B, Lg, "rgb", "cuda", prec)
torch.manual_seed(0)
with torch.no_grad():
    for n, v in eng.params.items():
        fan = v[0].numel() if v.dim() > 1 else 64
        v.uniform_(-1.0 / fan ** 0.5, 1.0 / fan ** 0.5)
for t in eng.taps.values():
    t.copy_(torch.relu(torch.randn_like(t)))
g7 = torch.randn(eng.P, 101, device="cuda") * 0.01
g14 = torch.randn(eng.P, 101, device="cuda") * 0.01
eng.single_stream = True
for _ in range(2):
    eng.forward(train=True, seed=1)
    eng.backward(g7, g14)
steps = list(eng.fwd_steps) + list(eng.bwd_steps)
names = ["+".join(PL._names(s)) for s in steps]
acc = [0.0] * len(steps)
st = torch.cuda.current_stream()
h = C.c_void_p(st.cuda_stream)
eng._set_dropout(True, None, 1)
eng.d_out7.copy_(g7.reshape(eng.d_out7.shape))
eng.d_out14.copy_(g14.reshape(eng.d_out14.shape))
for it in range(iters):
    evs = []
    for s in steps:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        s(h)
        b.record(st)
        evs.append((a, b))
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(evs):
        acc[i] += a.elapsed_time(b) * 1e3 / iters
tot = 0.0
for i, (n, t) in enumerate(zip(names, acc)):
    tot += t
    if flt in n:
        print(f"{i:4d} {t:8.1f} us  {n}")
print(f"TOTAL {tot:.1f} us over {len(steps)} steps (B={B} L={Lg} {prec}; event-bracketed, includes launch gaps)")
