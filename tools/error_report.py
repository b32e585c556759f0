"""Per-level error report of the sm_100a OFF path against the fp64 CPU oracle (north_star: "fp32 max-abs and relative
error reported per level; tf32 GEMM tolerance stated separately").

    python tools/error_report.py > profiles/parity_report.txt          (needs a B200; ~30 s)

For every OFF unit (level 3a..5b) the 160-channel slice it writes into its stage-fusion buffer -- 32 spatial-gradient
channels (RGB_OFF.py:611 / Flow_OFF.py:622) and 128 temporal-difference channels (:599-604) -- then the three
stage-fusion tensors as a whole, the heads, and the parameter gradients per layer family.  Columns: max |got - ref|,
the same divided by max |ref| of that tensor, for the fp32 mode (3xTF32 tcgen05) and the tf32 mode (tcgen05
kind::tf32).  The last column is the error of the reference's OWN fp32 CPU arithmetic (oracle run in float32, i.e. the
ATen CPU kernels the reference calls) against the same fp64 truth: the noise floor any fp32 implementation has.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import off_b200  # noqa
from off_b200 import engine as E, spec as S
import off_oracle as O

dev = torch.device("cuda")


def err(got, ref):
    d = (got.detach().double().cpu() - ref.double()).abs().max().item()
    return d, d / max(ref.double().abs().max().item(), 1e-30)


def rel_l2(got, ref):
    return (got.detach().double().cpu() - ref.double()).norm().item() / max(ref.double().norm().item(), 1e-30)


def run_case(variant, B, Lg, train):
    seed = 5
    taps, prm = O.make_taps(seed, B, Lg), O.make_params(seed, variant)
    masks = O.make_dropout_masks(seed, B, Lg) if train else None
    n_out = B * (Lg - 1) if variant == "rgb" else B
    r7, r14 = O.hash_normal(77, (n_out, 101)).double(), O.hash_normal(78, (n_out, 101)).double()
    lossf = lambda o: (o["fc7"].reshape(r7.shape) * r7.to(o["fc7"].dtype)).sum() + (o["fc14"].reshape(r14.shape) * r14.to(o["fc14"].dtype)).sum()
    ref, gref = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float64, loss=lossf)
    cpu32, gcpu32 = O.off_forward_backward(taps, prm, B, Lg, variant, masks, torch.float32, loss=lossf)
    res = {}
    for prec in ("fp32", "tf32"):
        eng = E.OFFEngine(B, Lg, variant, dev, prec)
        eng.load_params(prm)
        fc7, fc28, fc14 = eng.forward({k: v.to(dev) for k, v in taps.items()}, train=train, masks=masks)
        fus = {st: eng.buf["F" + st].permute(0, 3, 1, 2).contiguous().cpu() for st in S.STAGES}
        heads = {"fc7": fc7.cpu().clone(), "fc28": fc28.cpu().clone(), "fc14": fc14.cpu().clone()}
        grads = {n: g.cpu().clone() for n, g in eng.backward(r7.float().to(dev), r14.float().to(dev)).items()}
        torch.cuda.synchronize()
        res[prec] = (fus, heads, grads)
    print(f"\n=== variant {variant}, batch {B}, segments {Lg}, dropout {'train (injected masks)' if train else 'eval'} "
          f"(RGB_OFF.py:596-860 / Flow_OFF.py:606-884 on seeded synthetic taps) ===")
    hdr = f"{'tensor':34s} {'max|ref|':>9s} | {'fp32 abs':>9s} {'fp32 rel':>9s} | {'tf32 abs':>9s} {'tf32 rel':>9s} | {'cpu-fp32 rel':>12s}"
    print(hdr)
    print("-" * len(hdr))

    def line(name, getter, refv, cpuv):
        a32, r32 = err(getter("fp32"), refv)
        at, rt = err(getter("tf32"), refv)
        _, rc = err(cpuv, refv)
        print(f"{name:34s} {refv.abs().max().item():9.3e} | {a32:9.2e} {r32:9.2e} | {at:9.2e} {rt:9.2e} | {rc:12.2e}")

    for st, (ctot, s, members) in S.STAGES.items():
        key = "fusion" + st
        for tag, coff in members:
            if tag not in S.LEVELS:
                continue
            for part, lo, hi in (("spatial", coff, coff + S.DOWN_C), ("temporal", coff + S.DOWN_C, coff + S.UNIT_C)):
                line(f"level {tag} {part} [{s}x{s}]", lambda p, st=st, lo=lo, hi=hi: res[p][0][st][:, lo:hi],
                     ref[key][:, lo:hi], cpu32[key][:, lo:hi])
    for st in S.STAGES:
        key = "fusion" + st
        line(f"stage-fusion tensor {st} (all ch.)", lambda p, st=st: res[p][0][st], ref[key], cpu32[key])
    for h in ("fc7", "fc14", "fc28"):
        line(f"head {h}", lambda p, h=h: res[p][1][h], ref[h].reshape(res["fp32"][1][h].shape), cpu32[h].reshape(res["fp32"][1][h].shape))
    print(f"{'gradients (relative L2 per family)':34s} {'':9s} | {'fp32':>19s} | {'tf32':>19s} | {'cpu-fp32':>12s}")
    fams = [("unit 1x1 (gen, down)", lambda n: n.startswith(("motion_conv_gen_", "motion_spatial_down_"))),
            ("unit 3x3 spatial grad", lambda n: n.startswith("motion_spatial_grad_")),
            ("stage-entry KxK convs", lambda n: n in ("motion_conv_trans_28.weight", "motion_conv_trans_14.weight", "motion_conv_trans.weight")),
            ("residual blocks", lambda n: "_trans_" in n and not n.startswith(("motion_conv_trans_28.", "motion_conv_trans_14."))
             or n.startswith(("motion_conv1_trans.", "motion_conv2_trans.", "motion_conv3_trans.", "motion_conv_branch"))),
            ("FC heads", lambda n: n.startswith("fc_action_motion"))]
    for fname, pred in fams:
        names = [n for n in gref if pred(n) and gref[n].abs().max().item() > 0]
        if not names:
            continue
        w32 = max(rel_l2(res["fp32"][2][n], gref[n]) for n in names)
        wt = max(rel_l2(res["tf32"][2][n], gref[n]) for n in names)
        wc = max(rel_l2(gcpu32[n], gref[n]) for n in names)
        print(f"  worst of {len(names):3d} {fname:22s} {'':8s} | {w32:19.2e} | {wt:19.2e} | {wc:12.2e}")


if __name__ == "__main__":
    print(__doc__.split("\n\n")[0])
    print("device:", torch.cuda.get_device_name(0))
    run_case("rgb", 2, 3, False)
    run_case("flow", 2, 3, False)
    run_case("rgb", 2, 2, True)
