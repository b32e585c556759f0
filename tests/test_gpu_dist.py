"""GPU, >= 2 devices: clip-sharded data parallelism of the OFF path over NCCL (SURVEY.md sections 4-iv, 8e).

Each rank builds the engine with its LOCAL batch and its own clips; per-rank outputs must match the oracle run at the local
batch on those clips (the reference's flat-index quirk, RGB_OFF.py:609, makes the result depend on how clips are grouped),
and the all-reduced gradients must equal the MEAN of the per-rank oracle gradients.  Skipped with fewer than two GPUs; on
a machine with two or more, run `python -m pytest tests/test_gpu_dist.py -m gpu`.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import off_oracle as O

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, variant, b_local, length, precision, out):
    import off_b200  # noqa: F401
    from off_b200 import engine as E
    from off_b200.dist import DataParallelOFF
    from helpers import engine_gates
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    seed = 21
    # the global batch, cut by clip: rank r owns clips [r*b_local, (r+1)*b_local)
    taps_all = O.make_taps(seed, b_local * world, length)
    taps = {k: v.view(world, b_local * length, *v.shape[1:])[rank].contiguous() for k, v in taps_all.items()}
    prm = O.make_params(seed, variant)
    eng = E.OFFEngine(b_local, length, variant, dev, precision)
    if rank == 0:
        eng.load_params(prm)                                  # other ranks start from zeros: broadcast must fix that
    dp = DataParallelOFF(eng)
    dp.broadcast_parameters()
    n_out = b_local * (length - 1) if variant == "rgb" else b_local
    r7 = O.hash_normal(300 + rank, (n_out, 101)).double()
    r14 = O.hash_normal(400 + rank, (n_out, 101)).double()
    fc7, fc28, fc14 = eng.forward({k: v.to(dev) for k, v in taps.items()}, train=False)
    torch.cuda.synchronize()
    lossf = lambda o: (o["fc7"].reshape(r7.shape) * r7).sum() + (o["fc14"].reshape(r14.shape) * r14).sum()
    ref, gref = O.off_forward_backward(taps, prm, b_local, length, variant, None, torch.float64, loss=lossf,
                                       gates=engine_gates(eng))
    rel = lambda a, b: (a.detach().double().cpu() - b).abs().max().item() / b.abs().max().item()
    fwd_err = max(rel(fc7, ref["fc7"].reshape(fc7.shape)), rel(fc14, ref["fc14"].reshape(fc14.shape)),
                  rel(eng.buf["F28"].permute(0, 3, 1, 2), ref["fusion28"]))
    grads = dp.backward(r7.float().to(dev), r14.float().to(dev))
    torch.cuda.synchronize()
    worst = 0.0
    for n, g in grads.items():
        want = gref[n].to(dev)                                # mean over ranks of the per-rank oracle gradients
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        want /= world
        if want.abs().max().item() == 0:
            assert g.abs().max().item() == 0, n
            continue
        worst = max(worst, ((g.double() - want).norm() / want.norm()).item())
    res = torch.tensor([fwd_err, worst], device=dev, dtype=torch.float64)
    dist.all_reduce(res, op=dist.ReduceOp.MAX)
    if rank == 0:
        torch.save(res.cpu(), out)
    dist.destroy_process_group()


@pytest.mark.parametrize("variant,b_local,length,precision", [("rgb", 2, 3, "fp32"), ("flow", 1, 4, "tf32")])
def test_data_parallel_matches_per_rank_oracle(tmp_path, variant, b_local, length, precision):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(world, _free_port(), variant, b_local, length, precision, out), nprocs=world, join=True)
    fwd_err, worst = torch.load(out).tolist()
    print(f"[dp parity {precision} {variant} {world} ranks x {b_local} clips] fwd={fwd_err:.2e} allreduced_grad_rel_l2={worst:.2e}")
    if precision == "fp32":
        assert fwd_err < 1e-5 and worst < 2e-5, (fwd_err, worst)
    else:
        assert fwd_err < 1e-2 and worst < 0.2, (fwd_err, worst)
