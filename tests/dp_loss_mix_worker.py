"""torchrun worker for tests/test_engine_loss_mix_gpu.py: 2-rank Stage-I step in a pixel-NLE loss mix ('dcgan' / 'vae') over
NCCL vs the sequential-shards emulation. argv: mode, f32 | bf16, global batch."""
import json
import os
import sys

import torch
import torch.distributed as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import vaegan as O  # noqa: E402  (test infrastructure: deterministic weights / inputs)
from thesis_fmri_reconstruction_b200 import dp, engine, hp  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    td.init_process_group("nccl", device_id=torch.device("cuda", local))
    mode = sys.argv[1]
    adt = torch.float32 if sys.argv[2] == "f32" else torch.bfloat16
    B = int(sys.argv[3])
    P, S = O.make_vaegan(O.CFG64, seed=818)
    x = O.synthetic_images(B, seed=818)
    eps, z_p = O.synthetic_noise(B, 128, seed=818)
    lo, hi = dp.shard_range(B, rank, world)
    tr = engine.VaeGanStage1(P, S, hp.CFG64, 128, adt, dist_group=td.group.WORLD, mode=mode)
    tr.forward_backward(x[lo:hi].cuda(), eps[lo:hi].cuda(), z_p[lo:hi].cuda())
    tr.update(B)
    torch.cuda.synchronize()
    got = {pre: b.flat_g.clone() for pre, b in tr.buckets.items()}
    losses = tr.losses()
    # emulation on this GPU: the same shards one after the other through a world-size-1 engine, gradients summed
    tot, sums = None, torch.zeros(16, device="cuda")
    for r in range(world):
        l2, h2 = dp.shard_range(B, r, world)
        e1 = engine.VaeGanStage1(P, S, hp.CFG64, 128, adt, mode=mode)
        e1.forward_backward(x[l2:h2].cuda(), eps[l2:h2].cuda(), z_p[l2:h2].cuda())
        torch.cuda.synchronize()
        g = {pre: b.flat_g.clone() for pre, b in e1.buckets.items()}
        tot = g if tot is None else {k: tot[k] + g[k] for k in g}
        sums += e1.sc
    # buckets with a zero sum ('dcgan' trains no encoder) are reported by their largest element instead
    errs = {pre: ((got[pre] - tot[pre]).double().norm() / tot[pre].double().norm()).item() for pre in got
            if tot[pre].abs().max().item() > 0}
    sum_err = ((tr.sc[:6] - sums[:6]).abs().max() / sums[:6].abs().max()).item()
    gate = dp.gate_from_sums(sums[0].item(), sums[1].item(), B, tr.hp["margin"], tr.hp["equilibrium"],
                             train_dis_in=mode != "vae")
    res = dict(rank=rank, mode=mode, grad_err=errs, sum_err=sum_err, gate_dev=(losses["train_dis"], losses["train_dec"]),
               gate_host=gate, enc_grad_max=got["encoder."].abs().max().item())
    allres = [None] * world
    td.all_gather_object(allres, res)
    if rank == 0:
        print("DPRESULT " + json.dumps(allres))
    td.barrier()
    td.destroy_process_group()


if __name__ == "__main__":
    main()
