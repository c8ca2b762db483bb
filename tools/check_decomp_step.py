"""GraphedKLLoss(loss="decomp") row-sharded over NCCL and over the peer-memory exchange vs the single-process step on the global
batch (run under torchrun, >= 2 GPUs).  Three rounds of fresh inputs per shape exercise the exchange's buffer rotation.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29547 tools/check_decomp_step.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from intro_tc_vae_b200.graphs import GraphedKLLoss


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    ok = True

    def rel(a, b):
        return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()

    for B, D, N, beta, estimator in ((256, 128, 16704, 6.0, "mss"), (1024, 128, 16704, 0.5, "mws"), (296, 20, 5000, 4.0, "mss")):
        b_loc = B // world
        lo = rank * b_loc
        single = GraphedKLLoss(B, D, N, beta, dev, estimator=estimator, loss="decomp")
        sharded = {x: GraphedKLLoss(b_loc, D, N, beta, dev, group=dist.group.WORLD, estimator=estimator, exchange=x, loss="decomp")
                   for x in ("nccl", "peer")}
        for rnd in range(3):
            g = torch.Generator().manual_seed(B + D + 17 * rnd)
            mu_c = torch.randn(B, D, generator=g)
            lv_c = -2.0 + torch.randn(B, D, generator=g)
            eps_c = torch.randn(B, D, generator=g)
            l_f, dm_f, dl_f = (t.clone() for t in single(mu_c.to(dev), lv_c.to(dev), eps_c.to(dev)))
            # the global mean is the mean of the ranks' means (equal shards); the gradients of the ranks' means add up to
            # world times those of the global mean
            for x, step in sharded.items():
                loss, dmu, dlv = (t.clone() for t in step(*(t[lo:lo + b_loc].to(dev) for t in (mu_c, lv_c, eps_c))))
                loss_all = loss.reshape(1).clone()
                dist.all_reduce(loss_all)
                e = (abs(loss_all.item() / world - l_f.item()) / abs(l_f.item()),
                     rel(dmu, world * dm_f[lo:lo + b_loc]), rel(dlv, world * dl_f[lo:lo + b_loc]))
                good = e[0] < 1e-5 and e[1] < 1e-5 and e[2] < 1e-5
                ok = ok and good
                print(f"rank {rank} {x} B={B} D={D} {estimator} round {rnd}: loss rel {e[0]:.1e}  dmu rel {e[1]:.1e}  "
                      f"dlv rel {e[2]:.1e}  {'OK' if good else 'MISMATCH'}", flush=True)
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res = int(flag.item())
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0 if res == 1 else 1)       # graphs that captured collectives make destroy_process_group hang


if __name__ == "__main__":
    main()
