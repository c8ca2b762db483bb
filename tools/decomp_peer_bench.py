"""Time the row-sharded decomposition loss (ops.tc_decomp_loss_mean, forward + backward) with its two exchanges:

    nccl  group=...     all-gather of mu and logvar before the op, reduce-scatter of both column gradients after it
    peer  exchange=...  both steps inside the library's kernels over NVLink peer memory (peer.PeerExchange)

Run under torchrun with one process per GPU; the GLOBAL batch is held fixed, each rank owns B / world rows.  The two are timed
alternately within one call, in rounds, with CUDA events around `--iters` steps each (each step ends in torch.autograd.grad
w.r.t. z, mu and logvar; z is a leaf, so no reparameterize is timed).  Rank 0 prints one JSON line naming the GPU and its power
limit, then one per batch size with the median step time over the rounds (the slowest rank of each round).

    python -m torch.distributed.run --nproc-per-node 8 tools/decomp_peer_bench.py [--sizes 8192,1024] [--d 128]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from intro_tc_vae_b200 import ops, peer  # noqa: E402

N_DATA = 16704
BETA = 6.0


def _power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def step(inputs, **kw):
    z, mu, lv = inputs
    loss = ops.tc_decomp_loss_mean(z, mu, lv, N_DATA, BETA, "mss", **kw)[0]
    return (loss,) + torch.autograd.grad(loss, [z, mu, lv])


def time_steps(inputs, iters, **kw):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        step(inputs, **kw)
    stop.record()
    stop.synchronize()
    t = torch.tensor([start.elapsed_time(stop) / iters], device=inputs[0].device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)                       # a step is as slow as its slowest rank
    return t.item()


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", default="8192,1024")
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decomp_peer_bench: no CUDA device; these timings only mean something on the GPU")
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD
    if rank == 0:
        print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "power_limit": _power_limit(), "gpus": world, "d": args.d,
                          "iters_per_round": args.iters, "rounds": args.rounds}), flush=True)
    for b in (int(s) for s in args.sizes.split(",")):
        b_loc = b // world
        g = torch.Generator().manual_seed(b)
        mu_c = torch.randn(b, args.d, generator=g)
        lv_c = -2.0 + torch.randn(b, args.d, generator=g)
        z_c = mu_c + torch.randn(b, args.d, generator=g) * torch.exp(0.5 * lv_c)
        rows = slice(rank * b_loc, (rank + 1) * b_loc)
        inputs = [t[rows].to(dev).requires_grad_(True) for t in (z_c, mu_c, lv_c)]
        exch = peer.PeerExchange(b_loc, args.d, group, dev)
        ways = {"nccl": dict(group=group), "peer": dict(exchange=exch)}
        outs = {}
        for name, kw in ways.items():
            for _ in range(args.warmup):
                step(inputs, **kw)
            outs[name] = [t.detach() for t in step(inputs, **kw)]
        torch.cuda.synchronize()
        times = {name: [] for name in ways}
        for _ in range(args.rounds):                               # alternate, so that drift hits both alike
            for name, kw in ways.items():
                times[name].append(time_steps(inputs, args.iters, **kw))
        diffs = [float((p - n).abs().max() / n.abs().max().clamp_min(1e-30)) for p, n in zip(outs["peer"], outs["nccl"])]
        if rank == 0:
            res = {"B_global": b, "b_loc": b_loc}
            for name in times:
                res[f"{name}_ms"] = round(statistics.median(times[name]), 4)
                res[f"{name}_ms_spread"] = [round(min(times[name]), 4), round(max(times[name]), 4)]
            res["peer_saves_us"] = round(1000 * (res["nccl_ms"] - res["peer_ms"]), 1)
            res["max_rel_diff_loss_gz_gmu_glv"] = [f"{x:.2e}" for x in diffs]
            print(json.dumps(res), flush=True)
        torch.cuda.synchronize()
        dist.barrier()
        del exch
    sys.stdout.flush()
    os._exit(0)                          # as tools/check_sharded.py: skip the symmetric-memory / NCCL teardown at exit


if __name__ == "__main__":
    main()
