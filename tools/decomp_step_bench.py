"""Time one training step of the MI / TC / dimension-wise KL loss of solvers/tc.py:91-144 (reduce="mean") from the encoder
outputs: z = mu + eps * exp(logvar / 2), the loss, and its gradients w.r.t. mu and logvar.  Three variants:

    eager     ops.reparameterize -> ops.tc_decomp_loss_mean -> backward, issued from Python on every step
    autograd  GraphedKLLoss(loss="decomp", mode="autograd"): the same step captured in a CUDA graph and replayed
    direct    GraphedKLLoss(loss="decomp"): tcelbo_decomp_forward_ex / _backward_ex with the fused reparameterize, replayed

All three take the same seeded mu, logvar, eps.  They are timed alternately, in rounds, with CUDA events around `--iters` steps
each; the median step time of the rounds is reported, with the library's launches per step (tcelbo_launch_count of one
un-captured step).  Prints one line naming the GPU and its power limit, then one JSON line per batch size; needs a CUDA device.

    python tools/decomp_step_bench.py [--sizes 64,1024,8192] [--d 128] [--iters 20] [--rounds 5] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from decomp_bench import _power_limit  # noqa: E402
from intro_tc_vae_b200 import _lib, ops  # noqa: E402
from intro_tc_vae_b200.graphs import GraphedKLLoss  # noqa: E402

N_DATA = 16704
BETA = 6.0
VARIANTS = ("eager", "autograd", "direct")


def eager_step(mu, logvar, eps):
    """The unfused step with fresh leaves, as a user's training loop issues it."""
    mu, logvar = mu.detach().requires_grad_(True), logvar.detach().requires_grad_(True)
    z = ops.reparameterize(mu, logvar, eps)
    loss = ops.tc_decomp_loss_mean(z, mu, logvar, N_DATA, BETA, "mss")[0]
    loss.backward()
    return loss.detach(), mu.grad, logvar.grad


def time_steps(fn, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / iters


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", default="64,1024,8192")
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decomp_step_bench: no CUDA device; these timings only mean something on the GPU")
    lib = _lib.load()
    dev = torch.device("cuda:0")
    print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "power_limit": _power_limit(), "d": args.d,
                      "iters_per_round": args.iters, "rounds": args.rounds}), flush=True)
    for b in (int(s) for s in args.sizes.split(",")):
        g = torch.Generator().manual_seed(b)
        mu = torch.randn(b, args.d, generator=g).to(dev)
        lv = (-2.0 + torch.randn(b, args.d, generator=g)).to(dev)
        eps = torch.randn(b, args.d, generator=g).to(dev)
        graphed = {m: GraphedKLLoss(b, args.d, N_DATA, BETA, dev, mode=m, loss="decomp", warmup=args.warmup)
                   for m in ("autograd", "direct")}
        counting = {m: GraphedKLLoss(b, args.d, N_DATA, BETA, dev, mode=m, loss="decomp", capture=False, warmup=1)
                    for m in ("autograd", "direct")}
        for gr in graphed.values():                                       # static inputs, copied once: replays time the step only
            gr(mu, lv, eps)
        run = {"eager": lambda: eager_step(mu, lv, eps), "autograd": graphed["autograd"].replay, "direct": graphed["direct"].replay}
        res = {"B": b}
        outs = {}
        count = {"eager": run["eager"], "autograd": counting["autograd"].replay, "direct": counting["direct"].replay}
        for name in VARIANTS:
            for _ in range(args.warmup):
                run[name]()
            torch.cuda.synchronize()
            outs[name] = [t.detach().clone() for t in run[name]()]
            n0 = lib.tcelbo_launch_count()
            count[name]()                                                 # one un-captured step: what a replay launches
            res[f"{name}_tcelbo_launch_count"] = lib.tcelbo_launch_count() - n0
        times = {name: [] for name in VARIANTS}
        for _ in range(args.rounds):                                      # alternate, so that drift hits all three alike
            for name in VARIANTS:
                times[name].append(time_steps(run[name], args.iters))
        for name in VARIANTS:
            res[f"{name}_ms"] = round(statistics.median(times[name]), 4)
            res[f"{name}_ms_spread"] = [round(min(times[name]), 4), round(max(times[name]), 4)]
        ref = outs["eager"]
        for name in ("autograd", "direct"):
            res[f"{name}_max_rel_diff_loss_dmu_dlv"] = [
                f"{float((a - c).abs().max() / c.abs().max().clamp_min(1e-30)):.2e}" for a, c in zip(outs[name], ref)]
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
