"""Time the MI / TC / dimension-wise KL loss of solvers/tc.py:91-144 (reduce="mean", forward + backward) two ways:

    composition  ops.row_log_density twice + ops.tc_terms(var_of="col") + torch subtractions, means and combine
    fused        ops.tc_decomp_loss_mean (tcelbo::decomp_forward / decomp_backward)

Both take the same seeded z, mu, logvar (z a leaf, so no reparameterize is timed) and end in torch.autograd.grad with respect
to all three.  The two are timed alternately, in rounds, with CUDA events around `--iters` steps each; the median step time of
the rounds is reported.  The library's launches per step come from tcelbo_launch_count.  Prints one JSON line per batch size
plus one line naming the GPU and its power limit; needs a CUDA device.

    python tools/decomp_bench.py [--sizes 64,1024,8192] [--d 128] [--iters 20] [--rounds 5] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from intro_tc_vae_b200 import _lib, ops  # noqa: E402

N_DATA = 16704
BETA = 6.0


def _power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def composition(z, mu, lv):
    condx = ops.row_log_density(z, mu, lv)
    pz = ops.row_log_density(z)
    prod, joint = ops.tc_terms(z, mu, lv, N_DATA, "mss", "col")
    mi, tc, dimkl = (condx - joint).mean(), (joint - prod).mean(), (prod - pz).mean()
    return mi + BETA * tc + dimkl


def fused(z, mu, lv):
    return ops.tc_decomp_loss_mean(z, mu, lv, N_DATA, BETA, "mss")[0]


def step(fn, z, mu, lv):
    loss = fn(z, mu, lv)
    return (loss,) + torch.autograd.grad(loss, [z, mu, lv])


def time_steps(fn, inputs, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        step(fn, *inputs)
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
        raise SystemExit("decomp_bench: no CUDA device; these timings only mean something on the GPU")
    lib = _lib.load()
    dev = torch.device("cuda:0")
    print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "power_limit": _power_limit(), "d": args.d,
                      "iters_per_round": args.iters, "rounds": args.rounds}), flush=True)
    for b in (int(s) for s in args.sizes.split(",")):
        g = torch.Generator().manual_seed(b)
        mu_c = torch.randn(b, args.d, generator=g)
        lv_c = -2.0 + torch.randn(b, args.d, generator=g)
        z_c = mu_c + torch.randn(b, args.d, generator=g) * torch.exp(0.5 * lv_c)
        inputs = [t.to(dev).requires_grad_(True) for t in (z_c, mu_c, lv_c)]
        res = {"B": b}
        outs = {}
        for name, fn in (("composition", composition), ("fused", fused)):
            for _ in range(args.warmup):
                step(fn, *inputs)
            torch.cuda.synchronize()
            n0 = lib.tcelbo_launch_count()
            outs[name] = [t.detach() for t in step(fn, *inputs)]
            res[f"{name}_launches"] = lib.tcelbo_launch_count() - n0
        times = {"composition": [], "fused": []}
        for _ in range(args.rounds):                                  # alternate, so that drift hits both alike
            for name, fn in (("composition", composition), ("fused", fused)):
                times[name].append(time_steps(fn, inputs, args.iters))
        for name in times:
            res[f"{name}_ms"] = round(statistics.median(times[name]), 4)
            res[f"{name}_ms_spread"] = [round(min(times[name]), 4), round(max(times[name]), 4)]
        res["speedup"] = round(res["composition_ms"] / res["fused_ms"], 3)
        diffs = [float((a - c).abs().max() / c.abs().max().clamp_min(1e-30)) for a, c in zip(outs["fused"], outs["composition"])]
        res["max_rel_diff_loss_gz_gmu_glv"] = [f"{x:.2e}" for x in diffs]
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
