#!/usr/bin/env python
"""Benchmark of the TC-ELBO hot path (BASELINE.json metric: "TC-ELBO fwd+bwd log-densities/s (B^2*D)").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--zdim D] [--dump-outputs DIR]

A "step" is one compute_kl_loss-equivalent evaluation (SURVEY.md 8d): reparameterize + KL + TC
(minibatch stratified sampling) + (beta-1)*TC + KL, mean-reduced, and its backward to mu / logvar.
Workload at every N: BASELINE configs[2] at the size the north-star target is quoted on -- synthetic
latents, GLOBAL batch 8192, z_dim 128 (strong scaling: rank r owns rows [r*B/N, (r+1)*B/N), mu is
all-gathered over NCCL before the sweep and its gradient reduce-scattered after it).

Prints ONE JSON line on rank 0 (see the keys below).  `--impl reference` times the reference's own CPU implementation on the
host cores: the unmodified ops.py staged under oracle/_ref by __graft_entry__.build() (the oracle port if that is absent).

`--dump-outputs DIR` writes what the last timed step returned -- loss.npy (one entry per rank), grad_mu.npy and
grad_logvar.npy ([B, D], rows in global order), all float32 -- so that two builds can be compared output for output on
the same seeded inputs.  Gradients that would exceed 64 MB are reduced to a fixed seeded sample of rows, whose indices go to
rows.npy.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "tc_elbo_fwd_bwd_log_densities_per_s"
UNIT = "log-densities/s"
DATASET_SIZE = 16704          # UkiyoE-sized N (SURVEY.md 8d)
BETA = 0.5
CPU_SAMPLE_B = 1024           # bounded CPU sample: B=1024, D=128 (the reference keeps 4*B^2*D*4 bytes = 2 GiB for backward)
DUMP_BYTES = 64 * 10**6       # --dump-outputs budget


def synthetic_latents(b, d, seed=1234):
    """mu ~ N(0,1), logvar ~ N(-2,1), eps ~ N(0,1): about 5 % of the log-densities hit the -50 clamp."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    mu = torch.randn(b, d, generator=g)
    lv = -2.0 + torch.randn(b, d, generator=g)
    eps = torch.randn(b, d, generator=g)
    return mu, lv, eps


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_impl():
    """(module, kind): the UNMODIFIED reference's ops.py staged under oracle/_ref (kind "reference"; oracle/ref_loader.py
    copies it there wherever /root/reference exists and the copy travels with the snapshot), else the oracle port."""
    from oracle import ref_loader
    if ref_loader.available():
        return ref_loader.load_ops(), "reference"
    from oracle import tc_oracle
    return tc_oracle, "port"


def cpu_step(impl, mu, lv, n, beta):
    """One compute_kl_loss-equivalent step exactly as the reference composes it: reparameterize (ops.py:166-185, draws its own
    eps), kl_divergence + total_correlation -> (beta-1)*tc + kl (solvers/tc.py:83-89), backward.  Returns (fwd_s, bwd_s)."""
    mu = mu.detach().requires_grad_(True)
    lv = lv.detach().requires_grad_(True)
    t0 = time.perf_counter()
    z = impl.reparameterize(mu, lv)
    kl = impl.kl_divergence(lv, mu, reduce="mean")
    tc = impl.total_correlation(z, mu, lv, n, reduce="mean")
    loss = (beta - 1.0) * tc + kl
    loss.item()
    t1 = time.perf_counter()
    loss.backward()
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def time_cpu(b, d, steps, warmup):
    # all the host threads the box offers (torchrun exports OMP_NUM_THREADS=1 to its workers; the baseline must not inherit that)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        torch.set_num_threads(max(1, os.cpu_count() or 1))
    impl, kind = cpu_impl()
    mu, lv, _ = synthetic_latents(b, d)
    for _ in range(warmup):
        cpu_step(impl, mu, lv, DATASET_SIZE, BETA)
    times = [cpu_step(impl, mu, lv, DATASET_SIZE, BETA) for _ in range(steps)]
    return times, kind


def cpu_sample_note(b, d, kind, cores):
    what = ("the UNMODIFIED reference (ops.reparameterize / kl_divergence / total_correlation from the staged oracle/_ref/ops.py)"
            if kind == "reference" else "the oracle port of the reference's op sequence (oracle/tc_oracle.py)")
    return (f"B={b}, D={d}, N={DATASET_SIZE}: reparameterize + kl_divergence + total_correlation + backward, fp32, {what}, "
            f"{cores} torch threads of {os.cpu_count()} cpus; the reference keeps 4*B^2*D*4 bytes for backward (128 GiB at B=8192), "
            "so it is timed on this bounded sample and compared as a rate")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    b, d = CPU_SAMPLE_B, args.zdim
    times, kind = time_cpu(b, d, args.steps, args.warmup)
    t = sum(f + w for f, w in times) / len(times)
    value = b * b * d / t
    cores = torch.get_num_threads()
    # second, larger sample (BASELINE.md section 4 plan): B=2048 keeps 8 GiB for backward; two timed steps bound its cost
    extra = []
    try:
        t2, _ = time_cpu(2 * b, d, 2, 1)
        extra.append({"batch": 2 * b, "fwd_ms": 1e3 * min(f for f, _ in t2), "bwd_ms": 1e3 * min(w for _, w in t2),
                      "value": (2 * b) ** 2 * d / min(f + w for f, w in t2)})
    except Exception as exc:                             # e.g. a host without 8 GiB to spare
        extra.append({"batch": 2 * b, "error": f"{type(exc).__name__}: {exc}"[:120]})
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"tc_microbench (BASELINE configs[2]): global batch 8192, z_dim {d} (timed on a bounded CPU sample: B={b})",
                   "sample_batch": b, "z_dim": d, "dataset_size": DATASET_SIZE, "beta": BETA},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": cpu_sample_note(b, d, kind, cores),
                         "fwd_ms": 1e3 * sum(f for f, _ in times) / len(times), "bwd_ms": 1e3 * sum(w for _, w in times) / len(times),
                         "more_samples": extra},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, smax, power, reasons = [], [], [], set()
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, loss, dmu, dlogvar, world, rank):
    """Write one step's loss and gradients, gathered over the ranks, to out_dir on rank 0 (see --dump-outputs above)."""
    import torch.distributed as dist
    loss = loss.detach().reshape(1)
    if world > 1:
        parts = []
        for t in (loss, dmu, dlogvar):
            out = t.new_empty((world * t.shape[0],) + tuple(t.shape[1:]))
            dist.all_gather_into_tensor(out, t.contiguous())
            parts.append(out)
        loss, dmu, dlogvar = parts
    if rank != 0:
        return
    arrays = {"loss": loss, "grad_mu": dmu, "grad_logvar": dlogvar}
    b, d = dmu.shape
    # per kept row: two float32 gradient rows and a float64 index; 4 KiB for the loss and the .npy headers
    keep = (DUMP_BYTES - 4096 - 4 * world) // (8 * d + 8)
    if b > keep:
        rows = torch.randperm(b, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        idx = rows.to(dmu.device)
        arrays.update(grad_mu=dmu[idx], grad_logvar=dlogvar[idx], rows=rows.double())
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from intro_tc_vae_b200 import _lib, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device: the TC-ELBO path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    lib = _lib.load()

    B, D, N = args.batch, args.zdim, DATASET_SIZE
    if N < B - 1:                  # the stratified weights need N >= B-1 (ops.py:46: log of a negative weight is NaN otherwise)
        N = 4 * B
    assert B % world == 0, "global batch must divide by the number of ranks"
    b_loc = B // world
    lo = rank * b_loc
    mu_c, lv_c, eps_c = synthetic_latents(B, D)
    mu_h = mu_c[lo:lo + b_loc].contiguous().pin_memory()
    lv_h = lv_c[lo:lo + b_loc].contiguous().pin_memory()
    eps_h = eps_c[lo:lo + b_loc].contiguous().pin_memory()
    mu = mu_h.to(dev).requires_grad_(True)
    lv = lv_h.to(dev).requires_grad_(True)
    eps = eps_h.to(dev)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    # the drop-in path: the reference's own call sequence -- reparameterize (ops.py:166), then the solver's
    # compute_kl_loss(z, mu, logvar) with its default reduce="mean" (solvers/tc.py:58-89), then autograd's backward
    from intro_tc_vae_b200.solvers import TCLossMixin

    class _Dataset:
        def __len__(self):
            return N

    class _Solver(TCLossMixin):
        beta_kl = BETA
        dataset = _Dataset()
        process_group = group

        def write_scalar(self, *a, **k):
            pass

    solver = _Solver()

    def step(mu_t, lv_t, eps_t):
        mu_t.grad = None
        lv_t.grad = None
        z = ops.reparameterize(mu_t, lv_t, eps_t)
        loss = solver.compute_kl_loss(z, mu_t, lv_t)
        loss.backward()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- warm-up (eager), then capture the step in a CUDA graph (all ranks take the same branch)
    for _ in range(max(args.warmup, 3)):
        step(mu, lv, eps)
    barrier()
    graphed = None
    graph_note = "eager"
    exchange_note = "nccl" if world > 1 else "none"
    try:
        from intro_tc_vae_b200.graphs import GraphedKLLoss
        graphed = GraphedKLLoss(b_loc, D, N, BETA, dev, group=group, exchange=args.exchange, capture=not args.no_graph)
        exchange_note = graphed.exchange_kind
        graphed(mu.detach(), lv.detach(), eps)
        torch.cuda.synchronize()
        ref_loss = step(mu, lv, eps).item()
        got = graphed.loss.item()
        assert abs(got - ref_loss) <= 1e-5 * abs(ref_loss), (got, ref_loss)
        graph_note = ("cuda-graph replay of" if not args.no_graph else "eager launches of") + \
            " the whole step through the C ABI (tcelbo_klloss_forward_ex / _backward_ex: reparameterize and the batch mean fused, 6 launches)"
    except Exception as exc:                           # capture unsupported here: fall back to eager launches
        graphed = None
        graph_note = f"eager (graph capture failed: {type(exc).__name__}: {exc})"[:200]
    ok = torch.tensor([1 if graphed is not None else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() == 0:
        graphed = None
    if graphed is None:
        exchange_note = "nccl" if world > 1 else "none"
    if world > 1 and exchange_note == "peer":             # the drop-in solver gets its own symmetric buffers (collective construction)
        from intro_tc_vae_b200.peer import PeerExchange
        solver.peer_exchange = PeerExchange(b_loc, D, group, dev)

    def run_step():
        """-> (loss, grad_mu, grad_logvar) of this step."""
        if graphed is not None:
            return graphed.replay()
        return step(mu, lv, eps), mu.grad, lv.grad
    for _ in range(3):
        run_step()
    barrier()

    # ---- timed: K steps, inputs resident in HBM, L2 flushed between steps (outside the event pairs)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = lib.tcelbo_launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        flush_buf.fill_(k & 0xFF)
        starts[k].record()
        outputs = run_step()
        stops[k].record()
    barrier()
    t_wall1 = time.perf_counter()
    launches = lib.tcelbo_launch_count() - launches0
    if args.dump_outputs:                                  # before anything below reruns the step into the same buffers
        dump_outputs(args.dump_outputs, *outputs, world, rank)
    if graphed is not None:                                # replayed launches do not pass through the host-side counter:
        c0 = lib.tcelbo_launch_count()                     # count the kernels of one eager issue of the captured step function
        graphed._step()
        torch.cuda.synchronize()
        launches = (lib.tcelbo_launch_count() - c0) * args.steps
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))
    total_ms = max_over_ranks(dev_ms)
    ms_per_step = total_ms / args.steps
    value = B * B * D / (ms_per_step * 1e-3)

    # ---- e2e: the same step through the public API with HOST buffers (H2D of mu/logvar/eps, D2H of loss + grads)
    gmu_h = torch.empty(b_loc, D).pin_memory()
    glv_h = torch.empty(b_loc, D).pin_memory()
    loss_h = torch.empty(1).pin_memory()

    def e2e_step():
        if graphed is not None:                            # host buffers -> static graph inputs -> replay -> host
            loss, gmu_d, glv_d = graphed(mu_h, lv_h, eps_h)
        else:
            mu_d = mu_h.to(dev, non_blocking=True).requires_grad_(True)
            lv_d = lv_h.to(dev, non_blocking=True).requires_grad_(True)
            eps_d = eps_h.to(dev, non_blocking=True)
            loss = step(mu_d, lv_d, eps_d)
            gmu_d, glv_d = mu_d.grad, lv_d.grad
        gmu_h.copy_(gmu_d, non_blocking=True)
        glv_h.copy_(glv_d, non_blocking=True)
        loss_h.copy_(loss.detach().reshape(1), non_blocking=True)

    for _ in range(3):
        e2e_step()
    barrier()
    e_starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e_stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for k in range(args.steps):
        flush_buf.fill_(k & 0xFF)
        e_starts[k].record()
        e2e_step()
        e_stops[k].record()
    barrier()
    e2e_serial_ms = max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(e_starts, e_stops))) / args.steps

    # The headline e2e streams the same host batches through graphs.HostPipeline: copy-in, step and copy-out on three streams,
    # two batches deep, every step still moving its own inputs and results over PCIe inside the timed region (one event pair
    # around all K steps, the L2 flush writes included).
    from intro_tc_vae_b200.graphs import HostPipeline
    host_out = [(torch.empty(1).pin_memory(), torch.empty(b_loc, D).pin_memory(), torch.empty(b_loc, D).pin_memory()) for _ in range(2)]

    def timed_pipeline(step_fn, check=None):
        """-> (ms per step with the L2 flush writes excluded, ms per step of the whole region).  Per-step event pairs on the
        COMPUTE stream bracket [wait for this batch's copy-in .. its results staged for copy-out] -- a copy that is not hidden
        behind the previous batch's kernels shows up as waiting inside the pair -- plus the final drain of the copy-out stream;
        the flush writes run between the pairs, as in the HBM-resident measurement."""
        pipe = HostPipeline(step_fn, b_loc, D, dev, depth=2)

        def run(n, a0=None, a1=None):
            for k in range(n):
                flush_buf.fill_(k & 0xFF)
                if a0 is not None:
                    a0[k].record()
                pipe.submit(mu_h, lv_h, eps_h, *host_out[k % 2])
                if a1 is not None:
                    a1[k].record()
        run(3)
        pipe.drain()
        barrier()
        a0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        a1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        p0, p1, d0 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        p0.record()
        pipe.begin()
        run(args.steps, a0, a1)
        d0.record()
        pipe.fence()
        p1.record()
        barrier()
        if check is not None:                              # the streamed results are the serial path's results
            lo, gm, gl = host_out[(args.steps - 1) % 2]
            assert abs(lo.item() - check[0]) <= 1e-5 * abs(check[0]), (lo.item(), check[0])
            assert torch.allclose(gm, check[1], rtol=1e-4, atol=1e-5 * float(check[1].abs().max()) + 1e-12)
            assert torch.allclose(gl, check[2], rtol=1e-4, atol=1e-5 * float(check[2].abs().max()) + 1e-12)
        steps_ms = sum(x.elapsed_time(y) for x, y in zip(a0, a1)) + d0.elapsed_time(p1)
        return max_over_ranks(steps_ms) / args.steps, max_over_ranks(p0.elapsed_time(p1)) / args.steps

    serial_result = (loss_h.item(), gmu_h.clone(), glv_h.clone())

    def eager_fn(mu_s, lv_s, eps_s):
        with torch.enable_grad():
            mu_d, lv_d = mu_s.detach().requires_grad_(True), lv_s.detach().requires_grad_(True)
            loss = step(mu_d, lv_d, eps_s)
        return loss, mu_d.grad, lv_d.grad

    e2e_ms, e2e_region_ms = timed_pipeline(graphed if graphed is not None else eager_fn, serial_result)
    e2e_value = B * B * D / (e2e_ms * 1e-3)

    # ---- the same two measurements through the DROP-IN path (eager: reparameterize -> solver.compute_kl_loss -> backward)
    def timed(fn):
        for _ in range(3):
            fn()
        barrier()
        a0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        a1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        for k in range(args.steps):
            flush_buf.fill_(k & 0xFF)
            a0[k].record()
            fn()
            a1[k].record()
        barrier()
        return max_over_ranks(sum(x.elapsed_time(y) for x, y in zip(a0, a1))) / args.steps

    def dropin_e2e_step():
        mu_d = mu_h.to(dev, non_blocking=True).requires_grad_(True)
        lv_d = lv_h.to(dev, non_blocking=True).requires_grad_(True)
        eps_d = eps_h.to(dev, non_blocking=True)
        loss = step(mu_d, lv_d, eps_d)
        gmu_h.copy_(mu_d.grad, non_blocking=True)
        glv_h.copy_(lv_d.grad, non_blocking=True)
        loss_h.copy_(loss.detach().reshape(1), non_blocking=True)

    dropin_ms = timed(lambda: step(mu, lv, eps))
    dropin_e2e_serial_ms = timed(dropin_e2e_step)
    dropin_e2e_ms, dropin_e2e_region_ms = timed_pipeline(eager_fn, serial_result)
    t_region_end = time.perf_counter()
    if rank == 0:
        time.sleep(0.2)
        sampler.stop()
    clocks = sampler.summary(t_wall0, t_region_end) if rank == 0 else {}

    # ---- roofline of the dominant kernels, timed live with CUDA events on the launching stream
    roof = None
    # every rank runs these steps (they contain the collectives); only rank 0 brackets its kernels with events
    cur = torch.cuda.current_stream(dev)
    kern_ms = {}
    for kid, name in ((1, "tc_fwd_kernel"), (2, "tc_bwd_ds_kernel")):
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record(cur); ev1.record(cur)               # materialise the underlying cudaEvent_t handles
        ts = []
        for k in range(min(args.steps, 5)):
            flush_buf.fill_(k)
            if rank == 0:
                _lib.check(lib.tcelbo_profile_events(kid, ev0.cuda_event, ev1.cuda_event), "profile_events")
            step(mu, lv, eps)
            torch.cuda.synchronize()
            if rank == 0:
                lib.tcelbo_profile_events(0, None, None)
                ts.append(ev0.elapsed_time(ev1))
        if rank == 0:
            kern_ms[name] = sum(ts) / len(ts)
    barrier()
    if rank == 0:
        # SFU saturation probe in the same job (empirical ex2 peak)
        scratch = torch.zeros(16, device=dev)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        iters, ctas = 4096, sms * 8
        lib.tcelbo_ex2_peak(scratch.data_ptr(), 64, ctas, cur.cuda_stream)
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        lib.tcelbo_ex2_peak(scratch.data_ptr(), iters, ctas, cur.cuda_stream)
        p1.record()
        torch.cuda.synchronize()
        ex2_measured = ctas * 256 * 8 * iters / (p0.elapsed_time(p1) * 1e-3)
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        peak_nominal = sms * 16 * 1965.0e6                     # 16 MUFU lanes per SM per clock at the max SM clock
        peak_at_clock = sms * 16 * sm_mhz * 1e6
        rows_loc = b_loc
        alg_fwd = rows_loc * B * D + rows_loc * B              # ex2 per forward sweep on this rank
        dom = max(kern_ms, key=kern_ms.get)
        achieved = alg_fwd / (kern_ms[dom] * 1e-3)
        hbm_bytes = 48.0 * B * D                               # SURVEY.md 8d: algorithmic bytes of one evaluation
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic = None                                         # dram bytes per launch of the dominant kernel, from the committed ncu capture
        try:
            import csv
            rows = list(csv.reader(open(os.path.join(ROOT, "profiles", "r2_ncu_full_raw.csv"))))
            hdr, units = rows[0], rows[1]
            ik, ir, iw = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            for r in rows[2:]:
                if dom.replace("_kernel", "") in r[ik]:
                    traffic = float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0)
        except Exception:
            traffic = None
        roof = {
            "bound": "sfu", "kernel": dom, "achieved": achieved / 1e9, "peak": peak_nominal / 1e9, "unit": "Gex2/s",
            "frac": achieved / peak_nominal, "traffic": traffic,
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch of that kernel (bytes, profiles/r2_ncu_full_raw.csv, N=1 shape)",
            "peak_note": "148 SM x 16 MUFU/clk x 1.965 GHz (max SM clock); ex2_measured_gps is the in-job saturation probe",
            "ex2_measured_gps": ex2_measured / 1e9, "frac_of_measured_ex2": achieved / ex2_measured,
            "peak_at_observed_clock_gps": peak_at_clock / 1e9,
            "kernel_ms": kern_ms,
            "kernel_frac_of_sfu_peak": {k: alg_fwd / (v * 1e-3) / peak_nominal for k, v in kern_ms.items()},
            "step_algorithmic_ex2": 2 * B * B * D + 2 * B * B,
            "step_frac_of_sfu_peak": (2 * B * B * D + 2 * B * B) / world / (ms_per_step * 1e-3) / peak_nominal,
            "hbm": {"algorithmic_bytes_per_step": hbm_bytes, "achieved_gbs": hbm_bytes / (ms_per_step * 1e-3) / 1e9,
                    "peak_gbs": hbm_peak, "peak_source": "measured" if peaks else "fallback",
                    "frac": hbm_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak},
        }

    # ---- CPU baseline (rank 0, N == 1 only): bounded sample of the same workload on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times, kind = time_cpu(CPU_SAMPLE_B, D, steps=3, warmup=1)
        t = min(f + w for f, w in times)
        cores = torch.get_num_threads()
        cpu = {"value": CPU_SAMPLE_B * CPU_SAMPLE_B * D / t, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": cpu_sample_note(CPU_SAMPLE_B, D, kind, cores) + ", best of 3",
               "fwd_ms": 1e3 * min(f for f, _ in times), "bwd_ms": 1e3 * min(w for _, w in times)}

    # ---- BASELINE.json metric 2: Soft-Intro-TC train images/s on synthetic images (tools/train_bench.py harness around
    #      intro_tc_vae_b200.train_step.SoftIntroTCStep).  N=1: configs[1] shape (64x64, z 128, batch 64); N>1: configs[4] shape
    #      (128x128, z 256, batch 32 per GPU, data parallel with the TC estimator row-sharded over the ranks).
    train = None
    if not args.no_train:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import train_bench
            if world == 1:
                train = train_bench.measure(64, 128, 64, steps=args.steps, warmup=5, dev=dev)
                train["config"] = "BASELINE configs[1] shape: 64x64x3 synthetic images, conv arch, z_dim 128, batch 64, fp32 (no AMP in the reference)"
            else:
                train = train_bench.measure(128, 256, 32, steps=args.steps, warmup=5, dev=dev, group=group, peer=(exchange_note == "peer"))
                train["config"] = f"BASELINE configs[4] shape: 128x128x3 synthetic images, z_dim 256, beta_neg 512, batch 32 per GPU, data parallel x{world}"
        except Exception as exc:
            train = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        barrier()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"tc_microbench (BASELINE configs[2]): global batch {B}, z_dim {D}, N={N}, beta={BETA}, "
                                   "MSS estimator, row-variance density, fwd+bwd",
                       "global_batch": B, "z_dim": D, "rows_per_gpu": b_loc, "parallelism": f"row-shard x{world}",
                       "l2": "flushed between timed steps by writing a 256 MiB buffer (outside the event pairs)",
                       "launch": graph_note,
                       "exchange": {"none": "none (one GPU)", "nccl": "NCCL all-gather + reduce-scatter",
                                    "peer": "library kernels over NVLink peer memory (gather / reduce-scatter inside the prologue / finalize kernels, "
                                            "in-kernel flag barriers over symmetric memory)"}[exchange_note]},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "serial_ms_per_step": e2e_serial_ms,
                    "region_ms_per_step_incl_l2_flush": e2e_region_ms,
                    "h2d_bytes_per_step": 3 * b_loc * D * 4, "d2h_bytes_per_step": 2 * b_loc * D * 4 + 4,
                    "how": "graphs.HostPipeline: pinned host mu/logvar/eps -> device, graph replay, loss + both gradients -> pinned host, "
                           "every step; copies on side streams two batches deep.  ms_per_step = per-step event pairs on the compute stream "
                           "(from the wait for the batch's copy-in to its results staged for copy-out; the L2 flush writes run between "
                           "the pairs as in the HBM-resident measurement) + the final copy-out drain; region_ms_per_step_incl_l2_flush = "
                           "one event pair around all K steps; serial_ms_per_step = copies and step on one stream"},
            "dropin": {"what": "same step through the reference's signatures: ops.reparameterize -> TCLossMixin.compute_kl_loss(z, mu, logvar) "
                               "-> loss.backward(), eager launches, inputs resident in HBM",
                       "ms_per_step": dropin_ms, "value": B * B * D / (dropin_ms * 1e-3), "unit": UNIT},
            "e2e_dropin": {"value": B * B * D / (dropin_e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": dropin_e2e_ms,
                           "serial_ms_per_step": dropin_e2e_serial_ms, "region_ms_per_step_incl_l2_flush": dropin_e2e_region_ms,
                           "h2d_bytes_per_step": 3 * b_loc * D * 4, "d2h_bytes_per_step": 2 * b_loc * D * 4 + 4},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "train_images_per_s": (train or {}).get("value"),
            "train": train,
            "wall_s_timed_region": t_wall1 - t_wall0,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down of an NCCL communicator that was used inside a captured CUDA graph can block; the numbers are
        # already printed, so synchronise the ranks and leave without running destructors.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="GLOBAL batch (rows are sharded over the ranks)")
    ap.add_argument("--zdim", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the Soft-Intro-TC train images/s leg")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N>1: how the column operand / its gradient cross ranks (peer memory inside the kernels, or NCCL)")
    ap.add_argument("--no-graph", action="store_true", help="issue every step eagerly instead of replaying a captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss and gradients of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
