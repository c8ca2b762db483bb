"""Row-sharded MI / TC / dimension-wise KL decomposition over two exchanges vs the same global batch on one GPU (torchrun,
>= 2 GPUs):

  * NCCL-sharded (tc_decomp_loss_terms(..., group=...)) == peer-sharded (..., exchange=...) == single GPU, per-row terms
    and gradients of mu / logvar, three rounds on one PeerExchange (buffer rotation);
  * the simple loss (kl_tc_loss_terms(..., exchange=...)) interleaved with the decomposition on that same exchange;
  * TCLossMixin._compute_kl_loss_full through a solver that sets only peer_exchange (no process_group).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 tools/check_decomp_peer.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from intro_tc_vae_b200 import ops, peer
from intro_tc_vae_b200.solvers.tc import TCLossMixin


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def leaves(*ts):
    return [t.clone().requires_grad_(True) for t in ts]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD
    ok = True

    def report(tag, errs, tol):
        nonlocal ok
        good = all(e < t for e, t in zip(errs, tol))
        ok = ok and good
        print(f"rank {rank} {tag}: " + "  ".join(f"{e:.1e}" for e in errs) + f"  {'OK' if good else 'MISMATCH'}", flush=True)

    for B, D, N, beta in ((256, 128, 16704, 6.0), (1024, 128, 16704, 0.5), (296, 20, 5000, 4.0), (296, 22, 5000, 4.0)):
        b_loc = B // world
        rows = slice(rank * b_loc, (rank + 1) * b_loc)
        exch = peer.PeerExchange(b_loc, D, group, dev)
        for rnd in range(3):
            g = torch.Generator().manual_seed(B + D + 17 * rnd)
            mu_c = torch.randn(B, D, generator=g)
            lv_c = -2.0 + torch.randn(B, D, generator=g)
            eps_c = torch.randn(B, D, generator=g)
            w = [torch.linspace(a, b, B, device=dev) for a, b in ((0.5, 1.5), (-0.3, 0.8), (1.1, 0.2), (0.4, -0.6))]
            # single GPU, whole batch (every rank does it redundantly)
            mu_f, lv_f = leaves(mu_c.to(dev), lv_c.to(dev))
            z_f = ops.reparameterize(mu_f, lv_f, eps_c.to(dev))
            out_f = ops.tc_decomp_loss_terms(z_f, mu_f, lv_f, N, beta)
            sum((o * wk).sum() for o, wk in zip(out_f, w)).backward()
            res = {}
            for how in ("nccl", "peer"):
                mu, lv = leaves(mu_c[rows].to(dev), lv_c[rows].to(dev))
                z = ops.reparameterize(mu, lv, eps_c[rows].to(dev))
                kw = dict(group=group) if how == "nccl" else dict(exchange=exch)
                out = ops.tc_decomp_loss_terms(z, mu, lv, N, beta, **kw)
                sum((o * wk[rows]).sum() for o, wk in zip(out, w)).backward()
                res[how] = (out, mu.grad, lv.grad)
                errs = [rel(o.detach(), r.detach()[rows]) for o, r in zip(out, out_f)]
                errs += [rel(mu.grad, mu_f.grad[rows]), rel(lv.grad, lv_f.grad[rows])]
                report(f"decomp {how} B={B} D={D} round {rnd} (loss mi tc dimkl dmu dlv)", errs, [2e-6] * 4 + [1e-5] * 2)
            (o_n, gm_n, gl_n), (o_p, gm_p, gl_p) = res["nccl"], res["peer"]
            report(f"decomp peer-vs-nccl B={B} D={D} round {rnd} (loss dmu dlv)",
                   [rel(o_p[0].detach(), o_n[0].detach()), rel(gm_p, gm_n), rel(gl_p, gl_n)], [2e-6, 1e-5, 1e-5])
            # the simple loss on the same exchange, between two decomposition rounds
            mu_f, lv_f = leaves(mu_c.to(dev), lv_c.to(dev))
            out_f = ops.kl_tc_loss_terms(ops.reparameterize(mu_f, lv_f, eps_c.to(dev)), mu_f, lv_f, N, beta)
            sum((o * wk).sum() for o, wk in zip(out_f, w)).backward()
            mu, lv = leaves(mu_c[rows].to(dev), lv_c[rows].to(dev))
            out = ops.kl_tc_loss_terms(ops.reparameterize(mu, lv, eps_c[rows].to(dev)), mu, lv, N, beta, exchange=exch)
            sum((o * wk[rows]).sum() for o, wk in zip(out, w)).backward()
            report(f"simple peer B={B} D={D} round {rnd} (loss dmu dlv)",
                   [rel(out[0].detach(), out_f[0].detach()[rows]), rel(mu.grad, mu_f.grad[rows]), rel(lv.grad, lv_f.grad[rows])],
                   [2e-6, 1e-5, 1e-5])

        # the solver with only peer_exchange set: every rank's local mean, and the gradients of their sum
        class Solver(TCLossMixin):
            process_group = None
            peer_exchange = exch
            beta_kl = beta
            dataset = range(N)

            def write_scalar(self, *args):
                pass

        g = torch.Generator().manual_seed(B * 3 + D)
        mu_c, lv_c, eps_c = torch.randn(B, D, generator=g), -2.0 + torch.randn(B, D, generator=g), torch.randn(B, D, generator=g)
        mu_f, lv_f = leaves(mu_c.to(dev), lv_c.to(dev))
        loss_f = ops.tc_decomp_loss_terms(ops.reparameterize(mu_f, lv_f, eps_c.to(dev)), mu_f, lv_f, N, beta)[0]
        sum(loss_f[r * b_loc:(r + 1) * b_loc].mean() for r in range(world)).backward()
        mu, lv = leaves(mu_c[rows].to(dev), lv_c[rows].to(dev))
        loss = Solver()._compute_kl_loss_full(ops.reparameterize(mu, lv, eps_c[rows].to(dev)), mu, lv)
        loss.backward()
        report(f"solver peer_exchange only B={B} D={D} (loss dmu dlv)",
               [rel(loss.detach().reshape(1), loss_f.detach()[rows].mean().reshape(1)), rel(mu.grad, mu_f.grad[rows]),
                rel(lv.grad, lv_f.grad[rows])], [2e-6, 1e-5, 1e-5])
        torch.cuda.synchronize()
        dist.barrier()
        del exch

    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res = int(flag.item())
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    os._exit(0 if res == 1 else 1)       # as tools/check_sharded.py: skip the symmetric-memory / NCCL teardown at exit


if __name__ == "__main__":
    main()
