"""The Soft-Intro-TC update as two captured CUDA graphs (SURVEY.md 8f rank 3).

The reference's ``IntroSolver.train_step`` (solvers/intro.py:56-196) cannot be captured: it reads five scalars back to the
host (``.item()`` at :112-115, :155-158, :190-196), branches on ``torch.isnan`` (:162) and clips with a host-side norm.
At the reference's training batch (64) the step is launch-bound, so this module restates the same update in a form with no
host synchronisation at all:

* ``__call__(real, noise)`` copies the batch into static buffers, replays the encoder-phase graph and the decoder-phase
  graph, and returns the step's scalars as DEVICE tensors (read them whenever convenient; ``check_finite()`` does the
  reference's NaN test on demand);
* each phase is ``forward -> losses -> zero_grad -> backward -> [gradient all-reduce] -> clip -> Adam step`` with every
  loss term on the library's kernels: ``reparameterize``, the fused ``(beta-1)*TC + KL`` mean (solvers/tc.py:69-89), the
  per-sample reconstruction loss (ops.py:188-236) and the exp-ELBO terms with the TC loss folded in
  (solvers/intro.py:84-103, one fused evaluation per batch);
* ``kl_loss="full"`` trains with the beta-TCVAE decomposition ``mi + beta*tc + dimkl`` (``TCSovler._compute_kl_loss_full``,
  solvers/tc.py:91-144) instead of the simple ``(beta-1)*TC + KL``: the KL means and the exp-ELBO terms then run on the fused
  decomposition, and ``out`` also carries the encoder phase's ``mi`` / ``tc`` / ``dimkl`` means of the real batch (what the
  reference writes to ``tc_decomp``);
* data parallel: pass ``group`` -- the TC estimator is row-sharded over it (``exchange`` selects NCCL or the peer-memory
  kernels) and parameter gradients are averaged with one flattened all-reduce per phase, captured inside the graphs;
  ``SyncBatchNorm`` conversion is the caller's choice (``torch.nn.SyncBatchNorm.convert_sync_batchnorm``).

The optimizers must be ``capturable`` (``torch.optim.Adam(..., capturable=True)``).  The conv encoder / decoder stay the
caller's torch modules; ``model`` needs the reference's interface (models.py:301-355: ``encode``, ``decode``, ``sample``,
``decoder``, ``encoder``, ``cdim``, ``encoder.image_size``) and must call ``intro_tc_vae_b200.ops.reparameterize`` in its
``forward`` (which it does after ``intro_tc_vae_b200.install()``).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
from torch import Tensor
from torch._utils import _flatten_dense_tensors, _unflatten_dense_tensors

from . import ops
from .losses import exp_elbo, kl_tc_exp_elbo, reconstruction_loss, tc_decomp_exp_elbo


class SoftIntroTCStep:
    def __init__(self, model, optimizer_e, optimizer_d, dataset_size: int, batch_shape, *, recon_loss_type: str = "mse",
                 beta_kl: float = 1.0, beta_rec: float = 1.0, beta_neg: float = 256.0, gamma_r: float = 1e-8,
                 clip: Optional[float] = None, group=None, exchange=None, capture: bool = True, warmup: int = 3,
                 kl_loss: str = "simple"):
        if kl_loss not in ("simple", "full"):
            raise ValueError(f"kl_loss must be 'simple' or 'full', got {kl_loss!r}")
        self.kl_loss = kl_loss
        self.model, self.opt_e, self.opt_d = model, optimizer_e, optimizer_d
        self.n = int(dataset_size)
        self.kind = recon_loss_type
        self.beta_kl, self.beta_rec, self.beta_neg, self.gamma_r = float(beta_kl), float(beta_rec), float(beta_neg), float(gamma_r)
        self.clip = clip
        self.group, self.exchange = group, exchange
        self.world = 1
        if group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(group)
        self.scale = 1.0 / (model.cdim * model.encoder.image_size ** 2)           # solvers/vae.py:61
        dev = next(model.parameters()).device
        self.real = torch.zeros(tuple(batch_shape), device=dev)
        self.noise = torch.zeros(batch_shape[0], model.zdim, device=dev)
        self.out: Dict[str, Tensor] = {}
        self._z: Optional[Tensor] = None
        self.graph_e = self.graph_d = None
        if capture:
            for opt in (optimizer_e, optimizer_d):
                if not all(g.get("capturable", False) for g in opt.param_groups):
                    raise ValueError("SoftIntroTCStep(capture=True) needs optimizers built with capturable=True")
            snapshot = self._snapshot()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(max(warmup, 1)):
                    self._phase_e()
                    self._phase_d()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph_e = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_e):
                self._phase_e()
            self.graph_d = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_d, pool=self.graph_e.pool()):
                self._phase_d()
            self._restore(snapshot)            # warm-up and capture ran real updates: put weights, BN statistics and Adam state back

    # ---- warm-up must not consume training steps ------------------------------------------------------------------
    def _state_tensors(self):
        ts = list(self.model.parameters()) + list(self.model.buffers())
        for opt in (self.opt_e, self.opt_d):
            for st in opt.state.values():
                ts += [v for v in st.values() if torch.is_tensor(v)]
        return ts

    def _snapshot(self):
        return [(t, t.detach().clone()) for t in self._state_tensors()]

    def _restore(self, snapshot) -> None:
        known = {id(t) for t, _ in snapshot}
        with torch.no_grad():
            for t, saved in snapshot:
                t.copy_(saved)
            for t in self._state_tensors():    # optimizer state created during the warm-up (exp_avg, exp_avg_sq, step): back to its initial zeros,
                if id(t) not in known:         # in place -- the graphs hold these tensors' addresses
                    t.zero_()
            for p in self.model.parameters():  # gradients left by the warm-up: zero (the reference's first clip sees none)
                if p.grad is not None:
                    p.grad.zero_()

    # ---- pieces -------------------------------------------------------------------------------------------------
    def _trainable(self, encoder: bool) -> None:
        for p in self.model.encoder.parameters():
            p.requires_grad = encoder
        for p in self.model.decoder.parameters():
            p.requires_grad = not encoder

    def _kl_mean(self, z: Tensor, mu: Tensor, logvar: Tensor, record: bool = False) -> Tensor:
        """compute_kl_loss(z, mu, logvar) of the TC solver with the default reduce="mean" (solvers/tc.py:58-144); with
        kl_loss="full" and ``record``, the mi / tc / dimkl means go to ``out`` as the reference's tc_decomp scalars."""
        if self.kl_loss == "simple":
            return ops.kl_tc_loss_mean(z, mu, logvar, self.n, self.beta_kl, "mss", self.group, self.exchange)[0]
        loss, mi, tc, dimkl = ops.tc_decomp_loss_mean(z, mu, logvar, self.n, self.beta_kl, "mss", self.group, self.exchange)
        if record:
            self.out.update(mi=mi.detach(), tc=tc.detach(), dimkl=dimkl.detach())
        return loss

    def _exp_elbo(self, x: Tensor, recon: Tensor, z: Tensor, mu: Tensor, logvar: Tensor) -> Tensor:
        """mean_i exp(-2*scale*(beta_rec*rec_i + kl_i)), kl_i = compute_kl_loss(reduce="none", beta=beta_neg)  (solvers/intro.py:84-103)."""
        rec_rows = self.beta_rec * reconstruction_loss(x, recon, self.kind, "none")
        full = self.kl_loss == "full"
        if self.world == 1:
            fused = tc_decomp_exp_elbo if full else kl_tc_exp_elbo
            return fused(z, mu, logvar, rec_rows, self.n, self.beta_neg, self.scale)[0]
        terms = ops.tc_decomp_loss_terms if full else ops.kl_tc_loss_terms
        kl_rows = terms(z, mu, logvar, self.n, self.beta_neg, "mss", self.group, self.exchange)[0]
        return exp_elbo(rec_rows, kl_rows, self.scale)

    def _finish(self, loss: Tensor, optimizer, params, tag: str) -> None:
        optimizer.zero_grad(set_to_none=False)             # in place: the other phase's graph clips over these same .grad tensors
        loss.backward()
        if self.world > 1:                                 # data parallel: one flattened all-reduce of this phase's gradients
            import torch.distributed as dist
            grads = [p.grad for p in params if p.grad is not None]
            flat = _flatten_dense_tensors(grads)
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
            flat.div_(self.world)
            for g, f in zip(grads, _unflatten_dense_tensors(flat, grads)):
                g.copy_(f)
        if self.clip:                                      # over ALL parameters, like solvers/intro.py:112-115 (stale grads of the frozen half included)
            self.out["norm_" + tag] = torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.clip, foreach=True)
        optimizer.step()

    # ---- the two phases (solvers/intro.py:65-116 and 118-160) -------------------------------------------------------
    def _phase_e(self) -> None:
        m, real, noise = self.model, self.real, self.noise
        self._trainable(encoder=True)
        fake = m.sample(noise)
        mu, logvar = m.encode(real)
        z = ops.reparameterize(mu, logvar)
        rec = m.decoder(z)
        loss_rec = self.beta_rec * reconstruction_loss(real, rec, self.kind, "mean")
        loss_kl = self._kl_mean(z, mu, logvar, record=True)
        rec_mu, rec_lv, z_rec, rec_rec = m(rec.detach())
        fake_mu, fake_lv, z_fake, rec_fake = m(fake.detach())
        ee_rec = self._exp_elbo(rec, rec_rec, z_rec, rec_mu, rec_lv)
        ee_fake = self._exp_elbo(fake, rec_fake, z_fake, fake_mu, fake_lv)
        loss_e = self.scale * (loss_rec + loss_kl) + 0.25 * (ee_rec + ee_fake)
        self._finish(loss_e, self.opt_e, list(m.encoder.parameters()), "e")
        self._z = z.detach()
        self.out.update(loss_enc=loss_e.detach(), loss_kl=loss_kl.detach(), expelbo_fake=ee_fake.detach())

    def _phase_d(self) -> None:
        m, real, noise = self.model, self.real, self.noise
        self._trainable(encoder=False)
        fake = m.sample(noise)
        rec = m.decoder(self._z)
        loss_rec = self.beta_rec * reconstruction_loss(real, rec, self.kind, "mean")
        rec_mu, rec_lv = m.encode(rec)
        z_rec = ops.reparameterize(rec_mu, rec_lv)
        fake_mu, fake_lv = m.encode(fake)
        z_fake = ops.reparameterize(fake_mu, fake_lv)
        rec_rec = m.decode(z_rec.detach())
        rec_fake = m.decode(z_fake.detach())
        gamma = self.gamma_r * self.beta_rec
        loss_rec_rec = gamma * reconstruction_loss(rec.detach(), rec_rec, self.kind, "mean")
        loss_fake_rec = gamma * reconstruction_loss(fake.detach(), rec_fake, self.kind, "mean")
        kl_rec = self._kl_mean(z_rec, rec_mu, rec_lv)
        kl_fake = self._kl_mean(z_fake, fake_mu, fake_lv)
        loss_d = self.scale * (loss_rec + 0.5 * (kl_rec + kl_fake) + 0.5 * (loss_rec_rec + loss_fake_rec))
        self._finish(loss_d, self.opt_d, list(m.decoder.parameters()), "d")
        self.out.update(loss_dec=loss_d.detach(), loss_rec=loss_rec.detach(), diff_kl=(kl_fake - self.out["loss_kl"]).detach())

    # ---- public ---------------------------------------------------------------------------------------------------
    def __call__(self, real: Tensor, noise: Tensor) -> Dict[str, Tensor]:
        """One update on ``real`` [B,C,H,W] with the fake-batch latents ``noise`` [B,zdim] (solvers/intro.py:61 draws them with
        ``torch.randn`` on the host).  Returns device scalars: loss_enc, loss_dec, loss_kl, loss_rec, expelbo_fake, diff_kl,
        norm_e / norm_d (with ``clip``), mi / tc / dimkl (with kl_loss="full")."""
        self.real.copy_(real, non_blocking=True)
        self.noise.copy_(noise, non_blocking=True)
        if self.graph_e is not None:
            self.graph_e.replay()
            self.graph_d.replay()
        else:
            self._phase_e()
            self._phase_d()
        return self.out

    def check_finite(self) -> None:
        """solvers/intro.py:162-163 on demand (one host synchronisation)."""
        if bool(torch.isnan(self.out["loss_enc"]) | torch.isnan(self.out["loss_dec"])):
            raise RuntimeError("NaN loss")
