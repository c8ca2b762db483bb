"""TC loss composition behind the reference's solver signatures (reference ``solvers/tc.py:58-144``).

``TCLossMixin`` carries the three loss methods of ``TCSovler``; :func:`intro_tc_vae_b200.install` grafts them onto the
reference's own ``solvers.tc.TCSovler`` (whose ``compute_kl_loss`` dispatches to ``self._compute_kl_loss_simple`` and which
``solvers.intro_tc.IntroTCSovler`` forwards to, solvers/intro_tc.py:8-17), so the reference's ``train_step`` code runs
unchanged on top of the fused kernels.  The methods only read ``self.beta_kl``, ``len(self.dataset)`` and
``self.write_scalar``; this package ships no copy of the reference's solver classes.
"""
from __future__ import annotations

from typing import Optional

from torch import Tensor

from .. import ops
from .. import utils as _utils


class _WriterView:
    """``writer`` / ``cur_iter`` of the process-wide holder; the reference's class has no defaults (train.py:100-103,212 assign
    them before the first step), so a holder nobody has set up yet reads as "no writer, iteration 0"."""

    def __init__(self, holder):
        self.writer = getattr(holder, "writer", None)
        self.cur_iter = getattr(holder, "cur_iter", 0)


def _singleton_writer() -> _WriterView:
    """The writer holder the training driver updates: the reference's ``utils.SingletonWriter`` after
    :func:`intro_tc_vae_b200.install`, this package's otherwise."""
    return _WriterView(_utils.SingletonWriter())


def _sharding_of(solver, z: Tensor):
    """(process_group, peer_exchange) for a batch: the exchange only serves the shard shape it was built for; any other shape
    (e.g. a ragged last batch) falls back on the process group, and without one the call raises rather than silently run the
    estimator unsharded on the local rows."""
    group = getattr(solver, "process_group", None)
    exch = getattr(solver, "peer_exchange", None)
    if exch is not None and tuple(z.shape) != (exch.b_loc, exch.d):
        if group is None:
            raise RuntimeError(
                f"tcelbo: batch shape {tuple(z.shape)} does not match the peer exchange ({exch.b_loc}, {exch.d}) and no "
                "process_group is set to fall back on: the estimator would silently run unsharded on the local rows")
        exch = None                                                  # NCCL path
    return group, exch


class TCLossMixin:
    process_group = None          # set to a torch.distributed group to row-shard the estimator (SURVEY.md 8e)
    peer_exchange = None          # optionally a peer.PeerExchange for that group and shard shape: the all-gather /
                                  # reduce-scatter of both losses then run inside the library's kernels over NVLink

    def compute_kl_loss(self, z: Optional[Tensor], mu: Tensor, logvar: Tensor, reduce: str = "mean",
                        beta: float = None, write: bool = False) -> Tensor:
        """solvers/tc.py:58-67: dispatches to the 'simple' form (the only one the reference calls)."""
        return TCLossMixin._compute_kl_loss_simple(self, z, mu, logvar, reduce, beta, write)

    def _compute_kl_loss_simple(self, z: Optional[Tensor], mu: Tensor, logvar: Tensor, reduce: str = "mean",
                                beta: float = None, write: bool = False) -> Tensor:
        """solvers/tc.py:69-89: ``(beta - 1) * TC + KL``; an explicit ``beta=0.0`` is honoured."""
        if beta is None:
            beta = self.beta_kl
        dataset_size = len(self.dataset)
        group, exch = _sharding_of(self, z)
        if reduce == "mean":                                         # mean((b-1)*tc + kl) == (b-1)*mean(tc) + mean(kl)
            loss, kl = ops.kl_tc_loss_mean(z, mu, logvar, dataset_size, beta, "mss", group, exch)
        else:
            # one fused op: per-sample (beta-1)*tc_i + kl_i and kl_i (KL and the combine ride in the TC kernels' epilogues)
            loss, kl, _, _ = ops.kl_tc_loss_terms(z, mu, logvar, dataset_size, beta, "mss", group, exch)
        if write:                                                    # KL only, as in the reference (solvers/tc.py:87-88)
            kl_loss = kl if reduce == "mean" else (kl.sum() if reduce == "sum" else kl)
            self.write_scalar(_singleton_writer().cur_iter, "kl_loss_unscaled", kl_loss)
        if reduce == "sum":                                          # kl summed, tc per sample (ops.py:86-89 treats "sum" as none)
            return (loss - kl) + kl.sum()
        return loss

    def _compute_kl_loss_full(self, z: Optional[Tensor], mu: Tensor, logvar: Tensor, reduce: str = "mean",
                              beta: float = None, write: bool = False) -> Tensor:
        """solvers/tc.py:91-144: MI + beta * TC + dimension-wise KL, column-variance density, MSS.  One fused op: the row
        densities, the combine and (for reduce="mean") the batch means ride in the TC kernels' finalize steps."""
        if beta is None:
            beta = self.beta_kl
        dataset_size = len(self.dataset)
        group, exch = _sharding_of(self, z)
        sw = _singleton_writer()
        if reduce == "mean":
            loss, mi_loss, tc_loss, kl_loss = ops.tc_decomp_loss_mean(z, mu, logvar, dataset_size, beta, "mss", group, exch)
            if sw.writer:
                sw.writer.add_scalars(
                    "tc_decomp",
                    {"mi": mi_loss.data.item(), "tc": tc_loss.data.item(), "kl": kl_loss.data.item()},
                    global_step=sw.cur_iter)
        else:
            loss, mi_loss, tc_loss, kl_loss = ops.tc_decomp_loss_terms(z, mu, logvar, dataset_size, beta, "mss", group, exch)
        if write:
            self.write_scalar(sw.cur_iter, "kl_loss_unscaled", mi_loss + tc_loss + kl_loss)
        return loss
