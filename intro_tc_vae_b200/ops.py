"""Loss helpers of the TC-ELBO path with the reference's call signatures (reference ``ops.py``).

Every function that lies on the hot path runs hand-written sm_100a kernels through the C ABI of
``libtcelbo.so`` (include/tcelbo.h); inputs must be fp32 CUDA tensors -- there is no CPU or eager
fallback.  The B x B x D log-density tensor of ops.py:80-82 is never materialised: the fused op
returns ``(log_qz_prod, log_qz)`` directly and recomputes tiles in backward.

Reference map (file:line in the reference repository):
    total_correlation            ops.py:52-89
    tc_terms                     ops.py:80-84 + 104-115 / 92-101 fused (and solvers/tc.py:114-119 for var_of="col")
    tc_decomp_loss_*             solvers/tc.py:91-144 fused (MI + beta*TC + dimension-wise KL)
    kl_divergence / kl_no_reduce ops.py:136-163   (argument order: logvar, mu)
    reparameterize               ops.py:166-185
    log_importance_weight_matrix ops.py:32-49
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from .losses import reconstruction_loss          # ops.py:188-236 lives in ops in the reference
from .sharding import gather_rows, shard_rows

__all__ = [
    "total_correlation", "tc_terms", "kl_tc_loss_terms", "kl_tc_loss_mean", "tc_decomp_loss_terms", "tc_decomp_loss_mean",
    "reconstruction_loss", "kl_divergence", "kl_no_reduce", "reparameterize",
    "log_importance_weight_matrix", "row_log_density", "gaussian_log_density_torch", "gaussian_log_density",
    "minibatch_stratified_sampling", "minibatch_weighted_sampling",
]


# --------------------------------------------------------------------------------------------------
# argument plumbing
# --------------------------------------------------------------------------------------------------
def _check(name: str, t: Tensor) -> None:
    if not isinstance(t, Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} is on {t.device}: the B200 TC-ELBO path only runs on CUDA tensors (no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} is {t.dtype}: the B200 TC-ELBO path computes in fp32 only")
    if t.dim() != 2:
        raise ValueError(f"{name} must be [batch, latent], got shape {tuple(t.shape)}")


def _rows(t: Tensor) -> Tensor:
    """Row-major with unit inner stride (chunk views with pitch 2*D are passed through untouched)."""
    if t.stride(1) != 1 or t.stride(0) < t.size(1):
        t = t.contiguous()
    return t


def _stream(t: Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _alert_not_deterministic(what: str) -> None:
    """The backward sweeps add per-CTA partial column sums into grad_mu (and grad_logvar of the column-variance variant)
    with fp32 ``red.global.add``: the summation order, hence the last bits (~1e-7 relative), vary from launch to launch,
    whereas the reference's autograd path is deterministic.  Same contract as torch's own non-deterministic ops."""
    if torch.are_deterministic_algorithms_enabled():
        msg = (f"{what} does not have a deterministic implementation (fp32 atomic accumulation of the column gradient), but "
               "torch.use_deterministic_algorithms(True) is set")
        if torch.is_deterministic_algorithms_warn_only_enabled():
            import warnings
            warnings.warn(msg)
        else:
            raise RuntimeError(msg + "; pass warn_only=True to run it anyway")


# --------------------------------------------------------------------------------------------------
# the fused TC op:  torch.ops.tcelbo.tc_forward / tc_backward
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tcelbo::tc_forward", mutates_args=(), device_types="cuda")
def _tc_forward(z: Tensor, mu_all: Tensor, logvar: Tensor, row_offset: int, dataset_size: int,
                flags: int) -> Tuple[Tensor, Tensor, Tensor]:
    lib = _lib.load()
    z, mu_all, logvar = _rows(z), _rows(mu_all), _rows(logvar)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    nbytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, flags)
    if nbytes == 0:
        raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
    log_qz = torch.empty(b_loc, dtype=torch.float32, device=z.device)
    log_qz_prod = torch.empty(b_loc, dtype=torch.float32, device=z.device)
    with torch.cuda.device(z.device):
        st = lib.tcelbo_forward(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                logvar.data_ptr(), logvar.stride(0), b_loc, b_glob, row_offset, d, dataset_size, flags,
                                log_qz.data_ptr(), log_qz_prod.data_ptr(), ws.data_ptr(), nbytes, _stream(z))
    _lib.check(st, "tcelbo_forward")
    return log_qz, log_qz_prod, ws


@_tc_forward.register_fake
def _(z, mu_all, logvar, row_offset, dataset_size, flags):
    nbytes = _lib.load().tcelbo_workspace_bytes(z.shape[0], mu_all.shape[0], z.shape[1], flags)
    return (z.new_empty(z.shape[0]), z.new_empty(z.shape[0]), z.new_empty(nbytes, dtype=torch.uint8))


@torch.library.custom_op("tcelbo::tc_backward", mutates_args=(), device_types="cuda")
def _tc_backward(z: Tensor, mu_all: Tensor, logvar: Tensor, row_offset: int, dataset_size: int, flags: int,
                 g_log_qz: Tensor, g_log_qz_prod: Tensor, workspace: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    _alert_not_deterministic("tcelbo::tc_backward")
    lib = _lib.load()
    z, mu_all, logvar = _rows(z), _rows(mu_all), _rows(logvar)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    g_log_qz = g_log_qz.contiguous()
    g_log_qz_prod = g_log_qz_prod.contiguous()
    grad_z = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
    grad_mu = torch.empty(b_glob, d, dtype=torch.float32, device=z.device)
    grad_lv = torch.empty(logvar.shape[0], d, dtype=torch.float32, device=z.device)
    nscratch = lib.tcelbo_backward_scratch_bytes(b_loc, b_glob, d, flags)
    scratch = torch.empty(nscratch, dtype=torch.uint8, device=z.device)
    with torch.cuda.device(z.device):
        st = lib.tcelbo_backward(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                 logvar.data_ptr(), logvar.stride(0), b_loc, b_glob, row_offset, d, dataset_size, flags,
                                 g_log_qz.data_ptr(), g_log_qz_prod.data_ptr(),
                                 grad_z.data_ptr(), d, grad_mu.data_ptr(), d, grad_lv.data_ptr(), d,
                                 workspace.data_ptr(), workspace.numel(), scratch.data_ptr(), nscratch, _stream(z))
    _lib.check(st, "tcelbo_backward")
    return grad_z, grad_mu, grad_lv


@_tc_backward.register_fake
def _(z, mu_all, logvar, row_offset, dataset_size, flags, g_log_qz, g_log_qz_prod, workspace):
    return (z.new_empty(z.shape), mu_all.new_empty(mu_all.shape), logvar.new_empty(logvar.shape))


def _tc_setup_context(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    z, mu_all, logvar, row_offset, dataset_size, flags = inputs
    _, _, ws = output
    ctx.save_for_backward(z, mu_all, logvar, ws)
    ctx.meta = (row_offset, dataset_size, flags)


def _tc_autograd_backward(ctx, g_log_qz, g_log_qz_prod, _g_ws):
    z, mu_all, logvar, ws = ctx.saved_tensors
    row_offset, dataset_size, flags = ctx.meta
    if not flags & _lib.SAVE_FOR_BACKWARD:
        raise RuntimeError("tcelbo: forward ran without TCELBO_SAVE_FOR_BACKWARD but a gradient was requested")
    if g_log_qz is None and g_log_qz_prod is None:
        return None, None, None, None, None, None
    if g_log_qz is None:
        g_log_qz = torch.zeros(z.shape[0], dtype=torch.float32, device=z.device)
    if g_log_qz_prod is None:
        g_log_qz_prod = torch.zeros(z.shape[0], dtype=torch.float32, device=z.device)
    gz, gmu, glv = _tc_backward(z, mu_all, logvar, row_offset, dataset_size, flags, g_log_qz, g_log_qz_prod, ws)
    return gz, gmu, glv, None, None, None


_tc_forward.register_autograd(_tc_autograd_backward, setup_context=_tc_setup_context)


# --------------------------------------------------------------------------------------------------
# fused compute_kl_loss:  torch.ops.tcelbo.klloss_forward / klloss_backward
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tcelbo::klloss_forward", mutates_args=(), device_types="cuda")
def _klloss_forward(z: Tensor, mu_all: Tensor, logvar: Tensor, row_offset: int, dataset_size: int, flags: int,
                    beta: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (loss [B], kl [B], log_qz [B], log_qz_prod [B], loss_mean [], kl_mean [], workspace): the per-sample loss of
    solvers/tc.py:83-89 and its batch means, the latter reduced inside the finalize kernel (fixed summation order)."""
    lib = _lib.load()
    z, mu_all, logvar = _rows(z), _rows(mu_all), _rows(logvar)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    nbytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, flags)
    if nbytes == 0:
        raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
    out = [torch.empty(b_loc, dtype=torch.float32, device=z.device) for _ in range(4)]   # loss, kl, log_qz, log_qz_prod
    means = [torch.empty((), dtype=torch.float32, device=z.device) for _ in range(2)]
    fz = _lib.Fusion(loss_mean=means[0].data_ptr(), kl_mean=means[1].data_ptr())
    with torch.cuda.device(z.device):
        st = lib.tcelbo_klloss_forward_ex(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                          logvar.data_ptr(), logvar.stride(0), b_loc, b_glob, row_offset, d, dataset_size,
                                          flags, beta, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                          out[3].data_ptr(), ctypes.byref(fz), ws.data_ptr(), nbytes, _stream(z))
    _lib.check(st, "tcelbo_klloss_forward_ex")
    return out[0], out[1], out[2], out[3], means[0], means[1], ws


@_klloss_forward.register_fake
def _(z, mu_all, logvar, row_offset, dataset_size, flags, beta):
    nbytes = _lib.load().tcelbo_workspace_bytes(z.shape[0], mu_all.shape[0], z.shape[1], flags)
    b = z.shape[0]
    return (z.new_empty(b), z.new_empty(b), z.new_empty(b), z.new_empty(b), z.new_empty(()), z.new_empty(()),
            z.new_empty(nbytes, dtype=torch.uint8))


@torch.library.custom_op("tcelbo::klloss_backward", mutates_args=(), device_types="cuda")
def _klloss_backward(z: Tensor, mu_all: Tensor, logvar: Tensor, row_offset: int, dataset_size: int, flags: int, beta: float,
                     g_loss: Optional[Tensor], g_kl: Optional[Tensor], g_log_qz: Optional[Tensor], g_log_qz_prod: Optional[Tensor],
                     g_loss_mean: Optional[Tensor], g_kl_mean: Optional[Tensor],
                     workspace: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    _alert_not_deterministic("tcelbo::klloss_backward")
    lib = _lib.load()
    z, mu_all, logvar = _rows(z), _rows(mu_all), _rows(logvar)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    rows = [t.contiguous() if t is not None else None for t in (g_loss, g_kl, g_log_qz, g_log_qz_prod)]
    scal = [t.contiguous() if t is not None else None for t in (g_loss_mean, g_kl_mean)]
    grad_z = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
    grad_mu = torch.empty(b_glob, d, dtype=torch.float32, device=z.device)
    grad_lv = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
    nscratch = lib.tcelbo_backward_scratch_bytes(b_loc, b_glob, d, flags)
    scratch = torch.empty(nscratch, dtype=torch.uint8, device=z.device)
    ptr = lambda t: t.data_ptr() if t is not None else None                      # noqa: E731
    fz = _lib.Fusion(g_loss_mean=ptr(scal[0]), g_kl_mean=ptr(scal[1]))
    with torch.cuda.device(z.device):
        st = lib.tcelbo_klloss_backward_ex(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                           logvar.data_ptr(), logvar.stride(0), b_loc, b_glob, row_offset, d, dataset_size,
                                           flags, beta, *(ptr(t) for t in rows), ctypes.byref(fz),
                                           grad_z.data_ptr(), d, grad_mu.data_ptr(), d, grad_lv.data_ptr(), d,
                                           workspace.data_ptr(), workspace.numel(), scratch.data_ptr(), nscratch, _stream(z))
    _lib.check(st, "tcelbo_klloss_backward_ex")
    return grad_z, grad_mu, grad_lv


@_klloss_backward.register_fake
def _(z, mu_all, logvar, row_offset, dataset_size, flags, beta, g_loss, g_kl, g_log_qz, g_log_qz_prod, g_loss_mean, g_kl_mean,
      workspace):
    return (z.new_empty(z.shape), mu_all.new_empty(mu_all.shape), logvar.new_empty(logvar.shape))


def _klloss_setup_context(ctx, inputs, output):
    ctx.set_materialize_grads(False)          # unused outputs arrive as None instead of zero-filled tensors
    z, mu_all, logvar, row_offset, dataset_size, flags, beta = inputs
    ctx.save_for_backward(z, mu_all, logvar, output[6])
    ctx.meta = (row_offset, dataset_size, flags, beta)


def _klloss_autograd_backward(ctx, g_loss, g_kl, g_log_qz, g_log_qz_prod, g_loss_mean, g_kl_mean, _g_ws):
    z, mu_all, logvar, ws = ctx.saved_tensors
    row_offset, dataset_size, flags, beta = ctx.meta
    if not flags & _lib.SAVE_FOR_BACKWARD:
        raise RuntimeError("tcelbo: forward ran without TCELBO_SAVE_FOR_BACKWARD but a gradient was requested")
    if all(g is None for g in (g_loss, g_kl, g_log_qz, g_log_qz_prod, g_loss_mean, g_kl_mean)):
        return None, None, None, None, None, None, None
    gz, gmu, glv = _klloss_backward(z, mu_all, logvar, row_offset, dataset_size, flags, beta,
                                    g_loss, g_kl, g_log_qz, g_log_qz_prod, g_loss_mean, g_kl_mean, ws)
    return gz, gmu, glv, None, None, None, None


_klloss_forward.register_autograd(_klloss_autograd_backward, setup_context=_klloss_setup_context)


def _klloss(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str, group, exchange):
    """Shared front end of :func:`kl_tc_loss_terms` / :func:`kl_tc_loss_mean` -> the op's 6 tensor outputs."""
    for name, t in (("z", z), ("mu", mu), ("logvar", logvar)):
        _check(name, t)
    if not (z.shape == mu.shape == logvar.shape):
        raise ValueError(f"z, mu, logvar must have one shape, got {tuple(z.shape)}, {tuple(mu.shape)}, {tuple(logvar.shape)}")
    if estimator not in ("mss", "mws"):
        raise ValueError(f"estimator must be 'mss' or 'mws', got {estimator!r}")
    flags = (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | _lib.VAR_ROW
    if torch.is_grad_enabled() and (z.requires_grad or mu.requires_grad or logvar.requires_grad):
        flags |= _lib.SAVE_FOR_BACKWARD
    row_offset, mu_all = 0, mu
    if exchange is not None:
        from .peer import kl_tc_loss_terms_peer
        if estimator == "mss" and exchange.world * z.shape[0] == 1:
            raise ZeroDivisionError("float division by zero")
        loss, kl, log_qz, log_qz_prod = kl_tc_loss_terms_peer(z, mu, logvar, dataset_size, beta, flags, exchange)
        return loss, kl, log_qz, log_qz_prod, None, None
    if group is not None:
        import torch.distributed as dist
        if dist.get_world_size(group) > 1:
            row_offset, _ = shard_rows(group, z.shape[0], z.device)
            mu_all = gather_rows(mu, group)
    if estimator == "mss" and mu_all.shape[0] == 1:
        raise ZeroDivisionError("float division by zero")       # ops.py:44 with M = B-1 = 0
    return _klloss_forward(z, mu_all, logvar, row_offset, int(dataset_size), flags, float(beta))[:6]


def kl_tc_loss_terms(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str = "mss",
                     group=None, exchange=None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """One fused evaluation of ``TCSovler._compute_kl_loss_simple`` (solvers/tc.py:69-89) per sample:

        loss_i = (beta - 1) * (log_qz_i - log_qz_prod_i) + kl_i ,   kl_i = ops.py:161-163

    Returns ``(loss [B], kl [B], log_qz [B], log_qz_prod [B])``.  KL and the combine are folded into the TC
    kernels' finalize steps (forward and backward), so no separate KL or elementwise kernels are launched.
    ``group`` row-shards the batch exactly as in :func:`tc_terms` (NCCL all-gather / reduce-scatter around the kernels);
    ``exchange`` (a :class:`intro_tc_vae_b200.peer.PeerExchange`) row-shards it over the exchange's group with both
    exchange steps done by the library's kernels over NVLink peer memory instead.
    """
    return _klloss(z, mu, logvar, dataset_size, beta, estimator, group, exchange)[:4]


def kl_tc_loss_mean(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str = "mss",
                    group=None, exchange=None) -> Tuple[Tensor, Tensor]:
    """``reduce="mean"`` form of :func:`kl_tc_loss_terms`: 0-d ``(mean_i[(beta-1)*tc_i + kl_i], mean_i kl_i)``
    (solvers/tc.py:83-89 with the default reduce).  The means come out of the finalize kernel itself (deterministic
    last-CTA reduction) and their gradients enter the backward prologue as device scalars, so no reduction, expand or
    elementwise kernels surround the op.  Row-sharded calls return the mean over the local rows."""
    loss, kl, _, _, loss_mean, kl_mean = _klloss(z, mu, logvar, dataset_size, beta, estimator, group, exchange)
    if loss_mean is None:                                        # peer-memory path: per-row outputs only
        return loss.mean(), kl.mean()
    return loss_mean, kl_mean


# --------------------------------------------------------------------------------------------------
# fused MI / TC / dimension-wise KL decomposition:  torch.ops.tcelbo.decomp_forward / decomp_backward
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("tcelbo::decomp_forward", mutates_args=(), device_types="cuda")
def _decomp_forward(z: Tensor, mu_all: Tensor, logvar_all: Tensor, row_offset: int, dataset_size: int, flags: int,
                    beta: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (loss [B], mi [B], tc [B], dimkl [B], means [4], workspace): the per-sample terms of solvers/tc.py:91-144 on the
    column-variance density and their batch means (loss, mi, tc, dimkl), reduced inside the finalize kernel."""
    lib = _lib.load()
    z, mu_all, logvar_all = _rows(z), _rows(mu_all), _rows(logvar_all)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    nbytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, flags)
    if nbytes == 0:
        raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
    out = [torch.empty(b_loc, dtype=torch.float32, device=z.device) for _ in range(4)]   # loss, mi, tc, dimkl
    means = torch.empty(4, dtype=torch.float32, device=z.device)
    with torch.cuda.device(z.device):
        st = lib.tcelbo_decomp_forward(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                       logvar_all.data_ptr(), logvar_all.stride(0), b_loc, b_glob, row_offset, d, dataset_size,
                                       flags, beta, *(t.data_ptr() for t in out), means.data_ptr(), ws.data_ptr(), nbytes, _stream(z))
    _lib.check(st, "tcelbo_decomp_forward")
    return out[0], out[1], out[2], out[3], means, ws


@_decomp_forward.register_fake
def _(z, mu_all, logvar_all, row_offset, dataset_size, flags, beta):
    nbytes = _lib.load().tcelbo_workspace_bytes(z.shape[0], mu_all.shape[0], z.shape[1], flags)
    b = z.shape[0]
    return (z.new_empty(b), z.new_empty(b), z.new_empty(b), z.new_empty(b), z.new_empty(4), z.new_empty(nbytes, dtype=torch.uint8))


@torch.library.custom_op("tcelbo::decomp_backward", mutates_args=(), device_types="cuda")
def _decomp_backward(z: Tensor, mu_all: Tensor, logvar_all: Tensor, row_offset: int, dataset_size: int, flags: int, beta: float,
                     g_loss: Optional[Tensor], g_mi: Optional[Tensor], g_tc: Optional[Tensor], g_dimkl: Optional[Tensor],
                     g_means: Optional[Tensor], workspace: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    _alert_not_deterministic("tcelbo::decomp_backward")
    lib = _lib.load()
    z, mu_all, logvar_all = _rows(z), _rows(mu_all), _rows(logvar_all)
    b_loc, d = z.shape
    b_glob = mu_all.shape[0]
    ups = [t.contiguous() if t is not None else None for t in (g_loss, g_mi, g_tc, g_dimkl, g_means)]
    grad_z = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
    grad_mu = torch.empty(b_glob, d, dtype=torch.float32, device=z.device)
    grad_lv = torch.empty(b_glob, d, dtype=torch.float32, device=z.device)
    nscratch = lib.tcelbo_backward_scratch_bytes(b_loc, b_glob, d, flags)
    scratch = torch.empty(nscratch, dtype=torch.uint8, device=z.device)
    with torch.cuda.device(z.device):
        st = lib.tcelbo_decomp_backward(z.data_ptr(), z.stride(0), mu_all.data_ptr(), mu_all.stride(0),
                                        logvar_all.data_ptr(), logvar_all.stride(0), b_loc, b_glob, row_offset, d, dataset_size,
                                        flags, beta, *(t.data_ptr() if t is not None else None for t in ups),
                                        grad_z.data_ptr(), d, grad_mu.data_ptr(), d, grad_lv.data_ptr(), d,
                                        workspace.data_ptr(), workspace.numel(), scratch.data_ptr(), nscratch, _stream(z))
    _lib.check(st, "tcelbo_decomp_backward")
    return grad_z, grad_mu, grad_lv


@_decomp_backward.register_fake
def _(z, mu_all, logvar_all, row_offset, dataset_size, flags, beta, g_loss, g_mi, g_tc, g_dimkl, g_means, workspace):
    return (z.new_empty(z.shape), mu_all.new_empty(mu_all.shape), logvar_all.new_empty(logvar_all.shape))


def _decomp_setup_context(ctx, inputs, output):
    ctx.set_materialize_grads(False)          # unused outputs arrive as None instead of zero-filled tensors
    z, mu_all, logvar_all, row_offset, dataset_size, flags, beta = inputs
    ctx.save_for_backward(z, mu_all, logvar_all, output[5])
    ctx.meta = (row_offset, dataset_size, flags, beta)


def _decomp_autograd_backward(ctx, g_loss, g_mi, g_tc, g_dimkl, g_means, _g_ws):
    z, mu_all, logvar_all, ws = ctx.saved_tensors
    row_offset, dataset_size, flags, beta = ctx.meta
    if not flags & _lib.SAVE_FOR_BACKWARD:
        raise RuntimeError("tcelbo: forward ran without TCELBO_SAVE_FOR_BACKWARD but a gradient was requested")
    if all(g is None for g in (g_loss, g_mi, g_tc, g_dimkl, g_means)):
        return None, None, None, None, None, None, None
    gz, gmu, glv = _decomp_backward(z, mu_all, logvar_all, row_offset, dataset_size, flags, beta,
                                    g_loss, g_mi, g_tc, g_dimkl, g_means, ws)
    return gz, gmu, glv, None, None, None, None


_decomp_forward.register_autograd(_decomp_autograd_backward, setup_context=_decomp_setup_context)


def _decomp(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str, group, exchange):
    """Shared front end of :func:`tc_decomp_loss_terms` / :func:`tc_decomp_loss_mean` -> the op's 5 tensor outputs."""
    for name, t in (("z", z), ("mu", mu), ("logvar", logvar)):
        _check(name, t)
    if not (z.shape == mu.shape == logvar.shape):
        raise ValueError(f"z, mu, logvar must have one shape, got {tuple(z.shape)}, {tuple(mu.shape)}, {tuple(logvar.shape)}")
    if estimator not in ("mss", "mws"):
        raise ValueError(f"estimator must be 'mss' or 'mws', got {estimator!r}")
    flags = (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | _lib.VAR_COL
    if torch.is_grad_enabled() and (z.requires_grad or mu.requires_grad or logvar.requires_grad):
        flags |= _lib.SAVE_FOR_BACKWARD
    row_offset, mu_all, lv_all = 0, mu, logvar
    if exchange is not None:
        from .peer import tc_decomp_loss_terms_peer
        if estimator == "mss" and exchange.world * z.shape[0] == 1:
            raise ZeroDivisionError("float division by zero")
        return tc_decomp_loss_terms_peer(z, mu, logvar, dataset_size, beta, flags, exchange)
    if group is not None:
        import torch.distributed as dist
        if dist.get_world_size(group) > 1:
            row_offset, _ = shard_rows(group, z.shape[0], z.device)
            mu_all = gather_rows(mu, group)
            lv_all = gather_rows(logvar, group)
    if estimator == "mss" and mu_all.shape[0] == 1:
        raise ZeroDivisionError("float division by zero")       # ops.py:44 with M = B-1 = 0
    return _decomp_forward(z, mu_all, lv_all, row_offset, int(dataset_size), flags, float(beta))[:5]


def tc_decomp_loss_terms(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str = "mss",
                         group=None, exchange=None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """One fused evaluation of ``TCSovler._compute_kl_loss_full`` (solvers/tc.py:91-144), the beta-TCVAE loss, per sample:

        mi_i = log q(z_i|x_i) - log q(z_i),  tc_i = log q(z_i) - sum_d log q(z_id),  dimkl_i = sum_d log q(z_id) - log p(z_i)
        loss_i = mi_i + beta * tc_i + dimkl_i

    on the column-variance density (``tc_terms(..., var_of="col")``; ``log q(z_i|x_i)`` and ``log p(z_i)`` as in
    :func:`row_log_density`).  Returns ``(loss [B], mi [B], tc [B], dimkl [B])``.  The two row densities and the combine are
    folded into the TC kernels' finalize steps, forward and backward: three kernels each way.  ``group`` row-shards the batch
    exactly as :func:`tc_terms` with ``var_of="col"`` does (``mu`` and ``logvar`` all-gathered, column gradients
    reduce-scattered); outputs cover the local rows.  ``exchange`` (a :class:`intro_tc_vae_b200.peer.PeerExchange`) row-shards
    it over the exchange's group with both exchange steps, for ``mu`` and ``logvar``, done by the library's kernels over NVLink
    peer memory instead.
    """
    return _decomp(z, mu, logvar, dataset_size, beta, estimator, group, exchange)[:4]


def tc_decomp_loss_mean(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, estimator: str = "mss",
                        group=None, exchange=None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """``reduce="mean"`` form of :func:`tc_decomp_loss_terms`: 0-d ``(mean loss, mean mi, mean tc, mean dimkl)``.  The means
    come out of the finalize kernel (deterministic last-CTA reduction) and their gradients enter the backward prologue as
    device scalars.  Row-sharded calls (``group`` or ``exchange``) return the means over the local rows."""
    return tuple(_decomp(z, mu, logvar, dataset_size, beta, estimator, group, exchange)[4].unbind(0))


def tc_terms(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, estimator: str = "mss",
             var_of: str = "row", group=None) -> Tuple[Tensor, Tensor]:
    """Fused ``gaussian_log_density* -> minibatch_{stratified,weighted}_sampling``.

    Returns ``(log_qz_prod [B], log_qz [B])`` exactly like ops.py:104-115 / 92-101 applied to the
    [B,B,D] tensor of ops.py:80-82 (``var_of="row"``) or solvers/tc.py:114-116 (``var_of="col"``).

    ``group``: a torch.distributed process group whose ranks each hold ``B_loc`` consecutive rows of
    one global batch (rank r owns rows [r*B_loc, (r+1)*B_loc)); ``mu`` (and ``logvar`` for
    ``var_of="col"``) are all-gathered over NCCL, the weights use global indices, and the backward
    reduce-scatters the column gradients.  Outputs cover the local rows.
    """
    for name, t in (("z", z), ("mu", mu), ("logvar", logvar)):
        _check(name, t)
    if not (z.shape == mu.shape == logvar.shape):
        raise ValueError(f"z, mu, logvar must have one shape, got {tuple(z.shape)}, {tuple(mu.shape)}, {tuple(logvar.shape)}")
    if estimator not in ("mss", "mws"):
        raise ValueError(f"estimator must be 'mss' or 'mws', got {estimator!r}")
    if var_of not in ("row", "col"):
        raise ValueError(f"var_of must be 'row' or 'col', got {var_of!r}")
    flags = (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | (_lib.VAR_ROW if var_of == "row" else _lib.VAR_COL)
    if torch.is_grad_enabled() and (z.requires_grad or mu.requires_grad or logvar.requires_grad):
        flags |= _lib.SAVE_FOR_BACKWARD

    row_offset = 0
    mu_all, lv_op = mu, logvar
    if group is not None:
        import torch.distributed as dist
        if dist.get_world_size(group) > 1:
            row_offset, _ = shard_rows(group, z.shape[0], z.device)
            mu_all = gather_rows(mu, group)
            if var_of == "col":
                lv_op = gather_rows(logvar, group)
    b_glob = mu_all.shape[0]
    if estimator == "mss" and b_glob == 1:
        raise ZeroDivisionError("float division by zero")       # ops.py:44 with M = B-1 = 0
    log_qz, log_qz_prod, _ = _tc_forward(z, mu_all, lv_op, row_offset, int(dataset_size), flags)
    return log_qz_prod, log_qz


def total_correlation(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, reduce: str = "mean",
                      group=None) -> Tensor:
    """ops.py:52-89: ``log q(z) - sum_d log q(z_d)`` with minibatch stratified sampling; ``reduce="mean"``
    returns the batch mean, anything else the per-sample vector."""
    log_qz_prod, log_qz = tc_terms(z, mu, logvar, dataset_size, "mss", "row", group)
    tc = log_qz - log_qz_prod
    return tc.mean() if reduce == "mean" else tc


# --------------------------------------------------------------------------------------------------
# row-wise companions
# --------------------------------------------------------------------------------------------------
class _KLRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logvar: Tensor, mu: Tensor) -> Tensor:
        lib = _lib.load()
        logvar, mu = _rows(logvar), _rows(mu)
        b, d = logvar.shape
        out = torch.empty(b, dtype=torch.float32, device=logvar.device)
        with torch.cuda.device(logvar.device):
            st = lib.tcelbo_kl_forward(logvar.data_ptr(), logvar.stride(0), mu.data_ptr(), mu.stride(0), b, d,
                                       out.data_ptr(), _stream(logvar))
        _lib.check(st, "tcelbo_kl_forward")
        ctx.save_for_backward(logvar, mu)
        return out

    @staticmethod
    def backward(ctx, g: Tensor):
        lib = _lib.load()
        logvar, mu = ctx.saved_tensors
        b, d = logvar.shape
        g = g.contiguous()
        glv = torch.empty(b, d, dtype=torch.float32, device=logvar.device)
        gmu = torch.empty(b, d, dtype=torch.float32, device=logvar.device)
        with torch.cuda.device(logvar.device):
            st = lib.tcelbo_kl_backward(logvar.data_ptr(), logvar.stride(0), mu.data_ptr(), mu.stride(0), g.data_ptr(),
                                        b, d, glv.data_ptr(), d, gmu.data_ptr(), d, _stream(logvar))
        _lib.check(st, "tcelbo_kl_backward")
        return glv, gmu


def kl_no_reduce(logvar: Tensor, mu: Tensor) -> Tensor:
    """ops.py:161-163: per-sample KL(q(z|x) || N(0, I)) -> [B]."""
    _check("logvar", logvar)
    _check("mu", mu)
    if logvar.shape != mu.shape:
        raise ValueError("logvar and mu must have one shape")
    return _KLRows.apply(logvar, mu)


def kl_divergence(logvar: Tensor, mu: Tensor, reduce: str = "sum") -> Tensor:
    """ops.py:136-158.  Argument order is (logvar, mu); ``reduce`` in {"sum", "mean", anything else = none}."""
    kl = kl_no_reduce(logvar, mu)
    if reduce == "sum":
        return kl.sum()
    if reduce == "mean":
        return kl.mean()
    return kl


class _Reparam(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mu: Tensor, logvar: Tensor, eps: Tensor) -> Tensor:
        lib = _lib.load()
        mu, logvar, eps = _rows(mu), _rows(logvar), _rows(eps)
        b, d = mu.shape
        z = torch.empty(b, d, dtype=torch.float32, device=mu.device)
        with torch.cuda.device(mu.device):
            st = lib.tcelbo_reparam_forward(mu.data_ptr(), mu.stride(0), logvar.data_ptr(), logvar.stride(0),
                                            eps.data_ptr(), eps.stride(0), b, d, z.data_ptr(), d, _stream(mu))
        _lib.check(st, "tcelbo_reparam_forward")
        ctx.save_for_backward(logvar, eps)
        return z

    @staticmethod
    def backward(ctx, gz: Tensor):
        lib = _lib.load()
        logvar, eps = ctx.saved_tensors
        b, d = logvar.shape
        gz = _rows(gz)
        gmu = torch.empty(b, d, dtype=torch.float32, device=logvar.device)
        glv = torch.empty(b, d, dtype=torch.float32, device=logvar.device)
        with torch.cuda.device(logvar.device):
            st = lib.tcelbo_reparam_backward(logvar.data_ptr(), logvar.stride(0), eps.data_ptr(), eps.stride(0),
                                             gz.data_ptr(), gz.stride(0), b, d, gmu.data_ptr(), d, glv.data_ptr(), d,
                                             _stream(logvar))
        _lib.check(st, "tcelbo_reparam_backward")
        return gmu, glv, None


def reparameterize(mu: Tensor, logvar: Tensor, eps: Optional[Tensor] = None) -> Tensor:
    """ops.py:166-185: ``mu + eps * exp(0.5*logvar)``.  ``eps`` defaults to ``torch.randn`` drawn from the
    device generator exactly as the reference's ``torch.randn_like(std)`` does (same Philox offsets), so
    seeded runs produce the same samples; pass ``eps`` explicitly for RNG-free use."""
    _check("mu", mu)
    _check("logvar", logvar)
    if eps is None:
        eps = torch.randn(mu.shape, dtype=torch.float32, device=mu.device)
    else:
        _check("eps", eps)
    return _Reparam.apply(mu, logvar, eps)


class _RowDensity(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, mu: Optional[Tensor], logvar: Optional[Tensor]) -> Tensor:
        lib = _lib.load()
        x = _rows(x)
        mu = _rows(mu) if mu is not None else None
        logvar = _rows(logvar) if logvar is not None else None
        b, d = x.shape
        out = torch.empty(b, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            st = lib.tcelbo_rowdensity_forward(x.data_ptr(), x.stride(0),
                                               mu.data_ptr() if mu is not None else None, mu.stride(0) if mu is not None else 0,
                                               logvar.data_ptr() if logvar is not None else None,
                                               logvar.stride(0) if logvar is not None else 0, b, d, out.data_ptr(), _stream(x))
        _lib.check(st, "tcelbo_rowdensity_forward")
        ctx.has = (mu is not None, logvar is not None)
        ctx.save_for_backward(x, *(t for t in (mu, logvar) if t is not None))
        return out

    @staticmethod
    def backward(ctx, g: Tensor):
        lib = _lib.load()
        saved = list(ctx.saved_tensors)
        x = saved.pop(0)
        mu = saved.pop(0) if ctx.has[0] else None
        logvar = saved.pop(0) if ctx.has[1] else None
        b, d = x.shape
        g = g.contiguous()
        gx = torch.empty(b, d, dtype=torch.float32, device=x.device)
        gmu = torch.empty(b, d, dtype=torch.float32, device=x.device) if mu is not None else None
        glv = torch.empty(b, d, dtype=torch.float32, device=x.device) if logvar is not None else None
        with torch.cuda.device(x.device):
            st = lib.tcelbo_rowdensity_backward(
                x.data_ptr(), x.stride(0), mu.data_ptr() if mu is not None else None, mu.stride(0) if mu is not None else 0,
                logvar.data_ptr() if logvar is not None else None, logvar.stride(0) if logvar is not None else 0,
                g.data_ptr(), b, d, gx.data_ptr(), d, gmu.data_ptr() if gmu is not None else None, d,
                glv.data_ptr() if glv is not None else None, d, _stream(x))
        _lib.check(st, "tcelbo_rowdensity_backward")
        return gx, gmu, glv


def row_log_density(x: Tensor, mu: Optional[Tensor] = None, logvar: Optional[Tensor] = None) -> Tensor:
    """``gaussian_log_density(x, mu, logvar).sum(dim=1)`` (ops.py:24-29, solvers/tc.py:107,112) -> [B].
    ``mu=None, logvar=None`` is the standard-normal prior log p(z)."""
    _check("x", x)
    if mu is not None:
        _check("mu", mu)
    if logvar is not None:
        _check("logvar", logvar)
    return _RowDensity.apply(x, mu, logvar)


# --------------------------------------------------------------------------------------------------
# materialised-tensor helpers of the reference's ops.py (API parity; HBM-bound, off the fused path)
# --------------------------------------------------------------------------------------------------
def _bcast3(*ts: Tensor):
    """Broadcast to one shape of at most 3 dims; returns (views, shape3, element strides per operand)."""
    for i, t in enumerate(ts):
        if not isinstance(t, Tensor) or not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"operand {i} must be an fp32 CUDA tensor: the B200 path has no CPU fallback")
    views = torch.broadcast_tensors(*ts)
    shape = tuple(views[0].shape)
    if len(shape) > 3:
        raise NotImplementedError(f"at most 3 broadcast dims are supported, got shape {shape}")
    pad = 3 - len(shape)
    shape3 = (1,) * pad + shape
    strides = [(0,) * pad + tuple(v.stride()) for v in views]
    return views, shape, shape3, strides


class _Density(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, mu: Tensor, logvar: Tensor, floored: bool) -> Tensor:
        import ctypes
        lib = _lib.load()
        views, shape, shape3, strides = _bcast3(x, mu, logvar)
        out = torch.empty(shape, dtype=torch.float32, device=x.device)
        arr = lambda v: (ctypes.c_int64 * 3)(*v)
        with torch.cuda.device(x.device):
            st = lib.tcelbo_density_forward(int(floored), views[0].data_ptr(), views[1].data_ptr(), views[2].data_ptr(),
                                            arr(shape3), arr(strides[0]), arr(strides[1]), arr(strides[2]), out.data_ptr(), _stream(x))
        _lib.check(st, "tcelbo_density_forward")
        ctx.save_for_backward(x, mu, logvar)
        ctx.floored = floored
        return out

    @staticmethod
    def backward(ctx, g: Tensor):
        import ctypes
        lib = _lib.load()
        x, mu, logvar = ctx.saved_tensors
        views, shape, shape3, strides = _bcast3(x, mu, logvar)
        g = g.contiguous()
        gx, gmu, glv = (torch.empty(shape, dtype=torch.float32, device=x.device) for _ in range(3))
        arr = lambda v: (ctypes.c_int64 * 3)(*v)
        with torch.cuda.device(x.device):
            st = lib.tcelbo_density_backward(int(ctx.floored), views[0].data_ptr(), views[1].data_ptr(), views[2].data_ptr(),
                                             g.data_ptr(), arr(shape3), arr(strides[0]), arr(strides[1]), arr(strides[2]),
                                             gx.data_ptr(), gmu.data_ptr(), glv.data_ptr(), _stream(x))
        _lib.check(st, "tcelbo_density_backward")
        return gx.sum_to_size(x.shape), gmu.sum_to_size(mu.shape), glv.sum_to_size(logvar.shape), None


def gaussian_log_density_torch(x: Tensor, mu: Tensor, logvar: Tensor) -> Tensor:
    """ops.py:15-21: elementwise (broadcasting) Gaussian log-density with the 1e-4 variance floor
    (straight-through gradient) and the -50 clamp.  Materialises the broadcast shape -- use :func:`tc_terms`
    for the fused estimator."""
    return _Density.apply(x, mu, logvar, True)


def gaussian_log_density(x: Tensor, mu: Tensor, logvar: Tensor) -> Tensor:
    """ops.py:24-29: un-floored variant, clamped at -50."""
    return _Density.apply(x, mu, logvar, False)


class _Sampling(torch.autograd.Function):
    @staticmethod
    def forward(ctx, log_qz_prob: Tensor, dataset_size: int, flags: int):
        lib = _lib.load()
        lp = log_qz_prob.contiguous()
        b, d = lp.shape[0], lp.shape[2]
        dev = lp.device
        prod = torch.empty(b, dtype=torch.float32, device=dev)
        joint = torch.empty(b, dtype=torch.float32, device=dev)
        lse_d = torch.empty(b, d, dtype=torch.float32, device=dev)
        srow = torch.empty(b, b, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = lib.tcelbo_sampling_forward(lp.data_ptr(), b, d, dataset_size, flags, prod.data_ptr(), joint.data_ptr(),
                                             lse_d.data_ptr(), srow.data_ptr(), _stream(lp))
        _lib.check(st, "tcelbo_sampling_forward")
        ctx.save_for_backward(lp, lse_d, srow, joint)
        ctx.meta = (dataset_size, flags)
        return prod, joint

    @staticmethod
    def backward(ctx, g_prod, g_joint):
        lib = _lib.load()
        lp, lse_d, srow, joint = ctx.saved_tensors
        dataset_size, flags = ctx.meta
        b, d = lp.shape[0], lp.shape[2]
        g_prod = torch.zeros_like(joint) if g_prod is None else g_prod.contiguous()
        g_joint = torch.zeros_like(joint) if g_joint is None else g_joint.contiguous()
        glp = torch.empty_like(lp)
        with torch.cuda.device(lp.device):
            st = lib.tcelbo_sampling_backward(lp.data_ptr(), b, d, dataset_size, flags, g_prod.data_ptr(), g_joint.data_ptr(),
                                              lse_d.data_ptr(), srow.data_ptr(), joint.data_ptr(), glp.data_ptr(), _stream(lp))
        _lib.check(st, "tcelbo_sampling_backward")
        return glp, None, None


def _sampling(log_qz_prob: Tensor, batch_size: int, dataset_size: int, flags: int):
    if not isinstance(log_qz_prob, Tensor) or not log_qz_prob.is_cuda or log_qz_prob.dtype != torch.float32:
        raise RuntimeError("log_qz_prob must be an fp32 CUDA tensor: the B200 path has no CPU fallback")
    if log_qz_prob.dim() != 3 or log_qz_prob.shape[0] != batch_size or log_qz_prob.shape[1] != batch_size:
        raise ValueError(f"log_qz_prob must be [batch, batch, latent] with batch={batch_size}, got {tuple(log_qz_prob.shape)}")
    if batch_size == 1 and flags == _lib.EST_MSS:
        raise ZeroDivisionError("float division by zero")
    return _Sampling.apply(log_qz_prob, int(dataset_size), flags)


def minibatch_stratified_sampling(log_qz_prob: Tensor, batch_size: int, dataset_size: int):
    """ops.py:104-115 on a materialised [B,B,D] tensor: (sum_d LSE_j(logW + lp), LSE_j(logW + sum_d lp))."""
    return _sampling(log_qz_prob, batch_size, dataset_size, _lib.EST_MSS)


def minibatch_weighted_sampling(log_qz_prob: Tensor, batch_size: int, dataset_size: int):
    """ops.py:92-101 on a materialised [B,B,D] tensor."""
    return _sampling(log_qz_prob, batch_size, dataset_size, _lib.EST_MWS)


# --------------------------------------------------------------------------------------------------
# host-side helper kept for API parity (the kernels fold the matrix into three scalars)
# --------------------------------------------------------------------------------------------------
def log_importance_weight_matrix(batch_size: int, dataset_size: int) -> Tensor:
    """ops.py:32-49: fp32 [B,B] host tensor; flat stride-B writes hit columns 0 and 1, then W[B-2, 0]."""
    n = dataset_size
    m = batch_size - 1
    strat = (n - m) / (n * m)
    w = torch.full((batch_size, batch_size), 1.0 / m, dtype=torch.float32)
    w[:, 0] = 1.0 / n
    if batch_size > 1:
        w[:, 1] = strat
    w[m - 1, 0] = strat
    return w.log()
