"""Callers either side of the TC path (SURVEY.md 8f): the per-sample reconstruction loss (reference
``ops.py:188-236``) and the soft-intro exp-ELBO term (``solvers/intro.py:102-103``), as CUDA kernels behind
the reference's signatures.  fp32 CUDA tensors only (no CPU fallback)."""
from __future__ import annotations

import torch
from torch import Tensor

from . import _lib

_KINDS = {"mse": 0, "l1": 1, "bce": 2}


def _stream(t: Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


class _RecRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, recon: Tensor, kind: int) -> Tensor:
        lib = _lib.load()
        b, n = recon.shape
        out = torch.empty(b, dtype=torch.float32, device=recon.device)
        partial = torch.empty(b * lib.tcelbo_recloss_chunks(b, n), dtype=torch.float32, device=recon.device)
        with torch.cuda.device(recon.device):
            st = lib.tcelbo_recloss_forward(x.data_ptr(), recon.data_ptr(), b, n, kind, partial.data_ptr(), out.data_ptr(), _stream(recon))
        _lib.check(st, "tcelbo_recloss_forward")
        ctx.save_for_backward(x, recon)
        ctx.kind = kind
        return out

    @staticmethod
    def backward(ctx, g: Tensor):
        lib = _lib.load()
        x, recon = ctx.saved_tensors
        b, n = recon.shape
        g = g.contiguous()
        gr = torch.empty_like(recon)
        with torch.cuda.device(recon.device):
            st = lib.tcelbo_recloss_backward(x.data_ptr(), recon.data_ptr(), g.data_ptr(), b, n, ctx.kind, gr.data_ptr(), _stream(recon))
        _lib.check(st, "tcelbo_recloss_backward")
        return None, gr, None


def reconstruction_loss(x: Tensor, recon_x: Tensor, loss_type: str = "mse", reduction: str = "sum") -> Tensor:
    """ops.py:188-236: per-sample sum over pixels of mse / l1 / bce, then ``reduction`` in {"sum", "mean", "none"}
    over the batch.  ``x`` is treated as a constant (the reference detaches it)."""
    if x.size(0) == 0:
        raise AssertionError("empty batch")
    if reduction not in ("sum", "mean", "none"):
        raise NotImplementedError(reduction)
    if loss_type not in _KINDS:
        raise NotImplementedError(loss_type)
    for name, t in (("x", x), ("recon_x", recon_x)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"{name} must be an fp32 CUDA tensor: the B200 path has no CPU fallback")
    recon = recon_x.reshape(recon_x.size(0), -1).contiguous()
    xf = x.reshape(x.size(0), -1).detach().contiguous()
    if xf.shape != recon.shape:
        raise ValueError(f"x and recon_x must have the same number of elements per sample, got {tuple(xf.shape)} and {tuple(recon.shape)}")
    rows = _RecRows.apply(xf, recon, _KINDS[loss_type])
    if reduction == "sum":
        return rows.sum()
    if reduction == "mean":
        return rows.mean()
    return rows


class _ExpElbo(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rec_rows: Tensor, kl_rows: Tensor, scale: float) -> Tensor:
        lib = _lib.load()
        rec_rows, kl_rows = rec_rows.contiguous(), kl_rows.contiguous()
        b = rec_rows.shape[0]
        out = torch.empty(1, dtype=torch.float32, device=rec_rows.device)
        e_rows = torch.empty(b, dtype=torch.float32, device=rec_rows.device)
        with torch.cuda.device(rec_rows.device):
            st = lib.tcelbo_expelbo_forward(rec_rows.data_ptr(), kl_rows.data_ptr(), b, scale, out.data_ptr(), e_rows.data_ptr(), _stream(rec_rows))
        _lib.check(st, "tcelbo_expelbo_forward")
        ctx.save_for_backward(e_rows)
        ctx.scale = scale
        return out.reshape(())

    @staticmethod
    def backward(ctx, g: Tensor):
        lib = _lib.load()
        (e_rows,) = ctx.saved_tensors
        b = e_rows.shape[0]
        g = g.reshape(1).contiguous()
        g_rows = torch.empty_like(e_rows)
        with torch.cuda.device(e_rows.device):
            st = lib.tcelbo_expelbo_backward(e_rows.data_ptr(), g.data_ptr(), b, ctx.scale, g_rows.data_ptr(), _stream(e_rows))
        _lib.check(st, "tcelbo_expelbo_backward")
        return g_rows, g_rows, None


def exp_elbo(rec_per_sample: Tensor, kl_per_sample: Tensor, scale: float) -> Tensor:
    """solvers/intro.py:102-103: ``(-2 * scale * (rec_i + kl_i)).exp().mean()`` as one kernel each way."""
    if rec_per_sample.shape != kl_per_sample.shape or rec_per_sample.dim() != 1:
        raise ValueError("rec_per_sample and kl_per_sample must be [B] vectors of one shape")
    for name, t in (("rec_per_sample", rec_per_sample), ("kl_per_sample", kl_per_sample)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"{name} must be an fp32 CUDA tensor: the B200 path has no CPU fallback")
    return _ExpElbo.apply(rec_per_sample, kl_per_sample, float(scale))


class _FusedExpElbo(torch.autograd.Function):
    """solvers/intro.py:84-89 + 102-103 in one forward / one backward evaluation of a fused loss: the per-sample ``kl_i`` of
    ``compute_kl_loss(reduce="none", beta=beta_neg)`` never leaves the kernels; the exp-ELBO mean comes out of the forward finalize
    kernel and its gradient enters the backward prologue as a scalar.  ``decomp`` selects the loss form: False is the simple
    ``(beta-1)*tc_i + KL_i`` (solvers/tc.py:69-89, tcelbo_klloss_*_ex), True the decomposition ``mi_i + beta*tc_i + dimkl_i``
    (solvers/tc.py:91-144, tcelbo_decomp_*_ex).  Either way the op returns 4 per-row outputs, the first of which is kl_i."""

    @staticmethod
    def forward(ctx, z: Tensor, mu: Tensor, logvar: Tensor, rec_rows: Tensor, dataset_size: int, beta: float, scale: float, flags: int,
                decomp: bool):
        import ctypes
        lib = _lib.load()
        z, mu, logvar, rec_rows = z.contiguous(), mu.contiguous(), logvar.contiguous(), rec_rows.contiguous()
        b, d = z.shape
        dev = z.device
        nbytes = lib.tcelbo_workspace_bytes(b, b, d, flags)
        if nbytes == 0:
            raise NotImplementedError(f"tcelbo: unsupported shape b={b} d={d} (d must be <= 512)")
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        rows = [torch.empty(b, dtype=torch.float32, device=dev) for _ in range(5)]        # loss, (kl, log_qz, log_qz_prod | mi, tc, dimkl), e
        out = torch.empty((), dtype=torch.float32, device=dev)
        fz = _lib.Fusion(rec_rows=rec_rows.data_ptr(), scale=scale, expelbo=out.data_ptr(), e_rows=rows[4].data_ptr())
        args = (z.data_ptr(), d, mu.data_ptr(), d, logvar.data_ptr(), d, b, b, 0, d, dataset_size, flags, beta, *(t.data_ptr() for t in rows[:4]))
        with torch.cuda.device(dev):
            if decomp:
                st = lib.tcelbo_decomp_forward_ex(*args, None, ctypes.byref(fz), ws.data_ptr(), nbytes, _stream(z))
            else:
                st = lib.tcelbo_klloss_forward_ex(*args, ctypes.byref(fz), ws.data_ptr(), nbytes, _stream(z))
        _lib.check(st, "tcelbo_decomp_forward_ex" if decomp else "tcelbo_klloss_forward_ex")
        ctx.save_for_backward(z, mu, logvar, rows[4], ws)
        ctx.meta = (dataset_size, beta, scale, flags, decomp)
        ctx.mark_non_differentiable(rows[0])
        return out, rows[0]

    @staticmethod
    def backward(ctx, g_out: Tensor, _g_rows):
        import ctypes
        lib = _lib.load()
        z, mu, logvar, e_rows, ws = ctx.saved_tensors
        dataset_size, beta, scale, flags, decomp = ctx.meta
        b, d = z.shape
        dev = z.device
        g_out = g_out.reshape(()).contiguous()
        gz, gmu, glv = (torch.empty(b, d, dtype=torch.float32, device=dev) for _ in range(3))
        g_rec = torch.empty(b, dtype=torch.float32, device=dev)
        nscratch = lib.tcelbo_backward_scratch_bytes(b, b, d, flags)
        scratch = torch.empty(nscratch, dtype=torch.uint8, device=dev)
        fz = _lib.Fusion(scale=scale, e_rows=e_rows.data_ptr(), g_expelbo=g_out.data_ptr(), g_rec_rows=g_rec.data_ptr())
        args = (z.data_ptr(), d, mu.data_ptr(), d, logvar.data_ptr(), d, b, b, 0, d, dataset_size, flags, beta)
        tail = (gz.data_ptr(), d, gmu.data_ptr(), d, glv.data_ptr(), d, ws.data_ptr(), ws.numel(), scratch.data_ptr(), nscratch, _stream(z))
        with torch.cuda.device(dev):
            if decomp:
                st = lib.tcelbo_decomp_backward_ex(*args, None, None, None, None, None, ctypes.byref(fz), *tail)
            else:
                st = lib.tcelbo_klloss_backward_ex(*args, None, None, None, None, ctypes.byref(fz), *tail)
        _lib.check(st, "tcelbo_decomp_backward_ex" if decomp else "tcelbo_klloss_backward_ex")
        return gz, gmu, glv, g_rec, None, None, None, None, None


def _check_exp_elbo_args(z: Tensor, mu: Tensor, logvar: Tensor, rec_per_sample: Tensor) -> None:
    for name, t in (("z", z), ("mu", mu), ("logvar", logvar), ("rec_per_sample", rec_per_sample)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"{name} must be an fp32 CUDA tensor: the B200 path has no CPU fallback")
    if not (z.shape == mu.shape == logvar.shape) or z.dim() != 2 or rec_per_sample.shape != (z.shape[0],):
        raise ValueError("z, mu, logvar must be [B, D] of one shape and rec_per_sample [B]")
    if z.shape[0] == 1:
        raise ZeroDivisionError("float division by zero")       # ops.py:44 with M = B-1 = 0


def kl_tc_exp_elbo(z: Tensor, mu: Tensor, logvar: Tensor, rec_per_sample: Tensor, dataset_size: int, beta: float, scale: float):
    """``exp(-2*scale*(rec_i + kl_i)).mean()`` with ``kl_i = compute_kl_loss(z, mu, logvar, reduce="none", beta=beta)``
    (solvers/intro.py:84-89, 102-103; TC solver: solvers/tc.py:69-89) as ONE fused evaluation.  Returns
    ``(expelbo [], kl_rows [B] (detached))``; gradients flow to z, mu, logvar and rec_per_sample.  Single GPU."""
    _check_exp_elbo_args(z, mu, logvar, rec_per_sample)
    flags = _lib.EST_MSS | _lib.VAR_ROW | _lib.SAVE_FOR_BACKWARD
    return _FusedExpElbo.apply(z, mu, logvar, rec_per_sample, int(dataset_size), float(beta), float(scale), flags, False)


def tc_decomp_exp_elbo(z: Tensor, mu: Tensor, logvar: Tensor, rec_per_sample: Tensor, dataset_size: int, beta: float, scale: float):
    """The decomposition counterpart of :func:`kl_tc_exp_elbo`: ``exp(-2*scale*(rec_i + loss_i)).mean()`` with
    ``loss_i = mi_i + beta*tc_i + dimkl_i``, the per-sample loss of ``TCSovler._compute_kl_loss_full`` (solvers/tc.py:91-144,
    column-variance density, MSS), as ONE forward and ONE backward evaluation.  Returns ``(expelbo [], loss_rows [B] (detached))``;
    gradients flow to z, mu, logvar and rec_per_sample.  Single GPU."""
    _check_exp_elbo_args(z, mu, logvar, rec_per_sample)
    flags = _lib.EST_MSS | _lib.VAR_COL | _lib.SAVE_FOR_BACKWARD
    return _FusedExpElbo.apply(z, mu, logvar, rec_per_sample, int(dataset_size), float(beta), float(scale), flags, True)
