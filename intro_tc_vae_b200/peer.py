"""Peer-memory exchange for the row-sharded fused losses (SURVEY.md 8e): the two exchange steps of
``kl_tc_loss_terms(..., group=...)`` -- all-gather of the column operand ``mu`` before the forward sweep and
reduce-scatter of its gradient after the backward sweep -- done by the library's own kernels over NVLink peer
memory instead of NCCL (include/tcelbo.h: ``tcelbo_klloss_forward_peer`` / ``tcelbo_klloss_backward_peer``).
The decomposition loss (``tc_decomp_loss_terms``, column-variance density) exchanges ``mu`` and ``logvar`` the same way
(``tcelbo_decomp_forward_peer`` / ``tcelbo_decomp_backward_peer``); one exchange object serves both losses.

Each rank publishes its rows in a buffer from ``torch.distributed._symmetric_memory`` (mapped into every process of
the group); a stream-ordered cross-rank barrier follows, then

* forward : the column-prep kernel reads every rank's rows through a device table of peer pointers,
* backward: the sweep leaves the column sums in this rank's (symmetric) scratch, barrier, and the finalize kernel
  sums this rank's rows over all ranks' scratch buffers.

Two barriers of a few microseconds each replace two NCCL collectives, and the gathered operand / the scattered
gradient never take an extra trip through HBM.  Buffers are double-buffered so that one barrier per exchange is
enough (a buffer is rewritten two exchanges after it was read).  Everything is CUDA-graph capturable.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib


def available() -> bool:
    """True when this torch build has symmetric memory and the process group backend can rendezvous on it."""
    try:
        import torch.distributed._symmetric_memory  # noqa: F401
    except Exception:
        return False
    return torch.cuda.is_available()


class PeerExchange:
    """Symmetric buffers, barrier handles and device pointer tables for shards of ``[b_loc, d]`` on ``group``.

    Collective: every rank of the group must construct it (same arguments) at the same point of the program.
    """

    def __init__(self, b_loc: int, d: int, group=None, device=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        lib = _lib.load()
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.b_loc, self.d = int(b_loc), int(d)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        # one scratch serves both losses: the larger of the row-variance (simple loss) and column-variance (decomposition) plans
        self.scratch_bytes = max(lib.tcelbo_backward_scratch_bytes(self.b_loc, self.b_loc * self.world, self.d, var | _lib.SAVE_FOR_BACKWARD)
                                 for var in (_lib.VAR_ROW, _lib.VAR_COL))
        if self.scratch_bytes == 0:
            raise NotImplementedError(f"tcelbo: unsupported shard shape b_loc={b_loc} world={self.world} d={d}")
        pitch = (self.scratch_bytes + 255) // 256 * 256
        with torch.cuda.device(self.device):
            self.mu_sym = symm.empty(2, self.b_loc, self.d, dtype=torch.float32, device=self.device)
            self.lv_sym = symm.empty(2, self.b_loc, self.d, dtype=torch.float32, device=self.device)   # decomposition only
            self.scratch_sym = symm.empty(2, pitch, dtype=torch.uint8, device=self.device)
            name = self.group.group_name
            self.mu_hdl = symm.rendezvous(self.mu_sym, name)
            self.lv_hdl = symm.rendezvous(self.lv_sym, name)
            self.scratch_hdl = symm.rendezvous(self.scratch_sym, name)
            mu_step = self.b_loc * self.d * 4
            self.mu_tables = [torch.tensor([int(p) + k * mu_step for p in self.mu_hdl.buffer_ptrs], dtype=torch.int64,
                                           device=self.device) for k in range(2)]
            self.lv_tables = [torch.tensor([int(p) + k * mu_step for p in self.lv_hdl.buffer_ptrs], dtype=torch.int64,
                                           device=self.device) for k in range(2)]
            self.scratch_tables = [torch.tensor([int(p) + k * pitch for p in self.scratch_hdl.buffer_ptrs], dtype=torch.int64,
                                                device=self.device) for k in range(2)]
            # in-kernel barriers (tcelbo_peer_sync): 2 channels x world flag words per rank in symmetric memory, 4 local state words
            self.flags_sym = symm.empty(2 * self.world, dtype=torch.int32, device=self.device)
            self.flags_sym.zero_()
            self.flags_hdl = symm.rendezvous(self.flags_sym, name)
            self.flag_table = torch.tensor([int(p) for p in self.flags_hdl.buffer_ptrs], dtype=torch.int64, device=self.device)
            self.sync_state = torch.zeros(4, dtype=torch.int32, device=self.device)
            torch.cuda.synchronize(self.device)
            self.flags_hdl.barrier(channel=0)                       # every rank's flags are zero before anyone signals
            torch.cuda.synchronize(self.device)
        import os
        self.inkernel_sync = os.environ.get("TCELBO_PEER_SYNC", "kernel") != "host"
        self._sync_args = _lib.PeerSyncArgs(flag_parts=self.flag_table.data_ptr(), state=self.sync_state.data_ptr())
        self._n_fwd = 0
        self._n_bwd = 0

    def sync_arg(self):
        """ctypes pointer to the tcelbo_peer_sync of this exchange, or None when the host-side barriers are used."""
        import ctypes
        return ctypes.byref(self._sync_args) if self.inkernel_sync else None

    def publish(self, mu: Tensor, k: int, logvar: Optional[Tensor] = None) -> None:
        """Make this rank's rows of ``mu`` (and of ``logvar``, which the column-variance decomposition gathers too) visible to the
        other ranks (buffer k) and order the gather after everybody's publish: with in-kernel barriers one library kernel copies
        the rows and opens the barrier the prologue kernel waits on; otherwise copies + a symmetric-memory barrier on the stream."""
        if self.inkernel_sync:
            lib = _lib.load()
            st = torch.cuda.current_stream(self.device).cuda_stream
            if logvar is None:
                _lib.check(lib.tcelbo_peer_publish(mu.data_ptr(), mu.stride(0), self.b_loc, self.d, self.mu_sym[k].data_ptr(),
                                                   self.sync_arg(), st), "tcelbo_peer_publish")
            else:
                _lib.check(lib.tcelbo_peer_publish_mu_logvar(mu.data_ptr(), mu.stride(0), logvar.data_ptr(), logvar.stride(0),
                                                             self.b_loc, self.d, self.mu_sym[k].data_ptr(), self.lv_sym[k].data_ptr(),
                                                             self.sync_arg(), st), "tcelbo_peer_publish_mu_logvar")
        else:
            self.mu_sym[k].copy_(mu)
            if logvar is not None:
                self.lv_sym[k].copy_(logvar)
            self.mu_hdl.barrier(channel=0)

    def barrier_backward(self) -> None:
        if not self.inkernel_sync:
            self.scratch_hdl.barrier(channel=0)

    # -- buffer rotation ---------------------------------------------------------------------------
    def next_forward(self) -> int:
        k = self._n_fwd & 1
        self._n_fwd += 1
        return k

    def next_backward(self) -> int:
        k = self._n_bwd & 1
        self._n_bwd += 1
        return k

    def check(self, z: Tensor) -> None:
        if tuple(z.shape) != (self.b_loc, self.d):
            raise ValueError(f"PeerExchange was built for shards of {(self.b_loc, self.d)}, got {tuple(z.shape)}")
        if z.device != self.device:
            raise ValueError(f"PeerExchange lives on {self.device}, got a tensor on {z.device}")


class _PeerKLLoss(torch.autograd.Function):
    """solvers/tc.py:69-89 per sample on a row shard; same outputs / gradients as ops._klloss_forward behind
    sharding.gather_rows, with the exchange steps inside the library's kernels."""

    @staticmethod
    def forward(ctx, z: Tensor, mu: Tensor, logvar: Tensor, exch: PeerExchange, dataset_size: int, flags: int, beta: float):
        from .ops import _rows, _stream
        lib = _lib.load()
        z, mu, logvar = _rows(z), _rows(mu), _rows(logvar)
        exch.check(z)
        b_loc, d = z.shape
        b_glob = b_loc * exch.world
        nbytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, flags)
        if nbytes == 0:
            raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
        ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
        out = [torch.empty(b_loc, dtype=torch.float32, device=z.device) for _ in range(4)]
        k = exch.next_forward()
        with torch.cuda.device(z.device):
            exch.publish(mu.detach(), k)                            # this rank's rows -> its mapped buffer (+ barrier)
            st = lib.tcelbo_klloss_forward_peer(z.data_ptr(), z.stride(0), mu.data_ptr(), mu.stride(0),
                                                exch.mu_tables[k].data_ptr(), d, logvar.data_ptr(), logvar.stride(0),
                                                b_loc, exch.world, exch.rank, d, dataset_size, flags, beta,
                                                out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(),
                                                None, exch.sync_arg(), ws.data_ptr(), nbytes, _stream(z))
        _lib.check(st, "tcelbo_klloss_forward_peer")
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(z, mu, logvar, ws)
        ctx.exch = exch
        ctx.meta = (dataset_size, flags, beta)
        return out[0], out[1], out[2], out[3]

    @staticmethod
    def backward(ctx, g_loss, g_kl, g_log_qz, g_log_qz_prod):
        from .ops import _stream
        z, mu, logvar, ws = ctx.saved_tensors
        exch: PeerExchange = ctx.exch
        dataset_size, flags, beta = ctx.meta
        if not flags & _lib.SAVE_FOR_BACKWARD:
            raise RuntimeError("tcelbo: forward ran without TCELBO_SAVE_FOR_BACKWARD but a gradient was requested")
        # the exchange is collective: every rank runs it even if its own upstream gradients are all absent
        if g_loss is None:
            g_loss = torch.zeros(z.shape[0], dtype=torch.float32, device=z.device)
        g_loss = g_loss.contiguous()
        opt = [t.contiguous() if t is not None else None for t in (g_kl, g_log_qz, g_log_qz_prod)]
        b_loc, d = z.shape
        grad_z = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        grad_mu = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        grad_lv = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        lib = _lib.load()
        k = exch.next_backward()
        scratch = exch.scratch_sym[k]

        def call(phase: int) -> int:
            return lib.tcelbo_klloss_backward_peer(
                phase, z.data_ptr(), z.stride(0), mu.data_ptr(), mu.stride(0), logvar.data_ptr(), logvar.stride(0),
                b_loc, exch.world, exch.rank, d, dataset_size, flags, beta,
                g_loss.data_ptr(), *(t.data_ptr() if t is not None else None for t in opt),
                grad_z.data_ptr(), d, grad_mu.data_ptr(), d, grad_lv.data_ptr(), d,
                ws.data_ptr(), ws.numel(), scratch.data_ptr(), exch.scratch_bytes,
                exch.scratch_tables[k].data_ptr(), None, exch.sync_arg(), _stream(z))

        with torch.cuda.device(z.device):
            _lib.check(call(_lib.PEER_SWEEP), "tcelbo_klloss_backward_peer(sweep)")
            exch.barrier_backward()                                 # host-side barrier mode only; else the finalize kernel waits itself
            _lib.check(call(_lib.PEER_FINISH), "tcelbo_klloss_backward_peer(finish)")
        return grad_z, grad_mu, grad_lv, None, None, None, None


class _PeerDecompLoss(torch.autograd.Function):
    """solvers/tc.py:91-144 per sample on a row shard; same outputs / gradients as ops._decomp_forward behind
    sharding.gather_rows of mu and logvar, with the exchange steps inside the library's kernels."""

    @staticmethod
    def forward(ctx, z: Tensor, mu: Tensor, logvar: Tensor, exch: PeerExchange, dataset_size: int, flags: int, beta: float):
        from .ops import _rows, _stream
        lib = _lib.load()
        z, mu, logvar = _rows(z), _rows(mu), _rows(logvar)
        exch.check(z)
        b_loc, d = z.shape
        b_glob = b_loc * exch.world
        nbytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, flags)
        if nbytes == 0:
            raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
        ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
        out = [torch.empty(b_loc, dtype=torch.float32, device=z.device) for _ in range(4)]   # loss, mi, tc, dimkl
        means = torch.empty(4, dtype=torch.float32, device=z.device)
        k = exch.next_forward()
        with torch.cuda.device(z.device):
            exch.publish(mu.detach(), k, logvar.detach())           # this rank's rows -> its mapped buffers (+ barrier)
            st = lib.tcelbo_decomp_forward_peer(z.data_ptr(), z.stride(0), mu.data_ptr(), mu.stride(0), logvar.data_ptr(),
                                                logvar.stride(0), exch.mu_tables[k].data_ptr(), exch.lv_tables[k].data_ptr(), d,
                                                b_loc, exch.world, exch.rank, d, dataset_size, flags, beta,
                                                *(t.data_ptr() for t in out), means.data_ptr(), exch.sync_arg(),
                                                ws.data_ptr(), nbytes, _stream(z))
        _lib.check(st, "tcelbo_decomp_forward_peer")
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(z, mu, logvar, ws)
        ctx.exch = exch
        ctx.meta = (dataset_size, flags, beta)
        return out[0], out[1], out[2], out[3], means

    @staticmethod
    def backward(ctx, g_loss, g_mi, g_tc, g_dimkl, g_means):
        from .ops import _alert_not_deterministic, _stream
        _alert_not_deterministic("tcelbo_decomp_backward_peer")
        z, mu, logvar, ws = ctx.saved_tensors
        exch: PeerExchange = ctx.exch
        dataset_size, flags, beta = ctx.meta
        if not flags & _lib.SAVE_FOR_BACKWARD:
            raise RuntimeError("tcelbo: forward ran without TCELBO_SAVE_FOR_BACKWARD but a gradient was requested")
        ups = [t.contiguous() if t is not None else None for t in (g_loss, g_mi, g_tc, g_dimkl, g_means)]
        # the exchange is collective: every rank runs it even if its own upstream gradients are all absent
        if all(t is None for t in ups):
            ups[0] = torch.zeros(z.shape[0], dtype=torch.float32, device=z.device)
        b_loc, d = z.shape
        grad_z = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        grad_mu = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        grad_lv = torch.empty(b_loc, d, dtype=torch.float32, device=z.device)
        lib = _lib.load()
        k = exch.next_backward()
        scratch = exch.scratch_sym[k]

        def call(phase: int) -> int:
            return lib.tcelbo_decomp_backward_peer(
                phase, z.data_ptr(), z.stride(0), mu.data_ptr(), mu.stride(0), logvar.data_ptr(), logvar.stride(0),
                b_loc, exch.world, exch.rank, d, dataset_size, flags, beta,
                *(t.data_ptr() if t is not None else None for t in ups),
                grad_z.data_ptr(), d, grad_mu.data_ptr(), d, grad_lv.data_ptr(), d,
                ws.data_ptr(), ws.numel(), scratch.data_ptr(), exch.scratch_bytes,
                exch.scratch_tables[k].data_ptr(), exch.sync_arg(), _stream(z))

        with torch.cuda.device(z.device):
            _lib.check(call(_lib.PEER_SWEEP), "tcelbo_decomp_backward_peer(sweep)")
            exch.barrier_backward()                                 # host-side barrier mode only; else the finalize kernel waits itself
            _lib.check(call(_lib.PEER_FINISH), "tcelbo_decomp_backward_peer(finish)")
        return grad_z, grad_mu, grad_lv, None, None, None, None


def tc_decomp_loss_terms_peer(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, flags: int,
                              exchange: PeerExchange) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (loss, mi, tc, dimkl [b_loc], means [4] over the local rows)."""
    return _PeerDecompLoss.apply(z, mu, logvar, exchange, int(dataset_size), int(flags), float(beta))


def kl_tc_loss_terms_peer(z: Tensor, mu: Tensor, logvar: Tensor, dataset_size: int, beta: float, flags: int,
                          exchange: PeerExchange) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    return _PeerKLLoss.apply(z, mu, logvar, exchange, int(dataset_size), int(flags), float(beta))
