"""CUDA-graph capture of one TC-ELBO loss evaluation (forward + backward) for fixed shapes.

A row-sharded step at 8 GPUs is ~1 ms of kernels behind ~10 launches and two exchange steps, which eager
PyTorch cannot issue fast enough from one Python thread; replaying a captured graph removes the launch gaps.
Everything the library launches is capturable by construction (no host synchronisation, no allocation inside
the C ABI, explicit stream argument)."""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib, ops


class GraphedKLLoss:
    """``loss, dmu, dlogvar = graphed(mu, logvar, eps)`` with

        z    = mu + eps * exp(0.5 * logvar)                       (ops.py:183-185)
        loss = mean_i[(beta - 1) * tc_i + kl_i]                   (loss="simple": solvers/tc.py:69-89, reduce="mean")
        loss = mean_i[mi_i + beta * tc_i + dimkl_i]               (loss="decomp": solvers/tc.py:91-144, reduce="mean")

    evaluated and differentiated inside one CUDA graph.  ``mu``/``logvar``/``eps`` are ``[b_loc, d]`` fp32 CUDA
    tensors (or pinned host tensors: they are copied into the graph's static inputs on the current stream);
    the returned tensors are the graph's static outputs and are overwritten by the next call.

    ``group``: row-shard over the ranks of a process group; ``loss`` is then the mean over this rank's rows.
    ``exchange``: how the column operand and its gradient cross ranks -- ``"nccl"`` (all-gather / reduce-scatter,
    captured in the graph), ``"peer"`` (the library's own kernels over NVLink peer memory,
    :mod:`intro_tc_vae_b200.peer`), or ``"auto"`` (peer memory when it can be set up, NCCL otherwise).
    ``mode``: ``"direct"`` drives the C ABI itself (tcelbo_klloss_forward_ex / _backward_ex, or for loss="decomp"
    tcelbo_decomp_forward_ex / _backward_ex, with the reparameterize and batch-mean fusions: 6 launches for the whole step on one
    GPU, 7 with the peer exchange); ``"autograd"`` records the same step through ``torch.autograd`` (the public ops plus autograd's
    fill / accumulate kernels) and exists to cross-check the direct path.  ``loss="decomp"`` exchanges ``logvar`` (and its
    gradient) as well as ``mu``, since the column-variance density of the decomposition reads every row's variance.
    ``capture=False`` issues the same launches eagerly on every call instead of replaying a graph (for profilers that
    want to see individual launches).
    """

    def __init__(self, b_loc: int, d: int, dataset_size: int, beta: float, device, group=None,
                 estimator: str = "mss", warmup: int = 3, exchange: str = "nccl", mode: str = "direct", capture: bool = True,
                 loss: str = "simple"):
        if mode not in ("direct", "autograd"):
            raise ValueError(f"mode must be 'direct' or 'autograd', got {mode!r}")
        if loss not in ("simple", "decomp"):
            raise ValueError(f"loss must be 'simple' or 'decomp', got {loss!r}")
        self.loss_form = loss
        if estimator not in ("mss", "mws"):
            raise ValueError(f"estimator must be 'mss' or 'mws', got {estimator!r}")
        self.device = torch.device(device)
        self.mode = mode
        self.group = group
        self.world, self.rank = 1, 0
        self.exchange = None
        self.exchange_kind = "none"
        if group is not None:
            import torch.distributed as dist
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
            if self.world > 1:
                self.exchange_kind = "nccl"
                if exchange not in ("nccl", "peer", "auto"):
                    raise ValueError(f"exchange must be 'nccl', 'peer' or 'auto', got {exchange!r}")
                if exchange in ("peer", "auto"):
                    from . import peer
                    try:
                        self.exchange = peer.PeerExchange(b_loc, d, group, self.device)
                    except Exception:
                        if exchange == "peer":
                            raise
                    # the choice is collective: one rank without symmetric memory puts every rank on NCCL
                    ok = torch.tensor([1 if self.exchange is not None else 0], device=self.device)
                    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
                    if int(ok.item()) == 0:
                        if exchange == "peer":
                            raise RuntimeError("tcelbo: the peer-memory exchange could not be set up on every rank of the group")
                        self.exchange = None
                    else:
                        self.exchange_kind = "peer"
        self.b_loc, self.d = int(b_loc), int(d)
        self.mu = torch.zeros(b_loc, d, device=self.device, requires_grad=(mode == "autograd"))
        self.logvar = torch.zeros(b_loc, d, device=self.device, requires_grad=(mode == "autograd"))
        self.eps = torch.zeros(b_loc, d, device=self.device)
        self._args = (int(dataset_size), float(beta), estimator, group)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.loss: Optional[Tensor] = None
        self.dmu: Optional[Tensor] = None
        self.dlogvar: Optional[Tensor] = None
        with torch.no_grad():                              # benign values for the warm-up / capture passes
            self.logvar.fill_(-2.0)
        if mode == "direct":
            self._alloc_direct()
            step = self._direct_step if loss == "simple" else self._direct_decomp_step
        else:
            step = self._autograd_step
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                step()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        if mode == "autograd":
            self.mu.grad = None
            self.logvar.grad = None
        self._step = step
        if capture:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self.loss = step()
            self.graph = graph
        else:
            self.loss = step()
        if mode == "autograd":
            self.dmu, self.dlogvar = self.mu.grad, self.logvar.grad

    # ---- the step through torch.autograd -------------------------------------------------------------
    def _autograd_step(self) -> Tensor:
        n, beta, estimator, group = self._args
        self.mu.grad = None
        self.logvar.grad = None
        z = ops.reparameterize(self.mu, self.logvar, self.eps)
        if self.loss_form == "decomp":
            loss = ops.tc_decomp_loss_mean(z, self.mu, self.logvar, n, beta, estimator, group, self.exchange)[0]
        else:
            loss = ops.kl_tc_loss_terms(z, self.mu, self.logvar, n, beta, estimator, group, self.exchange)[0].mean()
        loss.backward()
        return loss.detach()

    # ---- the same step driven through the C ABI ------------------------------------------------------
    def _alloc_direct(self) -> None:
        lib = _lib.load()
        n, beta, estimator, _ = self._args
        dev, b_loc, d = self.device, self.b_loc, self.d
        decomp = self.loss_form == "decomp"
        self._flags = (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | (_lib.VAR_COL if decomp else _lib.VAR_ROW) | _lib.SAVE_FOR_BACKWARD
        b_glob = b_loc * self.world
        if estimator == "mss" and b_glob == 1:
            raise ZeroDivisionError("float division by zero")       # ops.py:44 with M = B-1 = 0
        ws_bytes = lib.tcelbo_workspace_bytes(b_loc, b_glob, d, self._flags)
        sc_bytes = lib.tcelbo_backward_scratch_bytes(b_loc, b_glob, d, self._flags)
        if ws_bytes == 0 or sc_bytes == 0:
            raise NotImplementedError(f"tcelbo: unsupported shape b_loc={b_loc} b_glob={b_glob} d={d} (d must be <= 512)")
        f32 = dict(dtype=torch.float32, device=dev)
        self._z = torch.empty(b_loc, d, **f32)
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        self._scratch = None if self.exchange is not None else torch.empty(sc_bytes, dtype=torch.uint8, device=dev)
        self._sc_bytes = sc_bytes
        self._rows = [torch.empty(b_loc, **f32) for _ in range(4)]        # loss, kl, log_qz, log_qz_prod
        self._g_loss = torch.full((b_loc,), 1.0 / b_loc, **f32)           # d mean / d loss_i (peer path: per-row upstream gradient)
        self._loss = torch.zeros((), **f32)                               # batch mean, written by the forward finalize kernel
        self._one = torch.ones((), **f32)                                 # dLoss / dloss_mean
        self._gz = torch.empty(b_loc, d, **f32)
        self.dmu = torch.empty(b_loc, d, **f32)
        self.dlogvar = torch.empty(b_loc, d, **f32)
        nccl = self.world > 1 and self.exchange is None
        self._mu_all = torch.empty(b_glob, d, **f32) if nccl else None
        self._gmu_all = torch.empty(b_glob, d, **f32) if nccl else None
        if decomp:
            self._means = torch.zeros(4, **f32)                           # loss, mi, tc, dimkl means, written by the finalize kernel
            self._g_means = torch.tensor([1.0, 0.0, 0.0, 0.0], **f32)     # dLoss / d means
            self._lv_all = torch.empty(b_glob, d, **f32) if nccl else None
            self._glv_all = torch.empty(b_glob, d, **f32) if nccl else None

    def _direct_step(self) -> Tensor:
        import torch.distributed as dist
        lib = _lib.load()
        n, beta, _, group = self._args
        b_loc, d, flags = self.b_loc, self.d, self._flags
        mu, lv, eps, z = self.mu, self.logvar, self.eps, self._z
        P = lambda t: t.data_ptr()                                       # noqa: E731
        rows = [P(t) for t in self._rows]
        exch = self.exchange
        import ctypes
        with torch.cuda.device(self.device), torch.no_grad():
            st = torch.cuda.current_stream(self.device).cuda_stream
            if exch is None:
                # 6 launches: prologue (reparameterize + row constants + column padding), forward sweep, finalize (+ batch mean),
                # backward prologue, fused backward sweep, finalize (+ the chain rule through z = mu + eps * std)
                mu_all, row_offset = mu, 0
                if self._mu_all is not None:
                    dist.all_gather_into_tensor(self._mu_all, mu, group=group)
                    mu_all, row_offset = self._mu_all, self.rank * b_loc
                fz = _lib.Fusion(eps=P(eps), ldeps=d, z_out=P(z), ldz_out=d, loss_mean=P(self._loss))
                _lib.check(lib.tcelbo_klloss_forward_ex(None, 0, P(mu_all), d, P(lv), d, b_loc, mu_all.shape[0], row_offset, d, n, flags,
                                                        beta, *rows, ctypes.byref(fz), P(self._ws), self._ws.numel(), st),
                           "tcelbo_klloss_forward_ex")
                gmu = self._gmu_all if self._gmu_all is not None else self.dmu
                fb = _lib.Fusion(eps=P(eps), ldeps=d, g_loss_mean=P(self._one))
                _lib.check(lib.tcelbo_klloss_backward_ex(None, 0, P(mu_all), d, P(lv), d, b_loc, mu_all.shape[0], row_offset, d, n, flags,
                                                         beta, None, None, None, None, ctypes.byref(fb), P(self._gz), d, P(gmu), d,
                                                         P(self.dlogvar), d, P(self._ws), self._ws.numel(),
                                                         P(self._scratch), self._sc_bytes, st), "tcelbo_klloss_backward_ex")
                if self._gmu_all is not None:
                    dist.reduce_scatter_tensor(self.dmu, self._gmu_all, op=dist.ReduceOp.SUM, group=group)
                return self._loss
            # peer-memory exchange: the library's prologue / finalize kernels gather mu and reduce-scatter its gradient over NVLink;
            # reparameterize and the batch mean are fused here too (publish copy, barrier, 3 + barrier + 3 launches)
            k = exch.next_forward()
            exch.publish(mu, k)
            fz = _lib.Fusion(eps=P(eps), ldeps=d, z_out=P(z), ldz_out=d, loss_mean=P(self._loss))
            _lib.check(lib.tcelbo_klloss_forward_peer(None, 0, P(mu), d, P(exch.mu_tables[k]), d, P(lv), d, b_loc, self.world,
                                                      self.rank, d, n, flags, beta, *rows, ctypes.byref(fz), exch.sync_arg(), P(self._ws), self._ws.numel(), st),
                       "tcelbo_klloss_forward_peer")
            k = exch.next_backward()
            scratch = exch.scratch_sym[k]
            fb = _lib.Fusion(eps=P(eps), ldeps=d, g_loss_mean=P(self._one))
            for phase in (_lib.PEER_SWEEP, _lib.PEER_FINISH):
                _lib.check(lib.tcelbo_klloss_backward_peer(phase, None, 0, P(mu), d, P(lv), d, b_loc, self.world, self.rank, d, n,
                                                           flags, beta, None, None, None, None,
                                                           P(self._gz), d, P(self.dmu), d, P(self.dlogvar), d,
                                                           P(self._ws), self._ws.numel(), P(scratch), exch.scratch_bytes,
                                                           P(exch.scratch_tables[k]), ctypes.byref(fb), exch.sync_arg(), st),
                           "tcelbo_klloss_backward_peer")
                if phase == _lib.PEER_SWEEP:
                    exch.barrier_backward()
        return self._loss

    def _direct_decomp_step(self) -> Tensor:
        import ctypes
        import torch.distributed as dist
        lib = _lib.load()
        n, beta, _, group = self._args
        b_loc, d, flags = self.b_loc, self.d, self._flags
        mu, lv, eps, z = self.mu, self.logvar, self.eps, self._z
        P = lambda t: t.data_ptr()                                       # noqa: E731
        rows = [P(t) for t in self._rows]                                # loss, mi, tc, dimkl
        exch = self.exchange
        fz = _lib.Fusion(eps=P(eps), ldeps=d, z_out=P(z), ldz_out=d)
        fb = _lib.Fusion(eps=P(eps), ldeps=d)
        with torch.cuda.device(self.device), torch.no_grad():
            st = torch.cuda.current_stream(self.device).cuda_stream
            if exch is None:
                # 6 launches: prologue (reparameterize + column packing), forward sweep, finalize (+ the four means), backward
                # prologue, sweep, finalize (+ the chain rule through z = mu + eps * std); NCCL: mu and logvar gathered around them
                mu_all, lv_all, row_offset = mu, lv, 0
                if self._mu_all is not None:
                    dist.all_gather_into_tensor(self._mu_all, mu, group=group)
                    dist.all_gather_into_tensor(self._lv_all, lv, group=group)
                    mu_all, lv_all, row_offset = self._mu_all, self._lv_all, self.rank * b_loc
                b_glob = mu_all.shape[0]
                _lib.check(lib.tcelbo_decomp_forward_ex(None, 0, P(mu_all), d, P(lv_all), d, b_loc, b_glob, row_offset, d, n, flags, beta,
                                                        *rows, P(self._means), ctypes.byref(fz), P(self._ws), self._ws.numel(), st),
                           "tcelbo_decomp_forward_ex")
                gmu = self._gmu_all if self._gmu_all is not None else self.dmu
                glv = self._glv_all if self._glv_all is not None else self.dlogvar
                _lib.check(lib.tcelbo_decomp_backward_ex(None, 0, P(mu_all), d, P(lv_all), d, b_loc, b_glob, row_offset, d, n, flags, beta,
                                                         None, None, None, None, P(self._g_means), ctypes.byref(fb), P(self._gz), d,
                                                         P(gmu), d, P(glv), d, P(self._ws), self._ws.numel(), P(self._scratch),
                                                         self._sc_bytes, st), "tcelbo_decomp_backward_ex")
                if self._gmu_all is not None:
                    dist.reduce_scatter_tensor(self.dmu, self._gmu_all, op=dist.ReduceOp.SUM, group=group)
                    dist.reduce_scatter_tensor(self.dlogvar, self._glv_all, op=dist.ReduceOp.SUM, group=group)
                return self._means[0]
            # peer-memory exchange: 7 launches (publish of mu and logvar, 3 forward, 2 in the sweep phase, 1 in the finish)
            k = exch.next_forward()
            exch.publish(mu, k, lv)
            _lib.check(lib.tcelbo_decomp_forward_peer_ex(None, 0, P(mu), d, P(lv), d, P(exch.mu_tables[k]), P(exch.lv_tables[k]), d,
                                                         b_loc, self.world, self.rank, d, n, flags, beta, *rows, P(self._means),
                                                         ctypes.byref(fz), exch.sync_arg(), P(self._ws), self._ws.numel(), st),
                       "tcelbo_decomp_forward_peer_ex")
            k = exch.next_backward()
            scratch = exch.scratch_sym[k]
            for phase in (_lib.PEER_SWEEP, _lib.PEER_FINISH):
                _lib.check(lib.tcelbo_decomp_backward_peer_ex(phase, None, 0, P(mu), d, P(lv), d, b_loc, self.world, self.rank, d, n,
                                                              flags, beta, None, None, None, None, P(self._g_means),
                                                              P(self._gz), d, P(self.dmu), d, P(self.dlogvar), d,
                                                              P(self._ws), self._ws.numel(), P(scratch), exch.scratch_bytes,
                                                              P(exch.scratch_tables[k]), ctypes.byref(fb), exch.sync_arg(), st),
                           "tcelbo_decomp_backward_peer_ex")
                if phase == _lib.PEER_SWEEP:
                    exch.barrier_backward()
        return self._means[0]

    def __call__(self, mu: Tensor, logvar: Tensor, eps: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        with torch.no_grad():
            self.mu.copy_(mu, non_blocking=True)
            self.logvar.copy_(logvar, non_blocking=True)
            self.eps.copy_(eps, non_blocking=True)
        return self.replay()

    def replay(self) -> Tuple[Tensor, Tensor, Tensor]:
        """Re-run on the inputs already resident in the static buffers."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self.loss = self._step()
            if self.mode == "autograd":
                self.dmu, self.dlogvar = self.mu.grad, self.logvar.grad
        return self.loss, self.dmu, self.dlogvar


class HostPipeline:
    """Streams HOST-resident batches through a loss step: host -> device copy, step, device -> host copy on three streams,
    ``depth``-deep, so that the PCIe transfers of neighbouring batches hide behind the kernels of the current one.

    ``step_fn(mu, logvar, eps) -> (loss, dmu, dlogvar)`` runs on the current stream on ``[b_loc, d]`` device tensors that stay
    valid until it returns (a :class:`GraphedKLLoss` instance is such a callable; so is an eager function that builds leaves
    from its arguments, calls ``compute_kl_loss`` and ``backward()``).  ``submit`` only enqueues work and returns the batch's
    sequence number; the pinned host outputs handed to it are complete after ``wait(seq)`` (or ``drain()``), and the pinned
    host inputs may be reused once ``inputs_consumed(seq)`` is true (always the case after ``wait(seq)``).
    """

    def __init__(self, step_fn, b_loc: int, d: int, device, depth: int = 2):
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.step_fn = step_fn
        self.device = torch.device(device)
        self.depth = int(depth)
        f32 = dict(dtype=torch.float32, device=self.device)
        self._in = [[torch.empty(b_loc, d, **f32) for _ in range(3)] for _ in range(depth)]
        self._out = [[torch.empty((), **f32), torch.empty(b_loc, d, **f32), torch.empty(b_loc, d, **f32)] for _ in range(depth)]
        ev = lambda: [torch.cuda.Event() for _ in range(depth)]
        self._in_ready, self._in_free, self._out_ready, self._out_done = ev(), ev(), ev(), ev()
        self.s_in = torch.cuda.Stream(self.device)
        self.s_out = torch.cuda.Stream(self.device)
        self.seq = 0
        torch.cuda.synchronize(self.device)

    def begin(self) -> None:
        """Order the copy streams after what the current stream has been given so far (e.g. a timing event)."""
        cur = torch.cuda.current_stream(self.device)
        self.s_in.wait_stream(cur)
        self.s_out.wait_stream(cur)

    def submit(self, mu_h: Tensor, logvar_h: Tensor, eps_h: Tensor, loss_h: Tensor, dmu_h: Tensor, dlogvar_h: Tensor) -> int:
        k, slot = self.seq, self.seq % self.depth
        cur = torch.cuda.current_stream(self.device)
        with torch.no_grad():
            with torch.cuda.stream(self.s_in):
                if k >= self.depth:
                    self.s_in.wait_event(self._in_free[slot])          # the step that last read this slot has been issued its reads
                for dst, src in zip(self._in[slot], (mu_h, logvar_h, eps_h)):
                    dst.copy_(src, non_blocking=True)
                self._in_ready[slot].record(self.s_in)
            cur.wait_event(self._in_ready[slot])
            loss, dmu, dlogvar = self.step_fn(*self._in[slot])
            self._in_free[slot].record(cur)
            if k >= self.depth:
                cur.wait_event(self._out_done[slot])                    # the device -> host copy that last read this slot
            o = self._out[slot]
            o[0].copy_(loss.detach().reshape(()))
            o[1].copy_(dmu)
            o[2].copy_(dlogvar)
            self._out_ready[slot].record(cur)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self._out_ready[slot])
                loss_h.copy_(o[0].reshape(loss_h.shape), non_blocking=True)
                dmu_h.copy_(o[1], non_blocking=True)
                dlogvar_h.copy_(o[2], non_blocking=True)
                self._out_done[slot].record(self.s_out)
        self.seq += 1
        return k

    def inputs_consumed(self, seq: int) -> bool:
        if seq >= self.seq:
            raise ValueError(f"batch {seq} has not been submitted")
        return self._in_free[seq % self.depth].query()                  # a later batch in the same slot only makes this conservative

    def wait(self, seq: int) -> None:
        """Block the host until batch ``seq``'s outputs are in its host buffers."""
        if seq >= self.seq:
            raise ValueError(f"batch {seq} has not been submitted")
        self._out_done[seq % self.depth].synchronize()                  # stream order: a later batch's copy implies this one's

    def fence(self) -> None:
        """Make the current stream wait for every device -> host copy submitted so far."""
        torch.cuda.current_stream(self.device).wait_stream(self.s_out)

    def drain(self) -> None:
        self.s_out.synchronize()
