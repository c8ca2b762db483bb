"""The peer-memory decomposition (tcelbo_decomp_forward_peer / _backward_peer) with P ranks played one after the other on one
GPU, and the two-GPU check of NCCL-sharded == peer-sharded == single GPU (tools/check_decomp_peer.py under torchrun).

The peer entry points take plain device pointer tables, so ordinary allocations stand in for the ranks' mapped buffers and
sync = NULL (the in-kernel barriers need the ranks to run concurrently): all forwards, then all sweeps, then all finishes."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _relerr(a, b):
    a = np.asarray(a.detach().cpu(), dtype=np.float64)
    b = np.asarray(b.detach().cpu(), dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _latents(B, D, family, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    if family == "base":
        mu = torch.randn(B, D, generator=g)
        lv = -2.0 + torch.randn(B, D, generator=g)
    else:                         # sharp posteriors: most log-densities clamped
        mu = 2.0 * torch.randn(B, D, generator=g)
        lv = -6.0 + 2.0 * torch.randn(B, D, generator=g)
    eps = torch.randn(B, D, generator=g)
    return mu, lv, eps


@pytest.mark.parametrize("B,D,parts,family,estimator", [
    (256, 128, 2, "base", "mss"),
    (384, 64, 4, "sharp", "mws"),
    (296, 20, 4, "base", "mss"),
    (296, 22, 4, "sharp", "mss"),            # d % 4 != 0: the scalar gather
    (512, 128, 8, "sharp", "mws"),
])
def test_decomp_peer_entry_points_emulated_on_one_gpu(B, D, parts, family, estimator):
    from intro_tc_vae_b200 import _lib, ops
    lib = _lib.load()
    N, beta = 16704, 3.5
    flags = (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | _lib.VAR_COL | _lib.SAVE_FOR_BACKWARD
    mu_c, lv_c, eps_c = _latents(B, D, family, seed=B + D)
    mu, lv = mu_c.to(DEV), lv_c.to(DEV)
    z = ops.reparameterize(mu, lv, eps_c.to(DEV))
    w = [torch.linspace(a, b, B, device=DEV) for a, b in ((0.2, 1.7), (-0.5, 0.5), (0.9, -0.3), (0.1, 0.6))]
    c = torch.tensor([0.7, -1.3, 0.4, 2.1], device=DEV)               # upstream gradient of every rank's four means
    b_loc = B // parts
    shards = [slice(r * b_loc, (r + 1) * b_loc) for r in range(parts)]

    # unsharded reference: the custom op on the global batch, each rank's means formed from its rows of the reference
    zf, muf, lvf = (t.clone().requires_grad_(True) for t in (z, mu, lv))
    rows_f = torch.ops.tcelbo.decomp_forward(zf, muf, lvf, 0, N, flags, beta)[:4]
    ref_means = [torch.stack([r[s].mean() for r in rows_f]) for s in shards]
    (sum((r * wk).sum() for r, wk in zip(rows_f, w)) + sum((c * m).sum() for m in ref_means)).backward()

    ws_bytes = lib.tcelbo_workspace_bytes(b_loc, B, D, flags)
    sc_bytes = lib.tcelbo_backward_scratch_bytes(b_loc, B, D, flags)
    st = torch.cuda.current_stream().cuda_stream
    P = lambda t: t.data_ptr()                                         # noqa: E731
    zs, mus, lvs = ([t[s].contiguous() for s in shards] for t in (z, mu, lv))
    pub_mu, pub_lv = [torch.empty(b_loc, D, device=DEV) for _ in range(parts)], [torch.empty(b_loc, D, device=DEV) for _ in range(parts)]
    for r in range(parts):                                             # without a sync struct the publish is a plain copy
        _lib.check(lib.tcelbo_peer_publish_mu_logvar(P(mus[r]), D, P(lvs[r]), D, b_loc, D, P(pub_mu[r]), P(pub_lv[r]), None, st),
                   "publish")
    mu_table = torch.tensor([P(t) for t in pub_mu], dtype=torch.int64, device=DEV)
    lv_table = torch.tensor([P(t) for t in pub_lv], dtype=torch.int64, device=DEV)
    ws = [torch.empty(ws_bytes, dtype=torch.uint8, device=DEV) for _ in range(parts)]
    scratch = [torch.empty(sc_bytes, dtype=torch.uint8, device=DEV) for _ in range(parts)]
    sc_table = torch.tensor([P(t) for t in scratch], dtype=torch.int64, device=DEV)
    rows = [[torch.empty(b_loc, device=DEV) for _ in range(4)] for _ in range(parts)]
    means = [torch.empty(4, device=DEV) for _ in range(parts)]
    for r in range(parts):
        n0 = lib.tcelbo_launch_count()
        _lib.check(lib.tcelbo_decomp_forward_peer(P(zs[r]), D, P(mus[r]), D, P(lvs[r]), D, P(mu_table), P(lv_table), D,
                                                  b_loc, parts, r, D, N, flags, beta, *[P(t) for t in rows[r]], P(means[r]),
                                                  None, P(ws[r]), ws_bytes, st), "decomp_forward_peer")
        assert lib.tcelbo_launch_count() - n0 == 3
    for k in range(4):
        assert _relerr(torch.cat([rows[r][k] for r in range(parts)]), rows_f[k]) < 2e-6
    for r, s in enumerate(shards):
        assert _relerr(means[r], ref_means[r]) < 2e-6
        # the gather packs the same column operands as the all-gathered call: the shard's outputs are bit-identical
        *rows_nccl, means_nccl, _ = torch.ops.tcelbo.decomp_forward(zs[r], mu, lv, s.start, N, flags, beta)
        assert all(torch.equal(a, b) for a, b in zip(rows[r], rows_nccl)) and torch.equal(means[r], means_nccl)

    gs = [[wk[s].contiguous() for wk in w] for s in shards]
    gz, gmu, glv = ([torch.empty(b_loc, D, device=DEV) for _ in range(parts)] for _ in range(3))
    for phase, launches in ((_lib.PEER_SWEEP, 2), (_lib.PEER_FINISH, 1)):
        for r in range(parts):
            n0 = lib.tcelbo_launch_count()
            _lib.check(lib.tcelbo_decomp_backward_peer(phase, P(zs[r]), D, P(mus[r]), D, P(lvs[r]), D, b_loc, parts, r, D, N, flags, beta,
                                                       *[P(t) for t in gs[r]], P(c), P(gz[r]), D, P(gmu[r]), D, P(glv[r]), D,
                                                       P(ws[r]), ws_bytes, P(scratch[r]), sc_bytes, P(sc_table), None, st),
                       "decomp_backward_peer")
            assert lib.tcelbo_launch_count() - n0 == launches
    assert _relerr(torch.cat(gz), zf.grad) < 1e-5
    assert _relerr(torch.cat(gmu), muf.grad) < 1e-5
    assert _relerr(torch.cat(glv), lvf.grad) < 1e-5


def test_two_gpu_decomp_peer_equals_nccl_and_single_when_available():
    """tools/check_decomp_peer.py under torchrun: NCCL-sharded == peer-sharded == single GPU for the decomposition, three rounds
    of buffer rotation, the simple and the decomposition loss interleaved on one exchange, and the solver with only
    peer_exchange set.  Needs two visible GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tools", "check_decomp_peer.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MISMATCH" not in out.stdout
