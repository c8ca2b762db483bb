"""The fused training step of the MI / TC / dimension-wise KL decomposition: tcelbo_decomp_forward_ex / _backward_ex with the
reparameterize and exp-ELBO fusions, their peer pair, losses.tc_decomp_exp_elbo, GraphedKLLoss(loss="decomp") and
SoftIntroTCStep(kl_loss="full"), against the unfused ops they replace, the golden values and the reference's train step."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from cases import CASES, make_inputs

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FINITE_CASES = [c for c in CASES if not c.startswith("nan_")]


def _relerr(a, b):
    a = np.asarray(a.detach().cpu() if torch.is_tensor(a) else a, dtype=np.float64)
    b = np.asarray(b.detach().cpu() if torch.is_tensor(b) else b, dtype=np.float64)
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
    return mu.to(DEV), lv.to(DEV), eps.to(DEV)


def _flags(estimator):
    from intro_tc_vae_b200 import _lib
    return (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | _lib.VAR_COL | _lib.SAVE_FOR_BACKWARD


P = lambda t: t.data_ptr() if t is not None else None                     # noqa: E731


def _st():
    return torch.cuda.current_stream().cuda_stream


class _Ex:
    """One single-GPU tcelbo_decomp_forward_ex / _backward_ex evaluation with its own buffers."""

    def __init__(self, mu, lv, N, beta, flags, z=None, eps=None, rec=None, scale=0.0):
        from intro_tc_vae_b200 import _lib
        self.lib, self._lib = _lib.load(), _lib
        B, D = mu.shape
        self.args = (mu, lv, B, D, N, beta, flags)
        self.z, self.eps, self.scale = z, eps, scale
        self.ws = torch.empty(self.lib.tcelbo_workspace_bytes(B, B, D, flags), dtype=torch.uint8, device=DEV)
        self.rows = [torch.empty(B, device=DEV) for _ in range(4)]
        self.means = torch.empty(4, device=DEV)
        self.z_out = torch.empty(B, D, device=DEV) if eps is not None else None
        self.e_rows = torch.empty(B, device=DEV) if rec is not None else None
        self.expelbo = torch.empty((), device=DEV) if rec is not None else None
        fz = _lib.Fusion(eps=P(eps), ldeps=D, z_out=P(self.z_out), ldz_out=D, rec_rows=P(rec), scale=scale,
                         expelbo=P(self.expelbo), e_rows=P(self.e_rows))
        _lib.check(self.lib.tcelbo_decomp_forward_ex(P(z), D, P(mu), D, P(lv), D, B, B, 0, D, N, flags, beta,
                                                     *[P(t) for t in self.rows], P(self.means), ctypes.byref(fz),
                                                     P(self.ws), self.ws.numel(), _st()), "tcelbo_decomp_forward_ex")

    def backward(self, g_rows=(None,) * 4, g_means=None, g_expelbo=None):
        mu, lv, B, D, N, beta, flags = self.args
        sc = torch.empty(self.lib.tcelbo_backward_scratch_bytes(B, B, D, flags), dtype=torch.uint8, device=DEV)
        gz, gmu, glv = (torch.empty(B, D, device=DEV) for _ in range(3))
        g_rec = torch.empty(B, device=DEV) if g_expelbo is not None else None
        fb = self._lib.Fusion(eps=P(self.eps), ldeps=D, scale=self.scale, e_rows=P(self.e_rows), g_expelbo=P(g_expelbo),
                              g_rec_rows=P(g_rec))
        self._lib.check(self.lib.tcelbo_decomp_backward_ex(P(self.z), D, P(mu), D, P(lv), D, B, B, 0, D, N, flags, beta,
                                                           *[P(t) for t in g_rows], P(g_means), ctypes.byref(fb),
                                                           P(gz), D, P(gmu), D, P(glv), D, P(self.ws), self.ws.numel(),
                                                           P(sc), sc.numel(), _st()), "tcelbo_decomp_backward_ex")
        return gz, gmu, glv, g_rec


@pytest.mark.parametrize("B,D", [(3, 20), (64, 128), (1000, 256), (300, 22)])
@pytest.mark.parametrize("family", ["base", "sharp"])
def test_fused_reparameterize_and_expelbo_forward_are_bit_identical(B, D, family):
    """z_out is tcelbo_reparam_forward's z; the four per-row terms and the means equal the plain forward on that z bit for bit,
    and asking for the exp-ELBO changes none of them."""
    from intro_tc_vae_b200 import ops
    N, beta, scale = 16704, 3.0, 1.0 / 768
    mu, lv, eps = _latents(B, D, family, seed=B + D)
    z = ops.reparameterize(mu, lv, eps)
    rec = torch.rand(B, device=DEV) * 50.0
    plain = _Ex(mu, lv, N, beta, _flags("mss"), z=z)
    fused = _Ex(mu, lv, N, beta, _flags("mss"), eps=eps)
    both = _Ex(mu, lv, N, beta, _flags("mss"), eps=eps, rec=rec, scale=scale)
    torch.cuda.synchronize()
    assert torch.equal(fused.z_out, z) and torch.equal(both.z_out, z)
    for ex in (fused, both):
        for a, b in zip(ex.rows + [ex.means], plain.rows + [plain.means]):
            assert torch.equal(a, b)
    e_ref = torch.exp(-2.0 * scale * (rec + plain.rows[0]))
    assert _relerr(both.e_rows, e_ref) < 1e-6
    assert _relerr(both.expelbo, e_ref.mean()) < 1e-6


@pytest.mark.parametrize("B", [3, 64, 1000])
@pytest.mark.parametrize("D", [20, 128, 256])
@pytest.mark.parametrize("family", ["base", "sharp"])
@pytest.mark.parametrize("estimator", ["mss", "mws"])
def test_fused_reparameterize_gradients_match_autograd(B, D, family, estimator):
    """With eps, grad_mu / grad_logvar are the gradients w.r.t. the encoder outputs: those of autograd through ops.reparameterize
    and ops.tc_decomp_loss_mean (a weighted sum of the four means)."""
    from intro_tc_vae_b200 import ops
    N, beta = 16704, 4.5
    mu_c, lv_c, eps = _latents(B, D, family, seed=3 * B + D)
    c = torch.tensor([1.0, 0.3, -0.7, 0.2], device=DEV)
    mu, lv = mu_c.clone().requires_grad_(True), lv_c.clone().requires_grad_(True)
    z = ops.reparameterize(mu, lv, eps)
    means = torch.stack(ops.tc_decomp_loss_mean(z, mu, lv, N, beta, estimator))
    (c * means).sum().backward()
    ex = _Ex(mu_c, lv_c, N, beta, _flags(estimator), eps=eps)
    gz, gmu, glv, _ = ex.backward(g_means=c)
    # the column sums are accumulated with fp32 red.global in launch-dependent order: at B = 1000 that alone moves the op's own
    # grad_mu by ~1e-6 (max-norm) from one run to the next, so the bound there is the run-to-run spread, not the formula
    tol = 1e-6 if B <= 64 else 3e-6
    assert _relerr(gmu, mu.grad) <= tol
    assert _relerr(glv, lv.grad) <= tol


@pytest.mark.parametrize("B,D", [(64, 128), (500, 32)])
def test_decomp_exp_elbo_matches_the_composition(B, D):
    """losses.tc_decomp_exp_elbo == tc_decomp_loss_terms + losses.exp_elbo: value, the gradients of mu / logvar through z and
    g_rec_rows (= the gradient of rec_per_sample)."""
    from intro_tc_vae_b200 import losses, ops
    N, beta, scale = 16704, 256.0, 1.0 / 3072
    mu_c, lv_c, eps = _latents(B, D, "base", seed=B)
    rec_c = 20.0 + 10.0 * torch.rand(B, device=DEV)
    outs = []
    for fused in (False, True):
        mu, lv, rec = (t.clone().requires_grad_(True) for t in (mu_c, lv_c, rec_c))
        z = ops.reparameterize(mu, lv, eps)
        if fused:
            ee, rows = losses.tc_decomp_exp_elbo(z, mu, lv, rec, N, beta, scale)
        else:
            rows = ops.tc_decomp_loss_terms(z, mu, lv, N, beta)[0]
            ee = losses.exp_elbo(rec, rows, scale)
        (3.0 * ee).backward()
        outs.append((ee.detach(), rows.detach(), mu.grad, lv.grad, rec.grad))
    (e0, r0, gm0, gl0, gr0), (e1, r1, gm1, gl1, gr1) = outs
    assert torch.equal(r1, r0)
    assert _relerr(e1, e0) < 1e-6
    assert _relerr(gr1, gr0) < 1e-6
    assert _relerr(gm1, gm0) < 1e-5
    assert _relerr(gl1, gl0) < 1e-5
    # the exp-ELBO enters the backward prologue through the same coefficients as a per-row gradient of the loss
    ex = _Ex(mu_c, lv_c, N, beta, _flags("mss"), eps=eps, rec=rec_c, scale=scale)
    g = torch.tensor(3.0, device=DEV)
    _, gmu_a, glv_a, g_rec = ex.backward(g_expelbo=g)
    _, gmu_b, glv_b, _ = ex.backward(g_rows=(g_rec, None, None, None))
    assert torch.equal(g_rec, gr1)
    assert _relerr(gmu_a, gmu_b) < 1e-6 and _relerr(glv_a, glv_b) < 1e-6


@pytest.mark.parametrize("name", FINITE_CASES)
def test_graphed_decomp_step_reproduces_golden(golden, name):
    from intro_tc_vae_b200.graphs import GraphedKLLoss
    case = CASES[name]
    pre = f"{name}/f32/"
    mu, lv, eps = (torch.tensor(a, dtype=torch.float32, device=DEV) for a in make_inputs(case))
    B, D = mu.shape
    g = GraphedKLLoss(B, D, case["N"], case["beta"], DEV, loss="decomp")
    loss, dmu, dlv = g(mu, lv, eps)
    torch.cuda.synchronize()
    ref = float(golden[pre + "full_mean"])
    assert abs(loss.item() - ref) < 1e-5 * abs(ref)
    assert _relerr(dmu, golden[pre + "full_mean_dmu"]) < 1e-4
    assert _relerr(dlv, golden[pre + "full_mean_dlv"]) < 1e-4


@pytest.mark.parametrize("B,D,estimator", [(64, 128, "mss"), (1024, 128, "mws"), (200, 20, "mss")])
@pytest.mark.parametrize("capture", [True, False])
def test_graphed_decomp_direct_equals_autograd_and_launches_six_kernels(B, D, estimator, capture):
    from intro_tc_vae_b200 import _lib
    from intro_tc_vae_b200.graphs import GraphedKLLoss
    lib = _lib.load()
    N, beta = 16704, 6.0
    direct = GraphedKLLoss(B, D, N, beta, DEV, estimator=estimator, loss="decomp", capture=capture)
    auto = GraphedKLLoss(B, D, N, beta, DEV, estimator=estimator, loss="decomp", mode="autograd", capture=capture)
    for seed, family in ((1, "base"), (2, "sharp"), (3, "base")):
        a = _latents(B, D, family, seed)
        l0, dm0, dl0 = (t.clone() for t in direct(*a))
        l1, dm1, dl1 = (t.clone() for t in auto(*a))
        torch.cuda.synchronize()
        tol = 1e-6 if B <= 64 else 3e-6              # red.global order of the column sums (see the gradient test above)
        assert _relerr(l0, l1) < 1e-6
        assert _relerr(dm0, dm1) < tol
        assert _relerr(dl0, dl1) < tol
    if not capture:
        n0 = lib.tcelbo_launch_count()
        direct.replay()
        assert lib.tcelbo_launch_count() - n0 == 6


@pytest.mark.parametrize("B,D,parts,family", [(256, 128, 2, "base"), (296, 20, 4, "sharp"), (512, 64, 4, "base")])
def test_peer_ex_pair_emulated_on_one_gpu(B, D, parts, family):
    """P ranks played one after the other through tcelbo_decomp_forward_peer_ex / _backward_peer_ex with eps and the exp-ELBO
    (sync = NULL, plain allocations for the mapped buffers) against one unsharded _ex call on the global batch.  Each rank's means
    and exp-ELBO cover its rows; with equal shards their gradients c and ge are the global ones P*c and P*ge."""
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    N, beta, scale = 16704, 2.5, 1.0 / 768
    flags = _flags("mss")
    mu, lv, eps = _latents(B, D, family, seed=B + parts)
    rec = 10.0 + 20.0 * torch.rand(B, device=DEV)
    c = torch.tensor([0.7, -1.3, 0.4, 2.1], device=DEV)
    ge = torch.tensor(0.8, device=DEV)
    full = _Ex(mu, lv, N, beta, flags, eps=eps, rec=rec, scale=scale)
    gz_f, gmu_f, glv_f, grec_f = full.backward(g_means=parts * c, g_expelbo=parts * ge)

    b_loc = B // parts
    shards = [slice(r * b_loc, (r + 1) * b_loc) for r in range(parts)]
    mus, lvs, epss, recs = ([t[s].contiguous() for s in shards] for t in (mu, lv, eps, rec))
    pub_mu = [t.clone() for t in mus]                          # what tcelbo_peer_publish_mu_logvar leaves in the mapped buffers
    pub_lv = [t.clone() for t in lvs]
    mu_table = torch.tensor([P(t) for t in pub_mu], dtype=torch.int64, device=DEV)
    lv_table = torch.tensor([P(t) for t in pub_lv], dtype=torch.int64, device=DEV)
    ws_bytes, sc_bytes = lib.tcelbo_workspace_bytes(b_loc, B, D, flags), lib.tcelbo_backward_scratch_bytes(b_loc, B, D, flags)
    ws = [torch.empty(ws_bytes, dtype=torch.uint8, device=DEV) for _ in range(parts)]
    scratch = [torch.empty(sc_bytes, dtype=torch.uint8, device=DEV) for _ in range(parts)]
    sc_table = torch.tensor([P(t) for t in scratch], dtype=torch.int64, device=DEV)
    rows = [[torch.empty(b_loc, device=DEV) for _ in range(4)] for _ in range(parts)]
    means = [torch.empty(4, device=DEV) for _ in range(parts)]
    z_out = [torch.empty(b_loc, D, device=DEV) for _ in range(parts)]
    e_rows = [torch.empty(b_loc, device=DEV) for _ in range(parts)]
    expelbo = [torch.empty((), device=DEV) for _ in range(parts)]
    keep = []
    for r in range(parts):
        fz = _lib.Fusion(eps=P(epss[r]), ldeps=D, z_out=P(z_out[r]), ldz_out=D, rec_rows=P(recs[r]), scale=scale,
                         expelbo=P(expelbo[r]), e_rows=P(e_rows[r]))
        n0 = lib.tcelbo_launch_count()
        _lib.check(lib.tcelbo_decomp_forward_peer_ex(None, 0, P(mus[r]), D, P(lvs[r]), D, P(mu_table), P(lv_table), D, b_loc, parts, r,
                                                     D, N, flags, beta, *[P(t) for t in rows[r]], P(means[r]), ctypes.byref(fz),
                                                     None, P(ws[r]), ws_bytes, _st()), "decomp_forward_peer_ex")
        assert lib.tcelbo_launch_count() - n0 == 3
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(z_out), full.z_out)
    for k in range(4):
        assert _relerr(torch.cat([rows[r][k] for r in range(parts)]), full.rows[k]) < 2e-6
    assert _relerr(torch.cat(e_rows), full.e_rows) < 2e-6
    for r, s in enumerate(shards):
        assert _relerr(means[r], torch.stack([t[s].mean() for t in full.rows])) < 2e-6
        assert _relerr(expelbo[r], full.e_rows[s].mean()) < 2e-6

    gz, gmu, glv = ([torch.empty(b_loc, D, device=DEV) for _ in range(parts)] for _ in range(3))
    g_rec = [torch.empty(b_loc, device=DEV) for _ in range(parts)]
    for phase, launches in ((_lib.PEER_SWEEP, 2), (_lib.PEER_FINISH, 1)):
        for r in range(parts):
            fb = _lib.Fusion(eps=P(epss[r]), ldeps=D, scale=scale, e_rows=P(e_rows[r]), g_expelbo=P(ge), g_rec_rows=P(g_rec[r]))
            keep.append(fb)
            n0 = lib.tcelbo_launch_count()
            _lib.check(lib.tcelbo_decomp_backward_peer_ex(phase, None, 0, P(mus[r]), D, P(lvs[r]), D, b_loc, parts, r, D, N, flags, beta,
                                                          None, None, None, None, P(c), P(gz[r]), D, P(gmu[r]), D, P(glv[r]), D,
                                                          P(ws[r]), ws_bytes, P(scratch[r]), sc_bytes, P(sc_table), ctypes.byref(fb),
                                                          None, _st()), "decomp_backward_peer_ex")
            assert lib.tcelbo_launch_count() - n0 == launches
    torch.cuda.synchronize()
    assert _relerr(torch.cat(g_rec), grec_f) < 1e-6
    assert _relerr(torch.cat(gz), gz_f) < 1e-5
    assert _relerr(torch.cat(gmu), gmu_f) < 1e-5
    assert _relerr(torch.cat(glv), glv_f) < 1e-5


@pytest.mark.parametrize("capture", [False, True])
def test_graphed_soft_intro_full_step_matches_the_reference_train_step(capture):
    """SoftIntroTCStep(kl_loss="full") performs the update of the reference's IntroTCSovler.train_step with the instance's
    compute_kl_loss pointed at TCSovler._compute_kl_loss_full (the beta-TCVAE loss), on the same seeds; it also reports the
    encoder phase's mi / tc / dimkl means."""
    import types
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip("oracle/_ref not staged")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_reference_dropin_gpu import N_DATA, _build
    dev = torch.device(DEV)
    B = 48
    batch = torch.rand(B, 3, 16, 16, generator=torch.Generator().manual_seed(5))
    with ref_loader.on_path():
        from solvers.tc import TCSovler
        model, solver = _build("intro-tc", dev, installed=False)
        solver.compute_kl_loss = types.MethodType(TCSovler._compute_kl_loss_full, solver)
        torch.manual_seed(11)
        torch.cuda.manual_seed(11)
        noise = torch.randn(B, model.zdim)
        torch.manual_seed(11)
        init_params = [p.detach().clone() for p in model.parameters()]
        ref_out = solver.train_step(batch, 0)
        ref_params = [p.detach().clone() for p in model.parameters()]
    from intro_tc_vae_b200 import utils as fast_utils
    saved_writer = fast_utils.SingletonWriter
    try:
        with ref_loader.on_path():
            import models
            import intro_tc_vae_b200
            from intro_tc_vae_b200.train_step import SoftIntroTCStep
            intro_tc_vae_b200.install()
            torch.manual_seed(0)
            model = models.SoftIntroVAE(arch="conv", cdim=3, zdim=32, channels=(16, 32), image_size=16).to(dev)
            opt_e = torch.optim.Adam(model.encoder.parameters(), lr=2e-4, capturable=True)
            opt_d = torch.optim.Adam(model.decoder.parameters(), lr=2e-4, capturable=True)
            step = SoftIntroTCStep(model, opt_e, opt_d, N_DATA, batch.shape, recon_loss_type="mse", beta_kl=0.5, beta_rec=0.75,
                                   beta_neg=512.0, gamma_r=1e-8, clip=100.0, capture=capture, kl_loss="full")
            torch.cuda.manual_seed(11)
            out = step(batch.to(dev), noise.to(dev))
            step.check_finite()
            got = {k: v.item() for k, v in out.items()}
    finally:
        fast_utils.SingletonWriter = saved_writer
    for key, tol in (("loss_enc", 1e-4), ("loss_kl", 1e-4), ("loss_rec", 1e-4), ("loss_dec", 2e-3)):
        assert abs(got[key] - ref_out[key]) <= tol * max(abs(ref_out[key]), 1e-3), (capture, key, got[key], ref_out[key])
    assert abs((got["mi"] + 0.5 * got["tc"] + got["dimkl"]) - got["loss_kl"]) <= 1e-4 * max(abs(got["loss_kl"]), 1e-3)
    u_ref = torch.cat([(q - p0).flatten() for q, p0 in zip(ref_params, init_params)])
    u_got = torch.cat([(p.detach() - p0).flatten() for p, p0 in zip(model.parameters(), init_params)])
    cos = torch.dot(u_ref, u_got) / (u_ref.norm() * u_got.norm())
    assert cos.item() > 0.99, (capture, cos.item())


def test_soft_intro_full_step_without_the_reference():
    """SoftIntroTCStep(kl_loss="full"), graphed, on a small conv model of this file's own: the reported loss_kl is the decomposition's
    mean of the real batch's latents, mi + beta_kl*tc + dimkl, and a replay on new data stays finite."""
    from intro_tc_vae_b200.train_step import SoftIntroTCStep
    from intro_tc_vae_b200 import ops
    torch.manual_seed(0)
    zdim, B = 16, 32

    class Enc(torch.nn.Module):
        image_size = 8

        def __init__(self):
            super().__init__()
            self.f = torch.nn.Linear(3 * 8 * 8, 2 * zdim)

        def forward(self, x):
            return self.f(x.flatten(1))

    class Model(torch.nn.Module):
        cdim = 3

        def __init__(self):
            super().__init__()
            self.zdim = zdim
            self.encoder, self.decoder = Enc(), torch.nn.Sequential(torch.nn.Linear(zdim, 3 * 8 * 8), torch.nn.Sigmoid())

        def encode(self, x):
            mu, logvar = self.encoder(x).chunk(2, dim=1)
            return mu, logvar

        def decode(self, z):
            return self.decoder(z).view(-1, 3, 8, 8)

        def sample(self, z):
            return self.decode(z)

        def forward(self, x):
            mu, logvar = self.encode(x)
            z = ops.reparameterize(mu, logvar)
            return mu, logvar, z, self.decode(z)

    model = Model().to(DEV)
    opt_e = torch.optim.Adam(model.encoder.parameters(), lr=2e-4, capturable=True)
    opt_d = torch.optim.Adam(model.decoder.parameters(), lr=2e-4, capturable=True)
    step = SoftIntroTCStep(model, opt_e, opt_d, 5000, (B, 3, 8, 8), beta_kl=0.5, beta_neg=64.0, kl_loss="full")
    for seed in (1, 2):
        g = torch.Generator().manual_seed(seed)
        out = step(torch.rand(B, 3, 8, 8, generator=g).to(DEV), torch.randn(B, zdim, generator=g).to(DEV))
        step.check_finite()
        got = {k: v.item() for k, v in out.items()}
        assert all(np.isfinite(v) for v in got.values()), got
        assert abs(got["mi"] + 0.5 * got["tc"] + got["dimkl"] - got["loss_kl"]) <= 1e-4 * max(abs(got["loss_kl"]), 1.0)


def test_two_gpu_graphed_decomp_step_equals_single_when_available():
    """tools/check_decomp_step.py under torchrun: GraphedKLLoss(loss="decomp") with exchange="nccl" and "peer", replayed over three
    rounds of buffer rotation, equals the single-process step on the global batch.  Needs two visible GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(root, "tools", "check_decomp_step.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MISMATCH" not in out.stdout
