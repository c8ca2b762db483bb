"""The fused MI / TC / dimension-wise KL decomposition (ops.tc_decomp_loss_terms / tc_decomp_loss_mean, the custom ops
tcelbo::decomp_forward / decomp_backward) against the reference's outputs and against the composition it replaces:
ops.row_log_density twice and ops.tc_terms(var_of="col") combined in torch (solvers/tc.py:91-144)."""
import numpy as np
import pytest
import torch

from cases import CASES, make_inputs

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-5
GRAD_RTOL = 1e-4
FINITE_CASES = [c for c in CASES if not c.startswith("nan_")]
DEV = "cuda:0"


def _ops():
    from intro_tc_vae_b200 import ops
    return ops


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
    return mu, lv, eps


def _flags(estimator, save=True):
    from intro_tc_vae_b200 import _lib
    return (_lib.EST_MSS if estimator == "mss" else _lib.EST_MWS) | _lib.VAR_COL | (_lib.SAVE_FOR_BACKWARD if save else 0)


def _composition(z, mu, lv, N, beta, estimator):
    """solvers/tc.py:91-144 per sample, from the separate ops -> (loss, mi, tc, dimkl)."""
    ops = _ops()
    condx = ops.row_log_density(z, mu, lv)
    pz = ops.row_log_density(z)
    prod, joint = ops.tc_terms(z, mu, lv, N, estimator, "col")
    mi, tc, dimkl = condx - joint, joint - prod, prod - pz
    return mi + beta * tc + dimkl, mi, tc, dimkl


@pytest.mark.parametrize("name", FINITE_CASES)
def test_golden_mean_and_gradients(golden, name):
    ops = _ops()
    case = CASES[name]
    N, beta = case["N"], case["beta"]
    pre = f"{name}/f32/"
    mu_np, lv_np, eps_np = make_inputs(case)
    mu = torch.tensor(mu_np, dtype=torch.float32, device=DEV, requires_grad=True)
    lv = torch.tensor(lv_np, dtype=torch.float32, device=DEV, requires_grad=True)
    z = ops.reparameterize(mu, lv, torch.tensor(eps_np, dtype=torch.float32, device=DEV))
    loss, mi, tc, dimkl = ops.tc_decomp_loss_mean(z, mu, lv, N, beta)
    assert loss.dim() == mi.dim() == tc.dim() == dimkl.dim() == 0
    ref = float(golden[pre + "full_mean"])
    assert abs(loss.item() - ref) < LOSS_RTOL * abs(ref)
    assert abs((mi + beta * tc + dimkl).item() - ref) < LOSS_RTOL * abs(ref)
    loss.backward()
    assert _relerr(mu.grad, golden[pre + "full_mean_dmu"]) < GRAD_RTOL
    assert _relerr(lv.grad, golden[pre + "full_mean_dlv"]) < GRAD_RTOL


@pytest.mark.parametrize("B,D", [(256, 128), (96, 32), (48, 256), (1000, 128)])
@pytest.mark.parametrize("family", ["base", "sharp"])
@pytest.mark.parametrize("estimator", ["mss", "mws"])
def test_fused_equals_composition(B, D, family, estimator):
    """Every per-row term and mean, and the gradients of a weighted sum of all eight outputs."""
    N, beta = 16704, 4.5
    mu_c, lv_c, eps_c = _latents(B, D, family, seed=41)
    w = [torch.linspace(a, b, B, device=DEV) for a, b in ((0.2, 1.7), (-0.5, 0.5), (0.9, -0.3), (0.1, 0.6))]
    c = (0.7, -1.3, 0.4, 2.1)
    outs = []
    for fused in (False, True):
        mu = mu_c.to(DEV).requires_grad_(True)
        lv = lv_c.to(DEV).requires_grad_(True)
        z = _ops().reparameterize(mu, lv, eps_c.to(DEV))
        if fused:
            *rows, means, _ = torch.ops.tcelbo.decomp_forward(z, mu, lv, 0, N, _flags(estimator), beta)
            means = means.unbind(0)
        else:
            rows = _composition(z, mu, lv, N, beta, estimator)
            means = [r.mean() for r in rows]
        (sum((r * wk).sum() for r, wk in zip(rows, w)) + sum(ck * m for ck, m in zip(c, means))).backward()
        outs.append(([r.detach() for r in rows], torch.stack([m.detach() for m in means]), mu.grad, lv.grad))
    (rows0, means0, gmu0, glv0), (rows1, means1, gmu1, glv1) = outs
    for r1, r0 in zip(rows1, rows0):
        assert _relerr(r1, r0) < 2e-6
    assert _relerr(means1, means0) < 2e-6
    assert _relerr(gmu1, gmu0) < 1e-5
    assert _relerr(glv1, glv0) < 1e-5


def test_row_densities_are_those_of_row_log_density():
    """condx and pz come from the same element formula as ops.row_log_density: mi + log_qz and log_qz_prod - dimkl
    reproduce them up to the rounding of the two subtractions."""
    ops = _ops()
    B, D, N = 300, 130, 16704
    mu_c, lv_c, eps_c = _latents(B, D, "sharp", seed=11)
    mu, lv = mu_c.to(DEV), lv_c.to(DEV)
    z = ops.reparameterize(mu, lv, eps_c.to(DEV))
    _, mi, tc, dimkl = ops.tc_decomp_loss_terms(z, mu, lv, N, 2.0)
    prod, joint = ops.tc_terms(z, mu, lv, N, "mss", "col")
    assert torch.equal(tc, joint - prod)
    assert _relerr(mi + joint, ops.row_log_density(z, mu, lv)) < 1e-6
    assert _relerr(prod - dimkl, ops.row_log_density(z)) < 1e-6


def test_nan_positions_match_composition():
    """N < B-1: the stratified weight is negative and its log NaN, as in the reference."""
    ops = _ops()
    case = CASES["nan_B8_D4"]
    mu_np, lv_np, eps_np = make_inputs(case)
    mu, lv, eps = (torch.tensor(a, dtype=torch.float32, device=DEV) for a in (mu_np, lv_np, eps_np))
    z = ops.reparameterize(mu, lv, eps)
    fused = ops.tc_decomp_loss_terms(z, mu, lv, case["N"], case["beta"])
    comp = _composition(z, mu, lv, case["N"], case["beta"], "mss")
    for f, c in zip(fused, comp):
        assert torch.equal(torch.isnan(f), torch.isnan(c))
    assert torch.isnan(fused[0]).any()
    assert all(torch.isnan(m) for m in ops.tc_decomp_loss_mean(z, mu, lv, case["N"], case["beta"])[:1])


@pytest.mark.parametrize("estimator", ["mss", "mws"])
def test_row_sharding_emulated_on_one_gpu(estimator):
    """Rank r owns rows [r*B/P, (r+1)*B/P) and sees all of mu / logvar: four shards through the custom op with row_offset give
    the unsharded rows, the unsharded gradients once the column gradients are summed, and the unsharded means on average."""
    B, D, N, beta, parts = 256, 64, 16704, 3.0, 4
    mu_c, lv_c, eps_c = _latents(B, D, "base", seed=7)
    mu, lv = mu_c.to(DEV), lv_c.to(DEV)
    z = _ops().reparameterize(mu, lv, eps_c.to(DEV))
    w = [torch.linspace(a, b, B, device=DEV) for a, b in ((0.5, 1.5), (-0.3, 0.8), (1.1, 0.2), (0.4, -0.6))]
    zf, muf, lvf = (t.clone().requires_grad_(True) for t in (z, mu, lv))
    *rows_f, means_f, _ = torch.ops.tcelbo.decomp_forward(zf, muf, lvf, 0, N, _flags(estimator), beta)
    sum((r * wk).sum() for r, wk in zip(rows_f, w)).backward()

    rows_s, means_s, gz_s = [[] for _ in range(4)], [], []
    gmu_sum, glv_sum = torch.zeros(B, D, device=DEV), torch.zeros(B, D, device=DEV)
    b_loc = B // parts
    for r in range(parts):
        lo, hi = r * b_loc, (r + 1) * b_loc
        zr = z[lo:hi].clone().requires_grad_(True)
        mua, lva = mu.clone().requires_grad_(True), lv.clone().requires_grad_(True)
        *rows, means, _ = torch.ops.tcelbo.decomp_forward(zr, mua, lva, lo, N, _flags(estimator), beta)
        sum((rk * wk[lo:hi]).sum() for rk, wk in zip(rows, w)).backward()
        for k in range(4):
            rows_s[k].append(rows[k].detach())
        means_s.append(means.detach())
        gz_s.append(zr.grad)
        gmu_sum += mua.grad
        glv_sum += lva.grad
    for k in range(4):
        assert _relerr(torch.cat(rows_s[k]), rows_f[k]) < 1e-6
    assert _relerr(torch.stack(means_s).mean(0), means_f) < 2e-6
    assert _relerr(torch.cat(gz_s), zf.grad) < 1e-5
    assert _relerr(gmu_sum, muf.grad) < 1e-5
    assert _relerr(glv_sum, lvf.grad) < 1e-5


def test_three_library_launches_each_way():
    from intro_tc_vae_b200 import _lib
    ops = _ops()
    lib = _lib.load()
    B, D, N = 512, 128, 16704
    mu_c, lv_c, eps_c = _latents(B, D, "base", seed=3)
    mu, lv = mu_c.to(DEV).requires_grad_(True), lv_c.to(DEV).requires_grad_(True)
    z = ops.reparameterize(mu, lv, eps_c.to(DEV)).detach().requires_grad_(True)    # a leaf: no reparameterize backward below
    for form in (ops.tc_decomp_loss_mean, ops.tc_decomp_loss_terms):
        n0 = lib.tcelbo_launch_count()
        loss = form(z, mu, lv, N, 6.0)[0]
        n1 = lib.tcelbo_launch_count()
        grads = torch.autograd.grad(loss.sum(), [z, mu, lv])
        n2 = lib.tcelbo_launch_count()
        assert (n1 - n0, n2 - n1) == (3, 3)
        assert all(torch.isfinite(g).all() for g in grads)


def test_cuda_graph_replay_equals_eager():
    """Forward and backward captured in one CUDA graph and replayed on new inputs give the eager results: nothing in the op
    synchronises with the host."""
    ops = _ops()
    B, D, N, beta = 320, 64, 16704, 5.0
    static = [torch.zeros(B, D, device=DEV) for _ in range(3)]        # mu, logvar, eps

    def step(mu_in, lv_in, eps_in):
        mu, lv = mu_in.detach().requires_grad_(True), lv_in.detach().requires_grad_(True)
        z = ops.reparameterize(mu, lv, eps_in)
        loss, mi, tc, dimkl = ops.tc_decomp_loss_mean(z, mu, lv, N, beta)
        rows = ops.tc_decomp_loss_terms(z, mu, lv, N, beta)
        gmu, glv = torch.autograd.grad(loss + 0.5 * mi - 0.25 * dimkl + (rows[2] * 0.01).sum(), [mu, lv])
        return torch.stack([loss, mi, tc, dimkl]).detach(), rows[0].detach(), gmu, glv

    for t, v in zip(static, _latents(B, D, "base", seed=100)):
        t.copy_(v)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step(*static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out_static = step(*static)
    for seed, family in ((101, "base"), (102, "sharp")):
        fresh = _latents(B, D, family, seed=seed)
        for t, v in zip(static, fresh):
            t.copy_(v)
        graph.replay()
        want = step(*(v.to(DEV) for v in fresh))
        torch.cuda.synchronize()
        for got, ref in zip(out_static, want):
            assert _relerr(got, ref) < 1e-6


def test_solver_full_path_reduce_none_and_errors():
    """TCLossMixin._compute_kl_loss_full with reduce="none" returns the per-sample loss of the composition; the error
    conventions of tc_terms hold (B == 1 under MSS divides by zero, D > 512 is outside the kernels)."""
    from intro_tc_vae_b200.solvers.tc import TCLossMixin
    ops = _ops()

    class Solver:
        process_group = None
        beta_kl = 3.0
        dataset = range(16704)
        written = []

        def write_scalar(self, it, tag, value):
            self.written.append(tag)

    B, D = 200, 48
    mu_c, lv_c, eps_c = _latents(B, D, "base", seed=5)
    mu, lv = mu_c.to(DEV), lv_c.to(DEV)
    z = ops.reparameterize(mu, lv, eps_c.to(DEV))
    s = Solver()
    per = TCLossMixin._compute_kl_loss_full(s, z, mu, lv, "none", None, True)
    assert per.shape == (B,) and s.written == ["kl_loss_unscaled"]
    assert _relerr(per, _composition(z, mu, lv, 16704, 3.0, "mss")[0]) < 2e-6
    one = torch.zeros(1, 8, device=DEV)
    with pytest.raises(ZeroDivisionError):
        ops.tc_decomp_loss_terms(one, one, one, 10, 2.0)
    ops.tc_decomp_loss_terms(one, one, one, 10, 2.0, "mws")             # MWS has no B-1
    big = torch.zeros(4, 520, device=DEV)
    with pytest.raises(NotImplementedError):
        ops.tc_decomp_loss_terms(big, big, big, 10, 2.0)
