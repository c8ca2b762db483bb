"""CPU checks of the fused MI / TC / dimension-wise KL decomposition (tcelbo_decomp_forward / _backward).

The formulation the kernels implement is modelled in NumPy fp32 on top of the column-variance model of
oracle/kernel_model.py (forward_colvar / backward_colvar) and checked against the reference's own outputs for
TCSovler._compute_kl_loss_full (solvers/tc.py:91-144, golden ``full_mean*``) before any GPU runs it.  The C entry
points must refuse a call without TCELBO_VAR_COL or with null pointers before they touch a device.
"""
import numpy as np
import pytest

from cases import CASES, make_inputs
from oracle import kernel_model as K

F = np.float32
FINITE_CASES = [c for c in CASES if not c.startswith("nan_")]


def _lp(x, mu, lv):
    """Un-floored element density of ops.py:24-29 with the kernels' roundings (tc_common.cuh: lp_unfloored), unclamped,
    plus t = x - mu and iv = exp(-lv) for the gradient."""
    t = (x - mu).astype(F)
    iv = np.exp(-lv).astype(F)
    with np.errstate(invalid="ignore"):
        return F(-0.5) * ((t * t) * iv + lv + K.LOG_2PI), t, iv


def decomp_forward(z, mu_all, lv_all, dataset_size, beta, estimator="mss", row_offset=0):
    """Per-row loss / mi / tc / dimkl of the finalize kernel's decomposition mode, plus what the backward needs."""
    z, mu_all, lv_all = z.astype(F), mu_all.astype(F), lv_all.astype(F)
    fw = K.forward_colvar(z, mu_all, lv_all, dataset_size, estimator, row_offset)
    rows = slice(row_offset, row_offset + z.shape[0])
    lpc, t, iv = _lp(z, mu_all[rows], lv_all[rows])
    lp0, t0, iv0 = _lp(z, np.zeros_like(z), np.zeros_like(z))
    condx = np.fmax(lpc, F(-50)).sum(axis=1, dtype=F)
    pz = np.fmax(lp0, F(-50)).sum(axis=1, dtype=F)
    J, P = fw["log_qz"], fw["log_qz_prod"]
    mi, tc, dimkl = condx - J, J - P, P - pz
    loss = mi + F(beta) * tc + dimkl
    rowd = dict(lpc=lpc, t=t, iv=iv, lp0=lp0, t0=t0, iv0=iv0, rows=rows)
    return dict(loss=loss, mi=mi, tc=tc, dimkl=dimkl, fw=fw, rowd=rowd, beta=F(beta))


def decomp_backward(dec, b_glob, g_loss=None, g_mi=None, g_tc=None, g_dimkl=None, g_means=None):
    """(grad_z, grad_mu_all, grad_logvar_all): the backward prologue's composition, the unchanged column-variance sweep and
    the finalize kernel's row-local terms (masked where lp < -50)."""
    b = dec["loss"].shape[0]
    gm = np.zeros(4, F) if g_means is None else np.asarray(g_means, F)
    up = [np.zeros(b, F) if g is None else np.asarray(g, F) for g in (g_loss, g_mi, g_tc, g_dimkl)]
    gl, gmi, gtc, gdk = (u + gm[q] / F(b) for q, u in enumerate(up))
    beta = dec["beta"]
    gJ = (beta - F(1)) * gl - gmi + gtc
    gP = (F(1) - beta) * gl - gtc + gdk
    gc = gl + gmi
    gpz = -(gl + gdk)
    gz, gmu, glv = K.backward_colvar(dec["fw"], gJ, gP)
    r = dec["rowd"]
    gcm = np.where(r["lpc"] >= F(-50), gc[:, None], F(0))
    gpm = np.where(r["lp0"] >= F(-50), gpz[:, None], F(0))
    gz = gz + (-gcm * r["t"] * r["iv"]) + (-gpm * r["t0"] * r["iv0"])
    gmu, glv = gmu.copy(), glv.copy()
    gmu[r["rows"]] += gcm * r["t"] * r["iv"]
    glv[r["rows"]] += gcm * F(0.5) * (r["t"] * r["t"] * r["iv"] - F(1))
    assert gmu.shape[0] == b_glob
    return gz, gmu, glv


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize("name", FINITE_CASES)
def test_decomposition_model_matches_reference(golden, name):
    """mean_i(mi + beta*tc + dimkl) and its gradients w.r.t. the encoder's mu / logvar through z = mu + eps*exp(logvar/2)."""
    case = CASES[name]
    mu, lv, eps = (a.astype(F) for a in make_inputs(case))
    std = np.exp(F(0.5) * lv)
    z = (mu + eps * std).astype(F)
    B, N, beta = case["B"], case["N"], case["beta"]
    pre = f"{name}/f64/"
    dec = decomp_forward(z, mu, lv, N, beta)
    ref = float(golden[pre + "full_mean"])
    assert abs(float(dec["loss"].mean(dtype=F)) - ref) <= 1e-5 * abs(ref)
    assert abs(float((dec["mi"].mean(dtype=F) + F(beta) * dec["tc"].mean(dtype=F) + dec["dimkl"].mean(dtype=F))) - ref) <= 1e-5 * abs(ref)
    gz, gmu, glv = decomp_backward(dec, B, g_means=[1, 0, 0, 0])
    assert _rel(gmu + gz, golden[pre + "full_mean_dmu"]) <= 1e-4
    assert _rel(glv + gz * eps * std * F(0.5), golden[pre + "full_mean_dlv"]) <= 1e-4


def test_decomposition_model_gradients_of_every_output():
    """Upstream gradients on all four rows and all four means give the sum of the separate gradients (the composition is
    linear in them), and sharding the rows with row_offset reproduces the unsharded model."""
    case = CASES["ragged_B37_D20"]
    mu, lv, eps = (a.astype(F) for a in make_inputs(case))
    z = (mu + eps * np.exp(F(0.5) * lv)).astype(F)
    B, N, beta = case["B"], case["N"], case["beta"]
    rng = np.random.default_rng(0)
    rows = [rng.standard_normal(B).astype(F) for _ in range(4)]
    means = rng.standard_normal(4).astype(F)
    dec = decomp_forward(z, mu, lv, N, beta)
    total = decomp_backward(dec, B, *rows, g_means=means)
    parts = [decomp_backward(dec, B, **{k: rows[q]}) for q, k in enumerate(("g_loss", "g_mi", "g_tc", "g_dimkl"))]
    parts.append(decomp_backward(dec, B, g_means=means))
    for k in range(3):
        assert _rel(total[k], sum(p[k] for p in parts)) < 1e-5
    bounds = [0, 9, 20, 37]
    gmu_sum, glv_sum, gzs = np.zeros_like(mu), np.zeros_like(lv), []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        d = decomp_forward(z[lo:hi], mu, lv, N, beta, row_offset=lo)
        for key in ("loss", "mi", "tc", "dimkl"):
            assert _rel(d[key], dec[key][lo:hi]) < 1e-6
        gz, gmu, glv = decomp_backward(d, B, *(r[lo:hi] for r in rows))
        gzs.append(gz); gmu_sum += gmu; glv_sum += glv
    full = decomp_backward(dec, B, *rows)
    assert _rel(np.concatenate(gzs), full[0]) < 1e-5
    assert _rel(gmu_sum, full[1]) < 1e-5
    assert _rel(glv_sum, full[2]) < 1e-5


def _buf():
    return np.zeros(64, np.float32)


def test_decomp_entry_points_refuse_without_column_variance_or_with_null_pointers():
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    hold = [_buf() for _ in range(12)]
    P = [h.ctypes.data for h in hold]
    B, D, N = 4, 8, 100
    col = _lib.EST_MSS | _lib.VAR_COL | _lib.SAVE_FOR_BACKWARD

    def fwd(flags, inputs=(P[0], P[1], P[2]), outs=(P[3], P[4], P[5], P[6])):
        return lib.tcelbo_decomp_forward(inputs[0], D, inputs[1], D, inputs[2], D, B, B, 0, D, N, flags, 2.0,
                                         *outs, None, None, 0, None)

    def bwd(flags, ups=(P[3], None, None, None, None), grads=(P[7], P[8], P[9])):
        return lib.tcelbo_decomp_backward(P[0], D, P[1], D, P[2], D, B, B, 0, D, N, flags, 2.0, *ups,
                                          grads[0], D, grads[1], D, grads[2], D, None, 0, None, 0, None)

    for st in (fwd(_lib.EST_MSS | _lib.SAVE_FOR_BACKWARD), bwd(_lib.EST_MWS | _lib.SAVE_FOR_BACKWARD)):
        assert st == _lib.ERR_INVALID
        assert b"TCELBO_VAR_COL" in lib.tcelbo_last_error()
    for outs in ((None, P[4], P[5], P[6]), (P[3], P[4], P[5], None)):
        assert fwd(col, outs=outs) == _lib.ERR_INVALID
        assert b"null output" in lib.tcelbo_last_error()
    assert fwd(col, inputs=(P[0], None, P[2])) == _lib.ERR_INVALID
    assert b"null input" in lib.tcelbo_last_error()
    assert bwd(col, grads=(P[7], None, P[9])) == _lib.ERR_INVALID
    assert b"null gradient" in lib.tcelbo_last_error()
    assert bwd(col, ups=(None, None, None, None, None)) == _lib.ERR_INVALID
    assert b"no upstream gradient" in lib.tcelbo_last_error()
    with pytest.raises(ValueError, match="TCELBO_VAR_COL"):
        _lib.check(fwd(_lib.EST_MSS), "tcelbo_decomp_forward")


def test_decomp_ops_are_public_and_refuse_cpu_tensors():
    import torch
    from intro_tc_vae_b200 import ops
    assert "tc_decomp_loss_terms" in ops.__all__ and "tc_decomp_loss_mean" in ops.__all__
    x = torch.zeros(4, 8)
    for fn in (ops.tc_decomp_loss_terms, ops.tc_decomp_loss_mean):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(x, x, x, 10, 2.0)


def test_decomp_workspace_holds_four_means_and_the_prior_coefficients():
    """The decomposition reuses the column-variance size queries; the backward scratch of a column-variance plan is larger than
    the row-variance one of the same shape by at least the extra [b_loc] array of log p(z) coefficients."""
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    for b, d in ((8, 4), (1000, 128), (8192, 128)):
        col = _lib.VAR_COL | _lib.SAVE_FOR_BACKWARD
        assert lib.tcelbo_workspace_bytes(b, b, d, col) > 0
        assert lib.tcelbo_backward_scratch_bytes(b, b, d, col) >= lib.tcelbo_backward_scratch_bytes(b, b, d, _lib.SAVE_FOR_BACKWARD) + 4 * b
