"""CPU-side checks: libtcelbo.so loads, exports every symbol include/tcelbo.h declares, the planner is
sane, and the Python ops refuse anything but fp32 CUDA tensors (no silent fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "tcelbo.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tcelbo_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    declared = _header_symbols()
    assert len(declared) >= 11
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/tcelbo.h but not exported by libtcelbo.so"
    assert set(declared) == set(_lib.EXPORTED_SYMBOLS)
    assert lib.tcelbo_version() == 3


def test_workspace_planner_without_gpu():
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    small = lib.tcelbo_workspace_bytes(64, 64, 128, 0)
    saved = lib.tcelbo_workspace_bytes(64, 64, 128, _lib.SAVE_FOR_BACKWARD)
    assert 0 < small < saved
    big = lib.tcelbo_workspace_bytes(8192, 8192, 128, _lib.SAVE_FOR_BACKWARD)
    assert 8192 * 8192 * 4 < big < 2 * 1024 ** 3          # joint matrix + partials, far below B*B*D*4 = 32 GiB
    shard = lib.tcelbo_workspace_bytes(4096, 32768, 512, _lib.SAVE_FOR_BACKWARD)   # BASELINE cfg 4 per rank
    assert shard < 8 * 1024 ** 3
    assert lib.tcelbo_workspace_bytes(64, 64, 513, 0) == 0  # d > 512 is outside the built kernels
    assert lib.tcelbo_workspace_bytes(0, 64, 16, 0) == 0


def test_argument_validation_returns_status_not_crash():
    from intro_tc_vae_b200 import _lib
    lib = _lib.load()
    st = lib.tcelbo_forward(None, 0, None, 0, None, 0, 4, 4, 0, 8, 10, 0, None, None, None, 0, None)
    assert st == _lib.ERR_INVALID
    assert b"null" in lib.tcelbo_last_error()
    with pytest.raises(ValueError):
        _lib.check(st, "tcelbo_forward")


def test_ops_reject_cpu_and_non_fp32_tensors():
    from intro_tc_vae_b200 import ops
    x = torch.zeros(4, 8)
    for fn in (lambda: ops.total_correlation(x, x, x, 10), lambda: ops.kl_divergence(x, x),
               lambda: ops.reparameterize(x, x), lambda: ops.row_log_density(x)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn()


def test_host_weight_matrix_matches_reference(golden):
    from intro_tc_vae_b200 import ops
    import numpy as np
    for b, n in ((2, 10), (3, 3), (5, 100), (8, 3)):
        with np.errstate(all="ignore"):
            np.testing.assert_array_equal(ops.log_importance_weight_matrix(b, n).numpy(), golden[f"logw/B{b}_N{n}"])
    with pytest.raises(ZeroDivisionError):
        ops.log_importance_weight_matrix(1, 10)


def test_kernel_formulation_model_matches_reference(golden):
    """The kernels' arithmetic (base-2 exponents, fixed shift, weight ratios, masked analytic gradients),
    modelled in numpy fp32, against the reference's fp64 outputs."""
    import numpy as np
    from cases import CASES, make_inputs
    from oracle import kernel_model as K

    def rel(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)

    for name in ("base_B64_D128", "stress_B64_D128", "ragged_B37_D20", "pair_B2_D16", "tiny_B3_D128"):
        case = CASES[name]
        mu, lv, eps = (a.astype(np.float32) for a in make_inputs(case))
        z = (mu + eps * np.exp(np.float32(0.5) * lv)).astype(np.float32)
        B, N, beta = case["B"], case["N"], case["beta"]
        pre = f"{name}/f64/"
        fw = K.forward_rowvar(z, mu, lv, N, "mss")
        assert rel(fw["log_qz_prod"], golden[pre + "log_qz_prod"]) < 1e-5
        assert rel(fw["log_qz"], golden[pre + "log_qz"]) < 1e-5
        g = np.full(B, (beta - 1) / B, np.float32)
        gz, gmu, glv = K.backward_rowvar(fw, g, -g)
        std = np.exp(0.5 * lv)
        assert rel(gz, golden[pre + "simple_mean_dz_partial"]) < 1e-4
        assert rel(gmu + gz + mu / B, golden[pre + "simple_mean_dmu"]) < 1e-4
        assert rel(glv + gz * eps * std * 0.5 - 0.5 * (1 - np.exp(lv)) / B, golden[pre + "simple_mean_dlv"]) < 1e-4
        gz2, gmu2, glv2 = K.backward_rowvar_sweep(fw, g, -g)            # the sweep's shifted-exponent arithmetic
        assert rel(gz2, golden[pre + "simple_mean_dz_partial"]) < 1e-4
        assert rel(gmu2 + gz2 + mu / B, golden[pre + "simple_mean_dmu"]) < 1e-4
        assert rel(glv2 + gz2 * eps * std * 0.5 - 0.5 * (1 - np.exp(lv)) / B, golden[pre + "simple_mean_dlv"]) < 1e-4
        fj = K.forward_colvar(z, mu, lv, N, "mss")
        assert rel(fj["log_qz_prod"], golden[pre + "varj_log_qz_prod"]) < 1e-5
        assert rel(fj["log_qz"], golden[pre + "varj_log_qz"]) < 1e-5
