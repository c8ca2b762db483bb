"""CPU checks of the fused decomposition entry points (tcelbo_decomp_forward_ex / _backward_ex and the peer pair
tcelbo_decomp_forward_peer_ex / _backward_peer_ex) and of the loss selectors of GraphedKLLoss and SoftIntroTCStep.

Every malformed call must come back as TCELBO_ERR_INVALID before the library touches a device, so these run without a GPU.
"""
import ctypes

import numpy as np
import pytest

B, D, N = 4, 8, 100
COL = 0 | 2 | 4                     # TCELBO_EST_MSS | TCELBO_VAR_COL | TCELBO_SAVE_FOR_BACKWARD
ROW = 0 | 4


@pytest.fixture(scope="module")
def lib():
    from intro_tc_vae_b200 import _lib
    return _lib.load()


_HOLD = [np.zeros(64, np.float32) for _ in range(20)]       # host buffers standing in for device pointers (never dereferenced)


@pytest.fixture(scope="module")
def P():
    return [h.ctypes.data for h in _HOLD]


def _fusion(P, **kw):
    from intro_tc_vae_b200 import _lib
    return _lib.Fusion(**{k: (P[v] if isinstance(v, int) and k not in ("ldeps", "ldz_out") else v) for k, v in kw.items()})


# which fusion members each direction accepts, by slot in P
FWD_OK = dict(eps=14, ldeps=D, z_out=15, ldz_out=D, rec_rows=16, expelbo=17, e_rows=18)
BWD_OK = dict(eps=14, ldeps=D, e_rows=18, g_expelbo=17, g_rec_rows=19)


def _fwd(lib, P, peer, fz=None, flags=COL, z=-1, outs=None):
    z = P[0] if z == -1 else z
    outs = (P[3], P[4], P[5], P[6]) if outs is None else outs
    f = ctypes.byref(fz) if fz is not None else None
    if peer:
        return lib.tcelbo_decomp_forward_peer_ex(z, D, P[1], D, P[2], D, P[10], P[11], D, B, 2, 0, D, N, flags, 2.0,
                                                 *outs, None, f, None, None, 0, None)
    return lib.tcelbo_decomp_forward_ex(z, D, P[1], D, P[2], D, B, B, 0, D, N, flags, 2.0, *outs, None, f, None, 0, None)


def _bwd(lib, P, peer, fz=None, flags=COL, z=-1, ups=None, grads=None):
    z = P[0] if z == -1 else z
    ups = (P[3], None, None, None, None) if ups is None else ups
    grads = (P[7], P[8], P[9]) if grads is None else grads
    f = ctypes.byref(fz) if fz is not None else None
    if peer:
        return lib.tcelbo_decomp_backward_peer_ex(1, z, D, P[1], D, P[2], D, B, 2, 0, D, N, flags, 2.0, *ups,
                                                  grads[0], D, grads[1], D, grads[2], D, None, 0, None, 0, P[12], f, None, None)
    return lib.tcelbo_decomp_backward_ex(z, D, P[1], D, P[2], D, B, B, 0, D, N, flags, 2.0, *ups, f,
                                         grads[0], D, grads[1], D, grads[2], D, None, 0, None, 0, None)


def _expect(lib, st, code, text):
    assert st == code, (st, lib.tcelbo_last_error())
    assert text.encode() in lib.tcelbo_last_error(), lib.tcelbo_last_error()


@pytest.mark.parametrize("peer", [False, True])
def test_decomp_forward_ex_refuses_invalid_calls(lib, P, peer):
    from intro_tc_vae_b200 import _lib
    bad = lambda st, text: _expect(lib, st, _lib.ERR_INVALID, text)          # noqa: E731
    bad(_fwd(lib, P, peer, flags=ROW), "TCELBO_VAR_COL")
    bad(_fwd(lib, P, peer, z=None), "null input")                            # no eps: z is read
    bad(_fwd(lib, P, peer, outs=(P[3], None, P[5], P[6])), "null output")
    for member in ("loss_mean", "kl_mean", "g_loss_mean", "g_kl_mean"):
        bad(_fwd(lib, P, peer, _fusion(P, **{member: 17})), "`means` / `g_means`")
    bad(_fwd(lib, P, peer, _fusion(P, eps=14, ldeps=D - 1), z=None), "row pitch")
    bad(_fwd(lib, P, peer, _fusion(P, eps=14, ldeps=D, z_out=15, ldz_out=D - 1), z=None), "row pitch")
    bad(_fwd(lib, P, peer, _fusion(P, rec_rows=16, expelbo=17)), "expelbo needs rec_rows and e_rows")
    bad(_fwd(lib, P, peer, _fusion(P, e_rows=18, expelbo=17)), "expelbo needs rec_rows and e_rows")
    # a well-formed call with every accepted member gets past validation and stops at the missing workspace
    _expect(lib, _fwd(lib, P, peer, _fusion(P, **FWD_OK), z=None), _lib.ERR_WORKSPACE, "workspace")


@pytest.mark.parametrize("peer", [False, True])
def test_decomp_backward_ex_refuses_invalid_calls(lib, P, peer):
    from intro_tc_vae_b200 import _lib
    bad = lambda st, text: _expect(lib, st, _lib.ERR_INVALID, text)          # noqa: E731
    bad(_bwd(lib, P, peer, flags=_lib.EST_MWS | _lib.SAVE_FOR_BACKWARD), "TCELBO_VAR_COL")
    bad(_bwd(lib, P, peer, z=None), "null input")
    bad(_bwd(lib, P, peer, grads=(P[7], None, P[9])), "null gradient")
    bad(_bwd(lib, P, peer, ups=(None,) * 5), "no upstream gradient")
    for member in ("loss_mean", "kl_mean", "g_loss_mean", "g_kl_mean"):
        bad(_bwd(lib, P, peer, _fusion(P, **{member: 17})), "`means` / `g_means`")
    bad(_bwd(lib, P, peer, _fusion(P, eps=14, ldeps=D - 1), z=None), "row pitch")
    bad(_bwd(lib, P, peer, _fusion(P, g_expelbo=17)), "g_expelbo needs the e_rows")
    bad(_bwd(lib, P, peer, flags=COL & ~_lib.SAVE_FOR_BACKWARD), "TCELBO_SAVE_FOR_BACKWARD")
    # g_expelbo alone is an upstream gradient; with eps z may be NULL
    _expect(lib, _bwd(lib, P, peer, _fusion(P, **BWD_OK), z=None, ups=(None,) * 5), _lib.ERR_WORKSPACE, "workspace")


def test_klloss_keeps_refusing_the_fused_reparameterize_on_column_variance(lib, P):
    from intro_tc_vae_b200 import _lib
    fz = _fusion(P, eps=14, ldeps=D)
    st = lib.tcelbo_klloss_forward_ex(None, D, P[1], D, P[2], D, B, B, 0, D, N, COL, 2.0, P[3], P[4], P[5], P[6],
                                      ctypes.byref(fz), None, 0, None)
    _expect(lib, st, _lib.ERR_UNSUPPORTED, "the fused reparameterize covers the row-variance density")


def test_new_entry_points_are_exported():
    from intro_tc_vae_b200 import _lib
    for name in ("tcelbo_decomp_forward_ex", "tcelbo_decomp_backward_ex", "tcelbo_decomp_forward_peer_ex",
                 "tcelbo_decomp_backward_peer_ex"):
        assert name in _lib.EXPORTED_SYMBOLS


def test_graphed_loss_and_train_step_refuse_unknown_loss_forms():
    from intro_tc_vae_b200.graphs import GraphedKLLoss
    from intro_tc_vae_b200.train_step import SoftIntroTCStep
    with pytest.raises(ValueError, match="loss must be"):
        GraphedKLLoss(64, 8, N, 2.0, "cpu", loss="full")
    with pytest.raises(ValueError, match="kl_loss must be"):
        SoftIntroTCStep(None, None, None, N, (4, 3, 8, 8), kl_loss="decomp")
