"""CPU checks of the peer-memory form of the MI / TC / dimension-wise KL decomposition (tcelbo_decomp_forward_peer /
_backward_peer, tcelbo_peer_publish_mu_logvar) and of the solver's guard around the exchange.

Every malformed call must come back as TCELBO_ERR_INVALID before the library touches a device, so these run without a GPU.
"""
import ctypes

import numpy as np
import pytest

B_LOC, D, N, RANKS = 4, 8, 100, 2
COL = 0 | 2 | 4                     # TCELBO_EST_MSS | TCELBO_VAR_COL | TCELBO_SAVE_FOR_BACKWARD


@pytest.fixture(scope="module")
def lib():
    from intro_tc_vae_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def ptrs():
    hold = [np.zeros(64, np.float32) for _ in range(16)]
    return hold, [h.ctypes.data for h in hold]


def _fwd(lib, P, flags=COL, z=-1, tables=None, ld_part=D, n_ranks=RANKS, rank=0, sync=None):
    z = P[0] if z == -1 else z
    mu_t, lv_t = (P[10], P[11]) if tables is None else tables
    return lib.tcelbo_decomp_forward_peer(z, D, P[1], D, P[2], D, mu_t, lv_t, ld_part, B_LOC, n_ranks, rank, D, N, flags, 2.0,
                                          P[3], P[4], P[5], P[6], None, sync, None, 0, None)


def _bwd(lib, P, phase=1, flags=COL, n_ranks=RANKS, rank=0, table=-1, ups=None, grads=None, sync=None):
    table = P[12] if table == -1 else table
    ups = (P[3], None, None, None, None) if ups is None else ups
    grads = (P[7], P[8], P[9]) if grads is None else grads
    return lib.tcelbo_decomp_backward_peer(phase, P[0], D, P[1], D, P[2], D, B_LOC, n_ranks, rank, D, N, flags, 2.0, *ups,
                                           grads[0], D, grads[1], D, grads[2], D, None, 0, None, 0, table, sync, None)


def _expect_invalid(lib, st, text):
    from intro_tc_vae_b200 import _lib
    assert st == _lib.ERR_INVALID
    assert text.encode() in lib.tcelbo_last_error()


def test_decomp_forward_peer_refuses_invalid_calls(lib, ptrs):
    from intro_tc_vae_b200 import _lib
    _, P = ptrs
    _expect_invalid(lib, _fwd(lib, P, flags=_lib.EST_MSS | _lib.SAVE_FOR_BACKWARD), "TCELBO_VAR_COL")
    _expect_invalid(lib, _fwd(lib, P, z=None), "null input")
    _expect_invalid(lib, _fwd(lib, P, tables=(None, P[11])), "null pointer table")
    _expect_invalid(lib, _fwd(lib, P, tables=(P[10], None)), "null pointer table")
    for kw in (dict(rank=RANKS), dict(rank=-1), dict(n_ranks=0), dict(ld_part=D - 1)):
        _expect_invalid(lib, _fwd(lib, P, **kw), "bad rank / n_ranks / ld_part")
    no_flags = _lib.PeerSyncArgs(flag_parts=None, state=P[13])
    _expect_invalid(lib, _fwd(lib, P, sync=ctypes.byref(no_flags)), "peer_sync")


def test_decomp_backward_peer_refuses_invalid_calls(lib, ptrs):
    from intro_tc_vae_b200 import _lib
    _, P = ptrs
    _expect_invalid(lib, _bwd(lib, P, flags=_lib.EST_MWS | _lib.SAVE_FOR_BACKWARD), "TCELBO_VAR_COL")
    for phase in (0, 3):
        _expect_invalid(lib, _bwd(lib, P, phase=phase), "phase")
    _expect_invalid(lib, _bwd(lib, P, phase=_lib.PEER_FINISH, table=None), "null scratch table")
    for kw in (dict(rank=RANKS), dict(rank=-1), dict(n_ranks=0)):
        _expect_invalid(lib, _bwd(lib, P, **kw), "bad rank / n_ranks")
    _expect_invalid(lib, _bwd(lib, P, grads=(P[7], None, P[9])), "null gradient")
    _expect_invalid(lib, _bwd(lib, P, ups=(None,) * 5), "no upstream gradient")
    no_state = _lib.PeerSyncArgs(flag_parts=P[13], state=None)
    _expect_invalid(lib, _bwd(lib, P, sync=ctypes.byref(no_state)), "peer_sync")


def test_publish_mu_logvar_refuses_invalid_calls(lib, ptrs):
    from intro_tc_vae_b200 import _lib
    _, P = ptrs

    def pub(mu=P[1], lv=P[2], ldlv=D, b_loc=B_LOC, dst=(P[10], P[11]), sync=None):
        return lib.tcelbo_peer_publish_mu_logvar(mu, D, lv, ldlv, b_loc, D, dst[0], dst[1], sync, None)

    _expect_invalid(lib, pub(lv=None), "null pointer")
    _expect_invalid(lib, pub(dst=(P[10], None)), "null pointer")
    _expect_invalid(lib, pub(ldlv=D - 1), "row pitch")
    _expect_invalid(lib, pub(b_loc=0), "b_loc")
    no_state = _lib.PeerSyncArgs(flag_parts=P[13], state=None)
    _expect_invalid(lib, pub(sync=ctypes.byref(no_state)), "peer_sync")


def test_klloss_peer_entry_points_still_refuse_column_variance(lib, ptrs):
    """The simple loss's peer entry points keep to the row-variance density; the refusal names the decomposition's own."""
    from intro_tc_vae_b200 import _lib
    _, P = ptrs
    st = lib.tcelbo_klloss_forward_peer(P[0], D, P[1], D, P[10], D, P[2], D, B_LOC, RANKS, 0, D, N, COL, 2.0,
                                        P[3], P[4], P[5], P[6], None, None, None, 0, None)
    assert st == _lib.ERR_UNSUPPORTED
    assert b"tcelbo_decomp_forward_peer" in lib.tcelbo_last_error()


class _StubExchange:
    b_loc, d = 16, 8


class _Solver:
    beta_kl = 2.0
    dataset = range(1000)
    process_group = None
    peer_exchange = _StubExchange()

    def write_scalar(self, *args):
        pass


@pytest.mark.parametrize("method", ["_compute_kl_loss_full", "_compute_kl_loss_simple"])
@pytest.mark.parametrize("reduce", ["mean", "none"])
def test_solver_refuses_a_mismatched_exchange_without_process_group(method, reduce):
    """A batch that does not match the exchange's shard shape, with no process group to fall back on, must raise instead of
    running the estimator over the local rows as if they were the whole batch.  The guard runs before any device work."""
    import torch
    from intro_tc_vae_b200.solvers.tc import TCLossMixin
    z = torch.zeros(12, 8)
    with pytest.raises(RuntimeError, match="silently run unsharded"):
        getattr(TCLossMixin, method)(_Solver(), z, z, z, reduce)
