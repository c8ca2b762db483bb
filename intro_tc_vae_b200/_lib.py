"""ctypes binding of libtcelbo.so (C ABI declared in include/tcelbo.h).

There is deliberately no fallback: if the shared library is missing or cannot be loaded, every op
of this package raises.  Build it with ``python -m intro_tc_vae_b200.build``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint32, c_void_p, POINTER

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libtcelbo.so")

# flags (include/tcelbo.h)
EST_MSS = 0
EST_MWS = 1
VAR_ROW = 0
VAR_COL = 2
SAVE_FOR_BACKWARD = 4
PEER_SWEEP, PEER_FINISH = 1, 2

ERR_INVALID, ERR_CUDA, ERR_WORKSPACE, ERR_UNSUPPORTED = 1, 2, 3, 4

_f = c_void_p          # device pointers are passed as integers (tensor.data_ptr())


class PeerSyncArgs(ctypes.Structure):
    """``tcelbo_peer_sync`` of include/tcelbo.h: in-kernel cross-rank barriers of the peer-memory exchange."""
    _fields_ = [("flag_parts", c_void_p), ("state", c_void_p)]


class Fusion(ctypes.Structure):
    """``tcelbo_fusion`` of include/tcelbo.h: optional prologue / epilogue fusions of the fused loss (None = off)."""
    _fields_ = [("eps", c_void_p), ("ldeps", c_int64), ("z_out", c_void_p), ("ldz_out", c_int64),
                ("loss_mean", c_void_p), ("kl_mean", c_void_p),
                ("rec_rows", c_void_p), ("scale", c_float), ("expelbo", c_void_p), ("e_rows", c_void_p),
                ("g_loss_mean", c_void_p), ("g_kl_mean", c_void_p), ("g_expelbo", c_void_p), ("g_rec_rows", c_void_p)]


_SIGNATURES = {
    "tcelbo_version": (c_int, []),
    "tcelbo_last_error": (c_char_p, []),
    "tcelbo_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_uint32]),
    "tcelbo_backward_scratch_bytes": (c_size_t, [c_int, c_int, c_int, c_uint32]),
    "tcelbo_forward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32,
                               _f, _f, c_void_p, c_size_t, c_void_p]),
    "tcelbo_backward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32,
                                _f, _f, _f, c_int64, _f, c_int64, _f, c_int64, c_void_p, c_size_t, c_void_p, c_size_t,
                                c_void_p]),
    "tcelbo_klloss_forward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32, c_float,
                                      _f, _f, _f, _f, c_void_p, c_size_t, c_void_p]),
    "tcelbo_klloss_backward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32, c_float,
                                       _f, _f, _f, _f, _f, c_int64, _f, c_int64, _f, c_int64, c_void_p, c_size_t, c_void_p, c_size_t,
                                       c_void_p]),
    "tcelbo_klloss_forward_ex": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32, c_float,
                                         _f, _f, _f, _f, POINTER(Fusion), c_void_p, c_size_t, c_void_p]),
    "tcelbo_klloss_backward_ex": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32, c_float,
                                          _f, _f, _f, _f, POINTER(Fusion), _f, c_int64, _f, c_int64, _f, c_int64, c_void_p, c_size_t,
                                          c_void_p, c_size_t, c_void_p]),
    "tcelbo_peer_publish": (c_int, [_f, c_int64, c_int, c_int, _f, POINTER(PeerSyncArgs), c_void_p]),
    "tcelbo_klloss_forward_peer": (c_int, [_f, c_int64, _f, c_int64, c_void_p, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64,
                                           c_uint32, c_float, _f, _f, _f, _f, POINTER(Fusion), POINTER(PeerSyncArgs), c_void_p, c_size_t, c_void_p]),
    "tcelbo_klloss_backward_peer": (c_int, [c_int, _f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, c_int, c_int, c_int64, c_uint32,
                                            c_float, _f, _f, _f, _f, _f, c_int64, _f, c_int64, _f, c_int64, c_void_p, c_size_t,
                                            c_void_p, c_size_t, c_void_p, POINTER(Fusion), POINTER(PeerSyncArgs), c_void_p]),
    "tcelbo_kl_forward": (c_int, [_f, c_int64, _f, c_int64, c_int, c_int, _f, c_void_p]),
    "tcelbo_kl_backward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int, c_int, _f, c_int64, _f, c_int64, c_void_p]),
    "tcelbo_reparam_forward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, _f, c_int64, c_void_p]),
    "tcelbo_reparam_backward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, _f, c_int64, _f, c_int64,
                                        c_void_p]),
    "tcelbo_reparam_backward_acc": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, _f, c_int64, _f, c_int64,
                                        c_void_p]),
    "tcelbo_rowdensity_forward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, c_int, c_int, _f, c_void_p]),
    "tcelbo_rowdensity_backward": (c_int, [_f, c_int64, _f, c_int64, _f, c_int64, _f, c_int, c_int,
                                           _f, c_int64, _f, c_int64, _f, c_int64, c_void_p]),
    "tcelbo_recloss_chunks": (c_int, [c_int, c_int64]),
    "tcelbo_recloss_forward": (c_int, [_f, _f, c_int, c_int64, c_int, _f, _f, c_void_p]),
    "tcelbo_recloss_backward": (c_int, [_f, _f, _f, c_int, c_int64, c_int, _f, c_void_p]),
    "tcelbo_expelbo_forward": (c_int, [_f, _f, c_int, c_float, _f, _f, c_void_p]),
    "tcelbo_expelbo_backward": (c_int, [_f, _f, c_int, c_float, _f, c_void_p]),
    "tcelbo_density_forward": (c_int, [c_int, _f, _f, _f, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64),
                                       _f, c_void_p]),
    "tcelbo_density_backward": (c_int, [c_int, _f, _f, _f, _f, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64),
                                        POINTER(c_int64), _f, _f, _f, c_void_p]),
    "tcelbo_sampling_forward": (c_int, [_f, c_int, c_int, c_int64, c_uint32, _f, _f, _f, _f, c_void_p]),
    "tcelbo_sampling_backward": (c_int, [_f, c_int, c_int, c_int64, c_uint32, _f, _f, _f, _f, _f, _f, c_void_p]),
    "tcelbo_launch_count": (ctypes.c_longlong, []),
    "tcelbo_profile_events": (c_int, [c_int, c_void_p, c_void_p]),
    "tcelbo_ex2_peak": (c_int, [_f, c_int, c_int, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class TcelboError(RuntimeError):
    """A libtcelbo.so entry point returned a non-zero status."""


def load() -> ctypes.CDLL:
    """Load libtcelbo.so once; raises if it is absent (no CPU / eager fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m intro_tc_vae_b200.build` "
            "(the TC-ELBO ops have no fallback implementation)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here means the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status == 0:
        return
    msg = load().tcelbo_last_error()
    msg = msg.decode() if msg else ""
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(f"{what}: {msg}")
    if status in (ERR_INVALID, ERR_WORKSPACE):
        raise ValueError(f"{what}: {msg}")
    raise TcelboError(f"{what} failed with status {status}: {msg}")
