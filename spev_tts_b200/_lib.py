"""ctypes binding of ``include/spev_b200.h`` (the C-ABI drop-in boundary).

There is no CPU fallback and no alternative backend: if ``libspev_b200.so`` is missing or the
device is not an sm_100 GPU, the calls below raise ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libspev_b200.so")

SPEV_OK = 0
SPEC_LD = 520
N_BINS = 513

c_f32p = C.POINTER(C.c_float)
c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)


class SpevTile(C.Structure):
    """``struct spev_tile`` (48 bytes)."""
    _fields_ = [("src0", C.c_int64), ("lo", C.c_int64), ("hi", C.c_int64), ("row0", C.c_int64),
                ("n", C.c_int32), ("t0", C.c_int32), ("T", C.c_int32), ("item", C.c_int32)]


class SpevPadArray(C.Structure):
    """``struct spev_pad_array``."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("row_bytes", C.c_int64),
                ("per_phone", C.c_int32), ("reserved", C.c_int32)]


class SpevBatch(C.Structure):
    """``struct spev_batch`` (include/spev_b200.h)."""
    _fields_ = [
        ("n_items", C.c_int32), ("n_ftiles", C.c_int32), ("n_ctiles", C.c_int32),
        ("reserved", C.c_int32), ("n_frames", C.c_int64),
        ("frame_off", C.c_void_p), ("ftiles", C.c_void_p), ("ctiles", C.c_void_p),
    ]


_SIGS = {
    "spev_abi_version": (C.c_int, []),
    "spev_last_error": (C.c_char_p, []),
    "spev_tile_frames": (C.c_int, []),
    "spev_tile_chunks": (C.c_int, []),
    "spev_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                              C.c_int, C.c_float, C.c_float]),
    "spev_destroy": (None, [C.c_void_p]),
    "spev_get_mel_basis": (C.c_int, [C.c_void_p, C.c_void_p]),
    "spev_get_mel_pinv": (C.c_int, [C.c_void_p, C.c_void_p]),
    "spev_get_window": (C.c_int, [C.c_void_p, C.c_void_p]),
    "spev_host_mel_basis": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]),
    "spev_host_pinv": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "spev_plan_frame_tiles": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "spev_plan_chunk_tiles": (C.c_int64, [C.c_void_p, C.c_int, C.c_void_p]),
    "spev_logmel": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p, C.c_int,
                              C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "spev_pcm16_to_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "spev_stft_power": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "spev_mel_project": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                   C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "spev_mel_to_mag": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_int, C.c_int,
                                  C.c_void_p, C.c_int64, C.c_void_p]),
    "spev_set_tensor_core": (C.c_int, [C.c_void_p, C.c_int]),
    "spev_nnls_objective": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int64,
                                      C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_istft": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_int64, C.c_void_p,
                             C.c_void_p]),
    "spev_stft": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p, C.c_int64,
                            C.c_void_p]),
    "spev_gl_phase_update": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                       C.c_int, C.c_void_p]),
    "spev_griffinlim_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "spev_griffinlim": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_uint64, C.c_int, C.c_float, C.c_void_p,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    "spev_frame_features": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_segment_pool": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float,
                                    C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "spev_segment_pool_log": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float,
                                        C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "spev_collate": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                               C.c_void_p]),
    "spev_transpose_batched": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                         C.c_int64, C.c_int64, C.c_void_p]),
    "spev_copy_segments_piece_bytes": (C.c_int, []),
    "spev_copy_segments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                     C.c_int64, C.c_void_p]),
    "spev_set_sm_limit": (C.c_int, [C.c_void_p, C.c_int]),
    "spev_lr_plan": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_lr_expand": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                 C.c_int64, C.c_void_p]),
    "spev_lr_expand_fused": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_int64, C.c_void_p]),
    "spev_variance_fuse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "spev_lr_expand_backward": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "spev_variance_fuse_backward_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int64]),
    "spev_variance_fuse_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "spev_duration_rule": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]),
    "spev_bucketize_embed": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                       C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_void_p]),
    "spev_pyin_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]),
    "spev_pyin_destroy": (None, [C.c_void_p]),
    "spev_pyin_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "spev_pyin_host_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_pyin_cmnd": (C.c_int, [C.c_void_p, C.POINTER(SpevBatch), C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_pyin_observe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "spev_pyin_decode_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64]),
    "spev_pyin_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "spev_pitch_pool": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double,
                                  C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGS))

_lib = None
_lock = threading.Lock()


def load() -> C.CDLL:
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: build it with `python -m spev_tts_b200.build` "
                    "(spev_tts_b200 has no CPU or PyTorch fallback)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGS.items():
                fn = getattr(lib, name)   # AttributeError if the symbol is not exported
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != SPEV_OK:
        msg = load().spev_last_error()
        raise RuntimeError(f"{what or 'spev'} failed (code {rc}): "
                           f"{msg.decode(errors='replace') if msg else ''}")
