"""CPU tests of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports
exactly the symbols include/spev_b200.h declares, its host helpers agree with the oracle, and
the product path fails loudly (never falls back) without a GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "spev_b200.h")).read()
    return sorted(set(re.findall(r"SPEV_API\s+[\w\s\*]+?\b(spev_\w+)\s*\(", src)))


def test_library_builds_exports_header_symbols_abi_3():
    import spev_tts_b200 as sp
    from spev_tts_b200 import build
    build.build()
    lib = sp.load()
    syms = header_symbols()
    assert len(syms) >= 24
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in spev_b200.h but not exported"
    assert sorted(sp.EXPORTED_SYMBOLS) == syms, "ctypes table and header disagree"
    out = subprocess.check_output(["nm", "-D", "--defined-only", sp.LIB_PATH], text=True)
    exported = sorted(l.split()[-1] for l in out.splitlines() if " T " in l)
    assert exported == syms, "library exports symbols outside the header (or misses some)"
    assert lib.spev_abi_version() == 3 and lib.spev_tile_chunks() == lib.spev_tile_frames() - 3


def test_sass_is_sm100a():
    import spev_tts_b200 as sp
    out = subprocess.check_output(["cuobjdump", "-lelf", sp.LIB_PATH], text=True)
    assert "sm_100a" in out


def test_host_constants_match_oracle():
    import spev_tts_b200 as sp
    lib = sp.load()
    for sr, fmin, fmax in ((22050, 0.0, 0.0), (22050, 0.0, 8000.0), (24000, 0.0, 0.0)):
        b = np.empty((80, 513), np.float32)
        assert lib.spev_host_mel_basis(sr, 1024, 80, fmin, fmax, b.ctypes.data) == 0
        ob = lr.mel_filter(sr=sr, n_fft=1024, n_mels=80, fmin=fmin, fmax=fmax or None)
        assert np.array_equal(b, ob)
        p = np.empty((513, 80), np.float32)
        assert lib.spev_host_pinv(ob.ctypes.data, 80, 513, p.ctypes.data) == 0
        op = np.linalg.pinv(ob)
        assert np.linalg.norm(p - op) / np.linalg.norm(op) < 1e-6


def test_plan_tiles_count_query_and_closed_forms():
    """spev_plan_frame_tiles / spev_plan_chunk_tiles: the count query (out == NULL) equals the number of tiles the fill
    writes, for waveform and ISTFT-output frame tiles and for default and explicit output lengths, and the counts are
    sum ceil(T/32), sum ceil((T-1)/29) and sum ceil(ceil(L/256)/29)."""
    import spev_tts_b200 as sp
    from spev_tts_b200 import batch as B
    lib = sp.load()
    tf, tc = lib.spev_tile_frames(), lib.spev_tile_chunks()
    rng = np.random.default_rng(0)
    ns = rng.integers(0, 200 * 256, 50).astype(np.int64)
    ns[:4] = [0, 255, 256, 32 * 256]
    frames = 1 + ns // 256
    starts = B.aligned_offsets(ns)[:-1]
    out_len = rng.integers(0, 260 * 200, 50).astype(np.int64)
    out_len[:4] = [0, 1, 256, 29 * 256 + 1]
    out_off = B.out_layout(frames, out_len)[0]
    def_off, def_len = B.out_layout(frames)

    def count_and_fill(fn, a, b):
        cnt = fn(frames.ctypes.data, a.ctypes.data, b.ctypes.data, len(frames), None)
        out = np.zeros(cnt + 1, dtype=B.TILE_DTYPE)           # one spare record, which the fill must not touch
        assert fn(frames.ctypes.data, a.ctypes.data, b.ctypes.data, len(frames), out.ctypes.data) == cnt
        assert out[cnt:].tobytes() == bytes(B.TILE_DTYPE.itemsize)
        return cnt
    for lo, n in ((starts, ns), (def_off, def_len)):
        assert count_and_fill(lib.spev_plan_frame_tiles, lo, n) == int(((frames + tf - 1) // tf).sum())
    assert count_and_fill(lib.spev_plan_chunk_tiles, def_off, def_len) == int(((frames - 1 + tc - 1) // tc).sum())
    nc = (out_len + 255) // 256
    assert count_and_fill(lib.spev_plan_chunk_tiles, out_off, out_len) == int(((nc + tc - 1) // tc).sum())
    # every frame / chunk covered exactly once
    assert B.plan_frame_tiles(frames, def_off, def_len)["n"].sum() == frames.sum()
    assert B.plan_chunk_tiles(frames, out_off=def_off, out_len=def_len)["n"].sum() == (frames - 1).sum()
    assert B.plan_chunk_tiles(frames, out_off=out_off, out_len=out_len)["n"].sum() == nc.sum()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu():
    import spev_tts_b200 as sp
    lib = sp.load()
    h = C.c_void_p()
    rc = lib.spev_create(C.byref(h), 0, 22050, 1024, 256, 1024, 80, 0.0, 0.0)
    assert rc == -3 and b"no CPU fallback" in lib.spev_last_error()
    with pytest.raises(RuntimeError):
        sp.logmel(np.zeros(4096, np.float32))
    with pytest.raises(RuntimeError):
        sp.LengthRegulator()(torch.zeros(1, 2, 3), torch.ones(1, 2, dtype=torch.int64))
    with pytest.raises(RuntimeError):
        sp.Vocoder().infer(np.zeros((80, 10), np.float32))
    with pytest.raises(RuntimeError):
        sp.bucketize(torch.zeros(3), torch.zeros(2))


def test_unsupported_config_is_an_error():
    import spev_tts_b200 as sp
    lib = sp.load()
    h = C.c_void_p()
    assert lib.spev_create(C.byref(h), 0, 22050, 2048, 512, 2048, 80, 0.0, 0.0) == -2
    assert b"n_fft=1024" in lib.spev_last_error()


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under spev_tts_b200/ may reference it."""
    pkg = os.path.join(ROOT, "spev_tts_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "librosa_restated" not in src, f


def test_host_fft_building_blocks():
    exe = os.path.join(ROOT, "tests", "host", "fft_check")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I/usr/local/cuda/include",
                           "-I" + os.path.join(ROOT, "spev_tts_b200", "csrc"),
                           os.path.join(ROOT, "tests", "host", "fft_check.cpp"), "-o", exe])
    assert subprocess.call([exe]) == 0


def test_header_is_valid_c99_and_struct_layout():
    """include/spev_b200.h compiles as strict C99 and spev_tile is 48 bytes (what the kernels assume)."""
    obj = os.path.join(ROOT, "tests", "host", "abi_c99.o")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           "-c", os.path.join(ROOT, "tests", "host", "abi_c99.c"), "-o", obj])
    from spev_tts_b200 import _lib, batch
    assert C.sizeof(_lib.SpevTile) == 48 == batch.TILE_DTYPE.itemsize
    assert C.sizeof(_lib.SpevBatch) == 48
    # every header symbol is referenced by the C probe
    src = open(os.path.join(ROOT, "tests", "host", "abi_c99.c")).read()
    for sym in header_symbols():
        assert f"USE({sym})" in src, sym


def test_host_entry_points_and_planners_reject_bad_arguments():
    import spev_tts_b200 as sp
    lib = sp.load()
    assert lib.spev_plan_frame_tiles(None, None, None, 3, None) == -1
    assert lib.spev_plan_chunk_tiles(None, None, None, 3, None) == -1
    frames, off, lens = (np.array(v, dtype=np.int64) for v in ([3, 3], [0, 1024], [512, -1]))
    assert lib.spev_plan_chunk_tiles(frames.ctypes.data, off.ctypes.data, None, 2, None) == -1    # out_off, no out_len
    assert b"out_len is null" in lib.spev_last_error()
    assert lib.spev_plan_chunk_tiles(frames.ctypes.data, None, None, 2, None) == -1
    assert lib.spev_plan_chunk_tiles(frames.ctypes.data, off.ctypes.data, lens.ctypes.data, 2, None) == -1
    assert b"out_len[1]" in lib.spev_last_error()
    assert lib.spev_plan_frame_tiles(frames.ctypes.data, None, lens.ctypes.data, 2, None) == -1   # no sample_lo
    assert b"sample_lo or n_samples is null" in lib.spev_last_error()
    assert lib.spev_plan_frame_tiles(frames.ctypes.data, off.ctypes.data, lens.ctypes.data, 2, None) == -1
    assert b"n_samples[1]" in lib.spev_last_error()
    from spev_tts_b200 import batch as B
    with pytest.raises(ValueError, match="out_len"):
        B.plan_chunk_tiles(frames, out_off=off, out_len=lens)
    with pytest.raises(ValueError, match="n_samples"):
        B.plan_frame_tiles(frames, off, lens)
    assert lib.spev_host_mel_basis(0, 1024, 80, 0.0, 0.0, None) == -1
    assert lib.spev_griffinlim_workspace_bytes(-5) == 0
    assert lib.spev_griffinlim_workspace_bytes(10) >= 10 * 520 * 16
    h = C.c_void_p()
    assert lib.spev_create(C.byref(h), 0, 22050, 1024, 256, 1024, 0, 0.0, 0.0) in (-1, -3)      # n_mels = 0
    assert lib.spev_create(None, 0, 22050, 1024, 256, 1024, 80, 0.0, 0.0) == -1
    assert lib.spev_logmel(None, None, None, None, 1, 1e-5, -10.0, 2.0, None) == -1             # null ctx
    assert b"ctx is null" in lib.spev_last_error()


# One bad call per entry point, each rejected before any CUDA call (so no device is needed): (name, args, rc, message).
# Dummy non-null pointers (16) stand in for buffers the check never reaches.
_P = 16
_NULL_CTX = [
    ("spev_logmel", (None, None, None, None, 0, 0.0, 0.0, 0.0, None)),
    ("spev_stft_power", (None, None, None, None, None)),
    ("spev_mel_project", (None, None, 1, None, 0, 0.0, 0.0, 0.0, None)),
    ("spev_mel_to_mag", (None, None, None, 0, 0, None, 520, None)),
    ("spev_nnls_objective", (None, None, 0, 0, None, 0, 1, 1, 0, 1, 0, None, None, None, None)),
    ("spev_istft", (None, None, None, 520, None, None)),
    ("spev_stft", (None, None, None, None, 520, None)),
    ("spev_gl_phase_update", (None, None, None, None, 520, None, None, 520, 0.5, 0, None)),
    ("spev_griffinlim", (None, None, None, 520, None, 0, 1, 0.99, None, None, 0, None)),
    ("spev_frame_features", (None, None, None, None, None, None)),
    ("spev_set_sm_limit", (None, 0)),
    ("spev_set_tensor_core", (None, 1)),
]
_BAD_CALLS = [(name, args, -1, b"ctx is null") for name, args in _NULL_CTX] + [
    ("spev_transpose_batched", (_P, _P, 4, 1, -1, 4, 4, 16, 4, 16, None), -1, b"transpose: negative shape"),
    ("spev_transpose_batched", (_P, _P, 3, 1, 4, 4, 4, 16, 4, 16, None), -2, b"4- or 8-byte elements only"),
    ("spev_collate", (_P, 13, _P, _P, None, 2, 4, 4, None), -1, b"at most 12 arrays"),
    ("spev_copy_segments", (_P, _P, _P, _P, _P, _P, -1, 1, None), -1, b"copy_segments: negative sizes"),
    ("spev_segment_pool", (_P, _P, _P, _P, 2, 0.0, 0.0, -3.0, 3.0, _P, None), -1, b"segment_pool: sigma == 0"),
    ("spev_segment_pool_log", (_P, 1e-5, _P, _P, _P, 2, 0.0, 0.0, -3.0, 3.0, _P, None), -1,
     b"segment_pool: sigma == 0"),
    ("spev_lr_plan", (_P, 0, -1, 4, _P, _P, _P, None, None), -1, b"lr_plan: negative shape"),
    ("spev_lr_expand", (None, 16, _P, 2, 4, _P, 8, None), -1, b"spev_lr_expand: null x/out"),
    ("spev_lr_expand_fused", (_P, 16, _P, 17, None, None, _P, 2, 4, _P, _P, 8, None), -1, b"lr_expand: bad shape"),
    ("spev_pcm16_to_f32", (_P, -1, _P, None), -1, b"pcm16_to_f32: n < 0"),
    ("spev_variance_fuse", (_P, _P, 1, None, None, _P, _P, _P, 2, 4, 0, _P, _P, 8, None), -1,
     b"variance_fuse: bad shape"),
    ("spev_lr_expand_backward", (_P, 0, 4, None, 0, None, None, None, _P, -1, 4, 8, _P, None, None), -1,
     b"lr_expand_backward: bad shape"),
    ("spev_variance_fuse_backward", (_P, _P, 6, None, None, _P, _P, 2, 4, 8, 8, _P, _P, _P, _P, _P, 1 << 20, None),
     -2, b"at most 5 curves"),
    ("spev_duration_rule", (_P, -1, 1.0, _P, None), -1, b"duration_rule: n < 0"),
    ("spev_bucketize_embed", (_P, 8, _P, 12001, 0, None, 0, _P, None, 0, None), -1, b"n_boundaries <= 12000"),
]


@pytest.mark.parametrize("name,args,rc,msg", _BAD_CALLS, ids=[f"{c[0]}-{i}" for i, c in enumerate(_BAD_CALLS)])
def test_entry_points_reject_bad_arguments_before_any_cuda_call(name, args, rc, msg):
    import spev_tts_b200 as sp
    lib = sp.load()
    assert getattr(lib, name)(*args) == rc
    assert msg in lib.spev_last_error()


def test_workspace_queries_and_piece_size():
    import spev_tts_b200 as sp
    lib = sp.load()
    assert lib.spev_griffinlim_workspace_bytes(-1) == 0
    for bad in ((-1, 2, 8, 8), (1, -1, 8, 8), (1, 2, -1, 8), (1, 2, 8, -1)):
        assert lib.spev_variance_fuse_backward_workspace_bytes(*bad) == 0
    assert lib.spev_variance_fuse_backward_workspace_bytes(1, 2, 8, 8) > 0
    assert lib.spev_copy_segments_piece_bytes() == 16384
