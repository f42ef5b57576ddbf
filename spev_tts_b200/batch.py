"""Device context and flat (ragged) batch descriptors for the C ABI.

A *flat batch* concatenates items (utterances or spectrograms) and describes them with prefix
offsets + per-CTA tile tables (planned by the library's ``spev_plan_*_tiles``), all built on
the host and uploaded in ONE host->device copy.  Framing follows librosa ``center=True``: an
item of ``N`` samples has ``T = 1 + N // hop`` frames and an ISTFT output of ``(T-1)*hop`` samples
(reference call sites: ``spev_real_metrics.py:363`` and ``:730-733``).
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib

HOP = 256
N_FFT = 1024


TILE_DTYPE = np.dtype([("src0", "<i8"), ("lo", "<i8"), ("hi", "<i8"), ("row0", "<i8"),
                       ("n", "<i4"), ("t0", "<i4"), ("T", "<i4"), ("item", "<i4")])   # struct spev_tile
assert TILE_DTYPE.itemsize == 48


def _plan(fn, frames, a, b):
    """Count query, then fill, of a C tile planner ``fn(frames, a, b, n_items, out)``; ``a``, ``b``: per-item int64
    arrays."""
    frames = np.ascontiguousarray(frames, dtype=np.int64).reshape(-1)
    a, b = (np.ascontiguousarray(x, dtype=np.int64).reshape(-1) for x in (a, b))
    if a.shape != frames.shape or b.shape != frames.shape:
        raise ValueError(f"{fn.__name__}: needs one entry per item ({len(frames)}) in every array")
    args = [frames.ctypes.data, a.ctypes.data, b.ctypes.data, len(frames)]
    n = fn(*args, None)
    if n < 0:
        raise ValueError(_lib.load().spev_last_error().decode(errors="replace"))
    out = np.empty(n, dtype=TILE_DTYPE)
    fn(*args, out.ctypes.data)
    return out


def plan_frame_tiles(frames, sample_lo, n_samples) -> np.ndarray:
    """``spev_plan_frame_tiles``: one ``spev_tile`` per <=32-frame tile; item i's samples are ``n_samples[i]`` at
    ``sample_lo[i]``."""
    return _plan(_lib.load().spev_plan_frame_tiles, frames, sample_lo, n_samples)


def plan_chunk_tiles(frames, *, out_off, out_len) -> np.ndarray:
    """``spev_plan_chunk_tiles``: one ``spev_tile`` per <=29-chunk ISTFT tile, full tiles first.  Item i writes
    ``out_len[i]`` samples at ``out_off[i]``, ``ceil(out_len[i] / 256)`` chunks, with ``lo`` / ``hi`` set to those
    bounds (see ``include/spev_b200.h``)."""
    return _plan(_lib.load().spev_plan_chunk_tiles, frames, out_off, out_len)


def aligned_offsets(n_samples: Sequence[int], align: int = 4) -> np.ndarray:
    """Item starts ``[U+1]`` (last entry = buffer size) with every start a multiple of ``align``
    samples, so that the kernels take the 16-byte cp.async staging path.  The <= align-1 filler
    samples between items are never read as signal."""
    ns = np.asarray(n_samples, dtype=np.int64)
    padded = (ns + align - 1) // align * align
    return np.concatenate([[0], np.cumsum(padded)]).astype(np.int64)


def out_layout(frames, out_len=None, out_off=None):
    """ISTFT output layout of a spectrogram batch -> (``out_off`` int64 [n_items], ``out_len`` int64 [n_items]).
    ``out_len`` is one length per item (or one for all; librosa's ``length=``), by default ``256 * max(T - 1, 0)``.
    Default offsets pack the items in order, each starting at a multiple of 4 samples (``aligned_offsets``); given
    offsets must keep the items apart."""
    frames = np.asarray(frames, dtype=np.int64).reshape(-1)
    if out_len is None:
        out_len = np.maximum(frames - 1, 0) * HOP
    lens = np.broadcast_to(np.asarray(out_len, dtype=np.int64), frames.shape).copy()
    if (lens < 0).any():
        raise ValueError("output lengths must be >= 0")
    if out_off is None:
        off = aligned_offsets(lens)[:-1]
    else:
        off = np.asarray(out_off, dtype=np.int64).reshape(-1)
        if off.shape != frames.shape:
            raise ValueError(f"out_off needs one offset per item ({len(frames)}), got {off.shape}")
        order = np.argsort(off, kind="stable")
        if (off < 0).any() or (off[order][1:] < (off + lens)[order][:-1]).any():
            raise ValueError("out_off: item outputs must not be negative or overlap")
    return off, lens


class Context:
    """Owns one ``spev_ctx`` (Hann window, twiddles, mel basis + pseudo-inverse for one
    ``(device, sr, n_fft, hop, win, n_mels, fmin, fmax)`` key)."""

    _cache: dict = {}
    _cache_lock = threading.Lock()

    def __init__(self, device: int, sr: int, n_fft: int, hop: int, win: int, n_mels: int,
                 fmin: float, fmax: Optional[float]):
        lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("spev_tts_b200 needs a CUDA (sm_100) device; there is no CPU path")
        self.lib = lib
        self.device = int(device)
        self.sr, self.n_fft, self.hop, self.win, self.n_mels = sr, n_fft, hop, win, n_mels
        self.fmin = float(fmin)
        self.fmax = float(fmax) if fmax is not None else 0.5 * sr
        h = C.c_void_p()
        _lib.check(lib.spev_create(C.byref(h), self.device, sr, n_fft, hop, win, n_mels,
                                   self.fmin, self.fmax), "spev_create")
        self.handle = h

    @classmethod
    def get(cls, device, *, sr=22050, n_fft=1024, hop=256, win=None, n_mels=80, fmin=0.0,
            fmax=None) -> "Context":
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"spev_tts_b200 runs on CUDA devices only (got {dev})")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        win = n_fft if win is None else win
        key = (idx, int(sr), int(n_fft), int(hop), int(win), int(n_mels), float(fmin),
               None if fmax is None else float(fmax))
        with cls._cache_lock:
            ctx = cls._cache.get(key)
            if ctx is None:
                ctx = cls(idx, int(sr), int(n_fft), int(hop), int(win), int(n_mels), fmin, fmax)
                cls._cache[key] = ctx
        return ctx

    def uniform_batch(self, n_items: int, n_frames: int, with_chunks: bool = True,
                      out_len: Optional[int] = None) -> "FlatBatch":
        """Descriptor of ``n_items`` equal-length spectrogram items, cached: the vocoder is called over and over with
        the same shapes, and planning + pinned staging + upload cost more than the kernels of a short utterance.
        ``out_len``: output samples per item (librosa's ``length=``; ``out_layout``'s default when None)."""
        out_len = int(out_layout([n_frames], out_len)[1][0])
        key = (int(n_items), int(n_frames), bool(with_chunks), out_len)
        cache = self.__dict__.setdefault("_uniform", {})
        fb = cache.get(key)
        if fb is None:
            if len(cache) >= 64:
                cache.pop(next(iter(cache)))
            fb = cache[key] = make_batch(self, n_frames=[n_frames] * n_items, with_chunks=with_chunks, out_len=out_len)
        return fb

    def side_stream(self) -> "torch.cuda.Stream":
        """A per-context helper stream (small read-backs that must not queue behind long kernel chains)."""
        st = self.__dict__.get("_side")
        if st is None:
            st = self.__dict__["_side"] = torch.cuda.Stream(torch.device("cuda", self.device))
        return st

    def set_tensor_core(self, enable: bool) -> None:
        """A/B switch: False forces the FFMA kernel for the mel->magnitude projection."""
        _lib.check(self.lib.spev_set_tensor_core(self.handle, 1 if enable else 0), "spev_set_tensor_core")

    def mel_basis(self) -> np.ndarray:
        out = np.empty((self.n_mels, _lib.N_BINS), dtype=np.float32)
        _lib.check(self.lib.spev_get_mel_basis(self.handle, out.ctypes.data), "spev_get_mel_basis")
        return out

    def mel_pinv(self) -> np.ndarray:
        out = np.empty((_lib.N_BINS, self.n_mels), dtype=np.float32)
        _lib.check(self.lib.spev_get_mel_pinv(self.handle, out.ctypes.data), "spev_get_mel_pinv")
        return out

    def window(self) -> np.ndarray:
        out = np.empty(self.n_fft, dtype=np.float32)
        _lib.check(self.lib.spev_get_window(self.handle, out.ctypes.data), "spev_get_window")
        return out

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.spev_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


@dataclass
class FlatBatch:
    """Host + device form of ``struct spev_batch``."""
    n_items: int
    n_frames: int
    frames: np.ndarray          # int64 [n_items]  frames per item
    sample_off: Optional[np.ndarray]   # int64 [n_items] absolute item starts (waveform batches)
    frame_off: np.ndarray       # int64 [n_items+1]
    n_ftiles: int
    n_ctiles: int
    table: torch.Tensor         # device uint8 buffer holding frame_off + tile tables
    desc: _lib.SpevBatch
    device: torch.device
    out_off: np.ndarray         # int64 [n_items] ISTFT output starts (``out_layout``)
    out_len: np.ndarray         # int64 [n_items] ISTFT output lengths (``out_layout``)

    @property
    def n_out_samples(self) -> int:
        """size of the flat ISTFT output buffer: the end of the last item"""
        return int((self.out_off + self.out_len).max(initial=0))

    def out_sample_off(self) -> np.ndarray:
        """[n_items + 1]: item i's output starts at entry i; the last entry is ``n_out_samples``.  Items may have gaps
        between them (starts rounded up to 4 samples, or given offsets), which no kernel writes."""
        return np.append(self.out_off, self.n_out_samples).astype(np.int64)

    def out_lengths(self) -> np.ndarray:
        """[n_items] ISTFT output samples per item."""
        return self.out_len.copy()

    def output_items(self, y: torch.Tensor) -> torch.Tensor:
        """``[n_items, L]`` items of an equal-length batch from its flat ISTFT output ``y`` (``n_out_samples``
        samples): a view when the items are back to back, a contiguous copy when starts are padded apart."""
        off, lens = self.out_sample_off()[:-1], self.out_lengths()
        L = int(lens[0]) if self.n_items else 0
        pitch = int(off[1] - off[0]) if self.n_items > 1 else L
        if (lens != L).any() or (np.diff(off) != pitch).any() or pitch < L:
            raise ValueError("output_items needs items of one length at one spacing")
        if y.dim() != 1 or not y.is_contiguous() or y.numel() < self.n_out_samples:
            raise ValueError(f"output_items: y must be a flat buffer of >= {self.n_out_samples} samples")
        items = y.as_strided((self.n_items, L), (pitch, 1), y.storage_offset() + (int(off[0]) if self.n_items else 0))
        return items if pitch == L else items.contiguous()


def make_batch(ctx: Context, *, n_samples: Optional[Sequence[int]] = None,
               n_frames: Optional[Sequence[int]] = None, sample_off: Optional[np.ndarray] = None,
               with_chunks: bool = False, pinned: bool = True, out_len=None,
               out_off: Optional[Sequence[int]] = None) -> FlatBatch:
    """Build the descriptor for items given by sample counts (waveform inputs) or frame counts
    (spectrogram inputs; frame tiles then describe their ISTFT outputs).
    ``sample_off[i]`` is the absolute start of item i in the flat sample buffer (default: items
    packed back to back).  Starts that are multiples of 4 samples take the 16-byte cp.async path;
    whatever lies between items is never read as signal (explicit [lo, hi) bounds per item).
    ``out_len`` / ``out_off`` (spectrogram inputs only): item i's ISTFT output has ``out_len[i]`` samples at
    ``out_off[i]`` (librosa's ``length=``; see ``out_layout`` for the defaults); frame and chunk tiles follow that
    layout."""
    dev = torch.device("cuda", ctx.device)
    if n_samples is not None and (out_len is not None or out_off is not None):
        raise ValueError("out_len / out_off describe ISTFT outputs: give n_frames, not n_samples")
    if n_samples is not None:
        ns = np.asarray(n_samples, dtype=np.int64).reshape(-1)
        frames = 1 + ns // HOP
        if sample_off is None:
            sample_off = np.concatenate([[0], np.cumsum(ns)])[:-1].astype(np.int64)
        else:
            sample_off = np.asarray(sample_off, dtype=np.int64).reshape(-1)[: len(ns)]
        ftiles = plan_frame_tiles(frames, sample_off, ns)
        out_off, out_len = out_layout(frames)
    else:
        frames = np.asarray(n_frames, dtype=np.int64).reshape(-1)
        sample_off = None
        out_off, out_len = out_layout(frames, out_len, out_off)
        ftiles = plan_frame_tiles(frames, out_off, out_len)
    n_items = int(len(frames))
    frame_off = np.concatenate([[0], np.cumsum(frames)]).astype(np.int64)
    ctiles = (plan_chunk_tiles(frames, out_off=out_off, out_len=out_len) if with_chunks
              else np.zeros(0, dtype=TILE_DTYPE))

    # one staging buffer: [ftiles | ctiles | frame_off]; tile tables first (16-byte aligned)
    parts = [ftiles.view(np.uint8).reshape(-1), ctiles.view(np.uint8).reshape(-1),
             frame_off.view(np.uint8).reshape(-1)]
    sizes = [p.size for p in parts]
    host = torch.from_numpy(np.concatenate(parts))
    if pinned:
        host = host.pin_memory()
    table = host.to(dev, non_blocking=True)
    base = table.data_ptr()
    assert base % 16 == 0
    d = _lib.SpevBatch()
    d.n_items = n_items
    d.n_ftiles = len(ftiles)
    d.n_ctiles = len(ctiles)
    d.n_frames = int(frame_off[-1])
    d.ftiles = base if len(ftiles) else None
    d.ctiles = base + sizes[0] if len(ctiles) else None
    d.frame_off = base + sizes[0] + sizes[1]
    fb = FlatBatch(n_items=n_items, n_frames=int(frame_off[-1]), frames=frames,
                   sample_off=sample_off, frame_off=frame_off, n_ftiles=len(ftiles),
                   n_ctiles=len(ctiles), table=table, desc=d, device=dev, out_off=out_off, out_len=out_len)
    fb._host = host   # keep the pinned staging buffer alive until the async copy is consumed
    return fb
