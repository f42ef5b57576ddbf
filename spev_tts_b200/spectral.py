"""Host-side mirror of the librosa calls on the reference's spectral hot path.

Same names, argument meaning and return shapes as the calls the reference makes
(``librosa.feature.melspectrogram`` at ``spev_real_metrics.py:363``;
``librosa.feature.inverse.mel_to_audio`` at ``:730-733``), but every flop runs in the sm_100a
kernels behind ``include/spev_b200.h``.  Inputs may be numpy arrays or torch tensors (any
device); the result comes back as the same kind (numpy -> numpy; torch -> torch on the
compute device).  Leading batch dimensions broadcast like librosa's.

Ragged batches (the cache build) use the ``*_flat`` functions, which take one flat device
buffer plus per-item lengths.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from .batch import HOP, N_FFT, Context, FlatBatch, make_batch, stream_ptr

ArrayLike = Union[np.ndarray, torch.Tensor]
REF_LOG_FLOOR, REF_LOG_LO, REF_LOG_HI = 1e-5, -10.0, 2.0   # spev_real_metrics.py:364-366


def default_device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("spev_tts_b200 needs a CUDA (sm_100) device; there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(a: ArrayLike, device: Optional[torch.device], dtype=torch.float32) -> Tuple[torch.Tensor, bool]:
    """-> (contiguous device tensor, was_numpy)"""
    was_numpy = not isinstance(a, torch.Tensor)
    t = torch.from_numpy(np.ascontiguousarray(a)) if was_numpy else a
    if device is None:
        device = t.device if t.is_cuda else default_device()
    t = t.to(device=device, dtype=dtype, non_blocking=True).contiguous()
    return t, was_numpy


def _ret(t: torch.Tensor, was_numpy: bool):
    return t.cpu().numpy() if was_numpy else t


def items_to_rows(t: torch.Tensor, pitch: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """librosa layout ``[b, R, T]`` -> frame-major rows ``[b*T, pitch]`` (first ``R`` columns; ``pitch`` defaults to ``R``)
    in one launch of ``spev_transpose_batched`` (float32 or complex64).  Pad columns are left as they are."""
    b, R, T = t.shape
    pitch = R if pitch is None else pitch
    t = t.contiguous()
    if out is None:
        out = torch.empty((b * T, pitch), dtype=t.dtype, device=t.device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.load().spev_transpose_batched(t.data_ptr(), out.data_ptr(), t.element_size(), b, R, T, T, R * T,
                                                      pitch, T * pitch, stream_ptr(t.device)), "spev_transpose_batched")
    return out


def rows_to_items(rows: torch.Tensor, b: int, T: int, R: int) -> torch.Tensor:
    """frame-major rows ``[b*T, pitch]`` -> librosa layout ``[b, R, T]`` (the first ``R`` columns of every row)."""
    pitch = rows.shape[1]
    out = torch.empty((b, R, T), dtype=rows.dtype, device=rows.device)
    with torch.cuda.device(rows.device):
        _lib.check(_lib.load().spev_transpose_batched(rows.data_ptr(), out.data_ptr(), rows.element_size(), b, T, R, pitch,
                                                      T * pitch, T, R * T, stream_ptr(rows.device)), "spev_transpose_batched")
    return out


def _check_fixed(n_fft, hop_length, win_length, window, center, pad_mode, power=2.0):
    if hop_length is None:
        hop_length = (win_length or n_fft) // 4
    if n_fft != N_FFT or hop_length != HOP or (win_length not in (None, N_FFT)):
        raise NotImplementedError(
            f"spev_tts_b200 implements the reference CONFIG only (n_fft=1024, hop=256, win=1024); "
            f"got n_fft={n_fft}, hop_length={hop_length}, win_length={win_length}")
    if window != "hann" or not center or pad_mode != "constant" or power != 2.0:
        raise NotImplementedError("only window='hann', center=True, pad_mode='constant', power=2.0 "
                                  "(the reference's librosa defaults) are implemented")


# ---------------------------------------------------------------------------------------------
# forward: STFT -> power -> mel (-> log)
# ---------------------------------------------------------------------------------------------
def logmel_flat(samples: torch.Tensor, n_samples: Sequence[int], *, sr=22050, n_mels=80, fmin=0.0,
                fmax=None, log=True, floor=REF_LOG_FLOOR, lo=REF_LOG_LO, hi=REF_LOG_HI,
                sample_off: Optional[np.ndarray] = None, out: Optional[torch.Tensor] = None,
                batch: Optional[FlatBatch] = None) -> Tuple[torch.Tensor, FlatBatch]:
    """Ragged batch: ``samples`` is one flat float32 CUDA tensor holding all items.
    Returns (``[F, n_mels]`` float32 -- the reference's stored cache layout ``mel.T``,
    ``spev_real_metrics.py:421`` -- and the batch descriptor with ``frame_off``)."""
    if not (samples.is_cuda and samples.dtype == torch.float32 and samples.is_contiguous()):
        raise ValueError("samples must be a contiguous float32 CUDA tensor")
    ctx = Context.get(samples.device, sr=sr, n_mels=n_mels, fmin=fmin, fmax=fmax)
    if batch is None:
        batch = make_batch(ctx, n_samples=n_samples, sample_off=sample_off)
    if out is None:
        out = torch.empty((batch.n_frames, n_mels), dtype=torch.float32, device=samples.device)
    _lib.check(ctx.lib.spev_logmel(ctx.handle, batch.desc, samples.data_ptr(), out.data_ptr(),
                                   1 if log else 0, float(floor), float(lo), float(hi),
                                   stream_ptr(samples.device)), "spev_logmel")
    return out, batch


def melspectrogram(*, y: ArrayLike, sr=22050, n_fft=2048, hop_length=512, win_length=None,
                   window="hann", center=True, pad_mode="constant", power=2.0, n_mels=128,
                   fmin=0.0, fmax=None, device=None):
    """Drop-in for ``librosa.feature.melspectrogram(y=...)`` -> ``[..., n_mels, T]``."""
    _check_fixed(n_fft, hop_length, win_length, window, center, pad_mode, power)
    t, was_numpy = _to_device(y, device)
    lead, n = t.shape[:-1], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    mel, fb = logmel_flat(t.reshape(-1), [n] * b, sr=sr, n_mels=n_mels, fmin=fmin, fmax=fmax, log=False)
    T = 1 + n // HOP
    mel = rows_to_items(mel, b, T, n_mels).view(*lead, n_mels, T)
    return _ret(mel, was_numpy)


def logmel(y: ArrayLike, *, sr=22050, n_mels=80, device=None):
    """The reference's four statements ``spev_real_metrics.py:363-367`` + the stored layout
    of ``:421``: ``[..., N] -> [..., T, n_mels]`` float32 log-mel clamped to [-10, 2]."""
    t, was_numpy = _to_device(y, device)
    lead, n = t.shape[:-1], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    mel, _ = logmel_flat(t.reshape(-1), [n] * b, sr=sr, n_mels=n_mels, log=True)
    return _ret(mel.view(*lead, 1 + n // HOP, n_mels), was_numpy)


def stft_power_flat(samples: torch.Tensor, n_samples: Sequence[int], *, sr=22050):
    """|STFT|^2 as ``[F, 520]`` (pad columns zero): A operand of the tensor-core mel GEMM."""
    ctx = Context.get(samples.device, sr=sr)
    batch = make_batch(ctx, n_samples=n_samples)
    out = torch.empty((batch.n_frames, _lib.SPEC_LD), dtype=torch.float32, device=samples.device)
    _lib.check(ctx.lib.spev_stft_power(ctx.handle, batch.desc, samples.data_ptr(), out.data_ptr(),
                                       stream_ptr(samples.device)), "spev_stft_power")
    return out, batch


def mel_project(power: torch.Tensor, *, sr=22050, n_mels=80, fmin=0.0, fmax=None, log=True,
                floor=REF_LOG_FLOOR, lo=REF_LOG_LO, hi=REF_LOG_HI):
    """Tensor-core (tcgen05 3xTF32) mel projection of a ``[F, 520]`` power spectrum."""
    ctx = Context.get(power.device, sr=sr, n_mels=n_mels, fmin=fmin, fmax=fmax)
    out = torch.empty((power.shape[0], n_mels), dtype=torch.float32, device=power.device)
    _lib.check(ctx.lib.spev_mel_project(ctx.handle, power.data_ptr(), power.shape[0], out.data_ptr(),
                                        1 if log else 0, float(floor), float(lo), float(hi),
                                        stream_ptr(power.device)), "spev_mel_project")
    return out


# ---------------------------------------------------------------------------------------------
# STFT / ISTFT (complex, librosa layout [..., 513, T])
# ---------------------------------------------------------------------------------------------
def _spec_to_internal(X: torch.Tensor) -> torch.Tensor:
    """[B, 513, T] complex64 -> [B*T, 520] complex64 (frame-major rows, pitch 520)."""
    B, nb, T = X.shape
    buf = torch.zeros((B * T, _lib.SPEC_LD), dtype=torch.complex64, device=X.device)
    return items_to_rows(X, _lib.SPEC_LD, out=buf)


def stft(y: ArrayLike, *, n_fft=2048, hop_length=None, win_length=None, window="hann", center=True,
         pad_mode="constant", device=None):
    """Drop-in for ``librosa.stft`` -> complex64 ``[..., 513, T]``."""
    _check_fixed(n_fft, hop_length, win_length, window, center, pad_mode)
    t, was_numpy = _to_device(y, device)
    lead, n = t.shape[:-1], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    T = 1 + n // HOP
    Tc = T
    if n % HOP:
        # spev_stft takes the ISTFT-output item layout ((T-1)*hop samples per item).  Zero-extend
        # to the next multiple of hop -- every one of the first T frames is unchanged because
        # centre padding is zeros -- compute T+1 frames and drop the last.
        t = torch.nn.functional.pad(t.reshape(b, n), (0, HOP - n % HOP)).contiguous()
        Tc = T + 1
    ctx = Context.get(t.device)
    batch = make_batch(ctx, n_frames=[Tc] * b)
    spec = torch.empty((b * Tc, _lib.SPEC_LD), dtype=torch.complex64, device=t.device)
    _lib.check(ctx.lib.spev_stft(ctx.handle, batch.desc, t.data_ptr(), spec.data_ptr(), _lib.SPEC_LD,
                                 stream_ptr(t.device)), "spev_stft")
    out = rows_to_items(spec, b, Tc, _lib.N_BINS)
    if Tc != T:
        out = out[:, :, :T].contiguous()
    out = out.reshape(*lead, _lib.N_BINS, T)
    return _ret(out, was_numpy)


def _check_length(length) -> Optional[int]:
    if length is None:
        return None
    if isinstance(length, (bool, np.bool_)) or not isinstance(length, (int, np.integer)) or length < 0:
        raise ValueError(f"length must be a non-negative integer or None, got {length!r}")
    return int(length)


def _gl_length(length, T: int) -> Optional[int]:
    """librosa's Griffin-Lim loop re-analyses each istft(length=L) output and needs T frames back: 1 + L // hop == T."""
    length = _check_length(length)
    if length is not None and 1 + length // HOP != T:
        raise ValueError(f"length={length} is outside [{(T - 1) * HOP}, {T * HOP - 1}], the lengths whose STFT has the "
                         f"T={T} frames of the input (librosa's Griffin-Lim loop needs 1 + length // {HOP} == T)")
    return length


def istft(X: ArrayLike, *, hop_length=None, win_length=None, n_fft=None, window="hann", center=True,
          dtype=None, length=None, device=None):
    """Drop-in for ``librosa.istft`` -> float32 ``[..., (T-1)*hop]``, or ``[..., length]`` with librosa's crop / zero
    padding (any ``length >= 0``).  The kernels write exactly ``length`` samples per item."""
    nb = X.shape[-2]
    _check_fixed(n_fft or 2 * (nb - 1), hop_length, win_length, window, center, "constant")
    length = _check_length(length)
    t, was_numpy = _to_device(X, device, dtype=torch.complex64)
    lead, T = t.shape[:-2], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    ctx = Context.get(t.device)
    batch = make_batch(ctx, n_frames=[T] * b, with_chunks=True, out_len=length)
    spec = _spec_to_internal(t.reshape(b, nb, T))
    y = torch.empty(batch.n_out_samples, dtype=torch.float32, device=t.device)
    _lib.check(ctx.lib.spev_istft(ctx.handle, batch.desc, spec.data_ptr(), _lib.SPEC_LD, y.data_ptr(),
                                  stream_ptr(t.device)), "spev_istft")
    items = batch.output_items(y)
    return _ret(items.view(*lead, items.shape[1]), was_numpy)


# ---------------------------------------------------------------------------------------------
# inverse: mel -> magnitude -> Griffin-Lim
# ---------------------------------------------------------------------------------------------
def mel_to_mag_flat(mel: torch.Tensor, batch: FlatBatch, ctx: Context, *, layout: int, is_log: bool,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty((batch.n_frames, _lib.SPEC_LD), dtype=torch.float32, device=mel.device)
    _lib.check(ctx.lib.spev_mel_to_mag(ctx.handle, batch.desc, mel.data_ptr(), layout, 1 if is_log else 0,
                                       out.data_ptr(), _lib.SPEC_LD, stream_ptr(mel.device)),
               "spev_mel_to_mag")
    return out


MAX_MEM_BLOCK = 2 ** 18      # librosa.util.utils.MAX_MEM_BLOCK: nnls solves this many bytes of columns at a time
NNLS_PGTOL = 1e-5            # scipy.optimize.fmin_l_bfgs_b default pgtol


def nnls_blocks(b: int, T: int, n_mels: int):
    """librosa.util.nnls's column blocks for ``b`` stacked ``[n_mels, T]`` float32 items:
    ``n_columns = max(1, MAX_MEM_BLOCK // (prod(B.shape[:-1]) * itemsize))``; one block if ``T <= n_columns``."""
    n_columns = max(1, MAX_MEM_BLOCK // (b * n_mels * 4))
    blocks = [(0, T)] if T <= n_columns else [(s0, min(T, s0 + n_columns)) for s0 in range(0, T, n_columns)]
    return n_columns, blocks


def nnls_refine(S: torch.Tensor, mel_rows: torch.Tensor, ctx: Context, b: int, T: int, *, is_log: bool, overlap=None) -> int:
    """The L-BFGS-B part of ``librosa.util.nnls`` (inside ``mel_to_stft``, ``spev_real_metrics.py:730``), in place on the
    warm start ``S = clip(pinv(A) M, 0) ** 0.5`` (``[b*T, 520]`` magnitude rows; ``mel_rows``: ``[b*T, n_mels]``).

    librosa cuts the columns into blocks of ``MAX_MEM_BLOCK // (prod(lead) * n_mels * 4)`` and runs scipy's L-BFGS-B on
    each, started at the warm start.  Its first act is the convergence test ``max |projected gradient| <= pgtol``; the
    objective carries a ``1 / B.size`` factor, so for blocks of >~ 40 columns of reference-range input the test passes
    at once and the warm start IS the answer.  One launch of ``spev_nnls_objective`` evaluates that test for every
    block (float64, as in librosa); only blocks that fail it -- short utterances, short remainder blocks -- are handed
    to ``scipy.optimize.fmin_l_bfgs_b`` (the very routine librosa calls, same arguments), with objective and gradient
    evaluated on the GPU.  Returns the number of blocks that iterated.

    ``overlap``: a callable that enqueues work which only READS ``S`` (``mel_to_audio`` passes the Griffin-Lim call): it runs
    right after the screening kernels have been launched, and their result is fetched through a side stream, so the host
    does not sit in a synchronisation while the device is idle.  If blocks do iterate, ``S`` changes afterwards (stream
    ordered behind that work) and the caller must redo it."""
    n_mels = ctx.n_mels
    n_columns, blocks = nnls_blocks(b, T, n_mels)
    dev = S.device
    lib, st = ctx.lib, stream_ptr(dev)
    pg = torch.empty(b * T, dtype=torch.float64, device=dev)          # per column, block after block
    val = torch.empty(b * T, dtype=torch.float64, device=dev)
    # Screening: librosa's blocks are equal-sized except the last, so all full blocks go in ONE launch (columns
    # [0, n_full * n_columns), objective scaled for one block) and the remainder in a second; pg comes back per column
    # in (item, column-of-the-launch) order.
    n_full = T // n_columns if T > n_columns else 0
    launches = []                                   # (t0, tb, size_cols, offset into pg)
    if n_full:
        launches.append((0, n_full * n_columns, n_columns, 0))
    if T - n_full * n_columns > 0:
        launches.append((n_full * n_columns, T - n_full * n_columns, 0, b * n_full * n_columns))

    def screen(mode, overlap=None):
        for t0, tb, sc, o in launches:
            _lib.check(lib.spev_nnls_objective(ctx.handle, S.data_ptr(), mode, S.shape[1], mel_rows.data_ptr(), 1 if is_log else 0,
                                               b, T, t0, tb, sc, val[o:].data_ptr(), None, pg[o:].data_ptr(), st),
                       "spev_nnls_objective")
        if overlap is None:
            host = pg.cpu().numpy()                 # (one synchronisation per pass)
        else:
            main = torch.cuda.current_stream(dev)
            side = ctx.side_stream()
            pinned = torch.empty(b * T, dtype=torch.float64, pin_memory=True)   # (torch's caching host allocator: per call, thread-safe)
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                pinned.copy_(pg, non_blocking=True)
            pg.record_stream(side)
            overlap()                               # e.g. the whole Griffin-Lim call, enqueued behind the screening
            side.synchronize()                      # waits for the screening + copy only
            host = pinned.numpy()
        out = {}
        for t0, tb, sc, o in launches:
            cols = host[o: o + b * tb].reshape(b, tb)
            for s0 in range(0, tb, sc or tb):
                out[(t0 + s0, t0 + min(tb, s0 + (sc or tb)))] = float(cols[:, s0: s0 + (sc or tb)].max(initial=0.0))
        return out
    # float32 screening pass; if any block lies within 10 % of the threshold the pass is repeated in float64
    norm = screen(2, overlap)
    if any(0.9 * NNLS_PGTOL <= v <= 1.1 * NNLS_PGTOL for v in norm.values()):
        norm = screen(1)
    todo = [blk for blk in blocks if norm[blk] > NNLS_PGTOL]
    if not todo:
        return 0
    try:
        from scipy.optimize import fmin_l_bfgs_b
    except ImportError as e:    # pragma: no cover
        raise RuntimeError("mel_to_stft(nnls='librosa') needs scipy (librosa's own dependency) for the L-BFGS-B "
                           "iterations of short blocks; pass nnls='pinv' for the warm start only") from e
    Sv = S.view(b, T, S.shape[1])
    for t0, t1 in todo:
        tb = t1 - t0
        x0 = Sv[:, t0:t1, : _lib.N_BINS].permute(0, 2, 1).double().square().contiguous()   # [b, 513, tb], librosa's order
        xd = torch.empty_like(x0)
        gd = torch.empty_like(x0)
        vd = torch.empty(b * tb, dtype=torch.float64, device=dev)
        pd = torch.empty(b * tb, dtype=torch.float64, device=dev)

        def fun(xflat):
            xd.copy_(torch.from_numpy(xflat).view_as(xd))
            _lib.check(lib.spev_nnls_objective(ctx.handle, xd.data_ptr(), 0, 0, mel_rows.data_ptr(), 1 if is_log else 0,
                                               b, T, t0, tb, 0, vd.data_ptr(), gd.data_ptr(), pd.data_ptr(), st),
                       "spev_nnls_objective")
            return float(vd.sum().item()), gd.cpu().numpy().reshape(-1)
        x, _, _ = fmin_l_bfgs_b(fun, x0.cpu().numpy().reshape(-1), bounds=[(0, None)] * x0.numel(), m=_lib.N_BINS)
        xs = torch.from_numpy(x).view_as(xd).to(dev).to(torch.float32).sqrt()               # astype(f32) then ** 0.5
        Sv[:, t0:t1, : _lib.N_BINS] = xs.permute(0, 2, 1)
    return len(todo)


def mel_to_stft(M: ArrayLike, *, sr=22050, n_fft=2048, power=2.0, fmin=0.0, fmax=None, nnls="librosa", device=None):
    """Drop-in for ``librosa.feature.inverse.mel_to_stft`` -> ``[..., 513, T]`` magnitudes.
    ``nnls="librosa"`` (default): librosa's result -- the warm start ``clip(pinv(basis) @ M, 0)`` refined by L-BFGS-B
    wherever librosa's own solver iterates (``nnls_refine``); ``nnls="pinv"``: the warm start only (no host
    synchronisation; identical for reference-range inputs of >~ 40 frames, see DESIGN.md "NNLS")."""
    _check_fixed(n_fft, HOP, None, "hann", True, "constant", power)
    if nnls not in ("librosa", "pinv"):
        raise ValueError("nnls must be 'librosa' or 'pinv'")
    t, was_numpy = _to_device(M, device)
    lead, n_mels, T = t.shape[:-2], t.shape[-2], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    ctx = Context.get(t.device, sr=sr, n_mels=n_mels, fmin=fmin, fmax=fmax)
    batch = make_batch(ctx, n_frames=[T] * b)
    # [b, n_mels, T] -> frame-major [b*T, n_mels]: the layout the tcgen05 GEMM path takes
    tm = items_to_rows(t.reshape(b, n_mels, T)).view(-1)
    S = mel_to_mag_flat(tm, batch, ctx, layout=0, is_log=False)
    if nnls == "librosa" and b * T > 0:
        nnls_refine(S, tm.view(b * T, n_mels), ctx, b, T, is_log=False)
    out = rows_to_items(S, b, T, _lib.N_BINS).reshape(*lead, _lib.N_BINS, T)
    return _ret(out, was_numpy)


def griffinlim_flat(S: torch.Tensor, batch: FlatBatch, ctx: Context, *, n_iter=32, momentum=0.99,
                    init_phase: Optional[torch.Tensor] = None, seed: int = 0,
                    out: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None):
    """``S``: ``[F, 520]`` float32 magnitudes; ``init_phase``: ``[F, 513]`` float32 radians or None.
    Returns the flat waveform buffer (item i at ``batch.out_sample_off()[i]``, ``batch.out_lengths()[i]`` samples).
    Item i runs librosa's ``griffinlim(length=out_len[i])`` (``make_batch(..., out_len=)``): every inner ISTFT writes
    those samples and the next STFT re-analyses them; items with frames must satisfy ``1 + out_len[i] // 256 == T_i``."""
    lib = ctx.lib
    bad = np.flatnonzero((batch.frames >= 1) & (1 + batch.out_len // HOP != batch.frames))
    if len(bad):
        i = int(bad[0])
        _gl_length(int(batch.out_len[i]), int(batch.frames[i]))      # raises, naming the valid range
    need = lib.spev_griffinlim_workspace_bytes(batch.n_frames)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=S.device)
    if out is None:
        out = torch.empty(batch.n_out_samples, dtype=torch.float32, device=S.device)
    _lib.check(lib.spev_griffinlim(ctx.handle, batch.desc, S.data_ptr(), S.shape[1],
                                   init_phase.data_ptr() if init_phase is not None else None,
                                   int(seed) & (2 ** 64 - 1), int(n_iter), float(momentum), out.data_ptr(),
                                   workspace.data_ptr(), workspace.numel(), stream_ptr(S.device)),
               "spev_griffinlim")
    return out


def _phase_to_internal(init_phase: ArrayLike, b: int, T: int, device) -> torch.Tensor:
    p, _ = _to_device(init_phase, device)
    return items_to_rows(p.reshape(b, _lib.N_BINS, T))


def griffinlim(S: ArrayLike, *, n_iter=32, hop_length=None, win_length=None, n_fft=None, window="hann",
               center=True, dtype=None, length=None, pad_mode="constant", momentum=0.99, init="random",
               random_state=None, init_phase: Optional[ArrayLike] = None, device=None):
    """Drop-in for ``librosa.griffinlim`` (``[..., 513, T]`` magnitudes -> ``[..., (T-1)*hop]``, or ``[..., length]``
    for ``(T-1)*hop <= length < T*hop``: librosa passes ``length`` to every inner istft, so the tail samples are
    rebuilt and re-analysed in each iteration).
    ``init_phase`` (radians, same shape as S) pins the starting phases for parity tests;
    otherwise phases are drawn on the device from ``random_state`` (None -> OS entropy, like
    librosa)."""
    nb = S.shape[-2]
    _check_fixed(n_fft or 2 * (nb - 1), hop_length, win_length, window, center, pad_mode)
    if init not in ("random",):
        raise NotImplementedError("griffinlim: only init='random' is on the reference path")
    length = _gl_length(length, S.shape[-1])
    t, was_numpy = _to_device(S, device)
    lead, T = t.shape[:-2], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    ctx = Context.get(t.device)
    batch = make_batch(ctx, n_frames=[T] * b, with_chunks=True, out_len=length)
    Sf = items_to_rows(t.reshape(b, nb, T), _lib.SPEC_LD, out=torch.zeros((b * T, _lib.SPEC_LD), dtype=torch.float32, device=t.device))
    ph = _phase_to_internal(init_phase, b, T, t.device) if init_phase is not None else None
    seed = int(np.random.SeedSequence(random_state).generate_state(2, dtype=np.uint32).view(np.uint64)[0])
    items = batch.output_items(griffinlim_flat(Sf, batch, ctx, n_iter=n_iter, momentum=momentum, init_phase=ph, seed=seed))
    return _ret(items.view(*lead, items.shape[1]), was_numpy)


def mel_to_audio(M: ArrayLike, *, sr=22050, n_fft=2048, hop_length=None, win_length=None, window="hann",
                 center=True, pad_mode="constant", power=2.0, n_iter=32, length=None, dtype=np.float32,
                 fmin=0.0, fmax=None, momentum=0.99, init_phase: Optional[ArrayLike] = None,
                 random_state=None, is_log=False, nnls="librosa", device=None):
    """Drop-in for ``librosa.feature.inverse.mel_to_audio`` (call site
    ``spev_real_metrics.py:730-733``): ``[..., n_mels, T]`` mel power -> ``[..., (T-1)*hop]``, or ``[..., length]``
    for ``(T-1)*hop <= length < T*hop`` (copy-synthesis: ``length=len(y)`` of the source signal; see ``griffinlim``).
    ``is_log=True`` fuses the reference's ``np.exp`` (``:729``) into the first kernel.  ``nnls``: see ``mel_to_stft``
    (``"pinv"`` keeps the whole call free of host synchronisation)."""
    _check_fixed(n_fft, hop_length, win_length, window, center, pad_mode, power)
    if nnls not in ("librosa", "pinv"):
        raise ValueError("nnls must be 'librosa' or 'pinv'")
    length = _gl_length(length, M.shape[-1])
    t, was_numpy = _to_device(M, device)
    lead, n_mels, T = t.shape[:-2], t.shape[-2], t.shape[-1]
    b = int(np.prod(lead)) if lead else 1
    ctx = Context.get(t.device, sr=sr, n_mels=n_mels, fmin=fmin, fmax=fmax)
    batch = ctx.uniform_batch(b, T, with_chunks=True, out_len=length)
    tm = items_to_rows(t.reshape(b, n_mels, T)).view(-1)                  # frame-major -> tensor-core GEMM
    S = mel_to_mag_flat(tm, batch, ctx, layout=0, is_log=is_log)
    ph = _phase_to_internal(init_phase, b, T, t.device) if init_phase is not None else None
    seed = int(np.random.SeedSequence(random_state).generate_state(2, dtype=np.uint32).view(np.uint64)[0])
    out = {}

    def run_gl():
        out["y"] = griffinlim_flat(S, batch, ctx, n_iter=n_iter, momentum=momentum, init_phase=ph, seed=seed,
                                   out=out.get("y"))
    if nnls == "librosa" and b * T > 0:
        # Griffin-Lim is enqueued on the warm start while the host fetches the screening result; in the (rare: short
        # utterances, short remainder blocks) case that librosa's solver iterates, S is refined and the loop redone
        if nnls_refine(S, tm.view(b * T, n_mels), ctx, b, T, is_log=is_log, overlap=run_gl) > 0 or "y" not in out:
            run_gl()
    else:
        run_gl()
    items = batch.output_items(out["y"])
    return _ret(items.view(*lead, items.shape[1]), was_numpy)
