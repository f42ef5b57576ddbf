"""CPU tests of ``length=`` (librosa's exact-length inverse transforms): the restated istft against torch.istft, the
Griffin-Lim loop with ``length`` against torchaudio, and the host planner of the output-length layout."""
import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr
from spev_tts_b200 import batch as B
from tests import length_ref, synth


def _lengths(T):
    """Shorter than (T-1)*256 (frames drop), (T-1)*256, +1, T*256 - 1, and longer than the signal (zero padding)."""
    full = (T - 1) * 256
    out = [full - 300, full - 1, full, full + 1, T * 256 - 1, (T + 1) * 256, (T + 3) * 256 + 17]
    return sorted({L for L in out if L > 0})


@pytest.mark.parametrize("T", [1, 2, 3, 33, 100])
def test_istft_length_vs_torch_float64(T):
    rng = np.random.default_rng(T)
    X = rng.standard_normal((513, T)) + 1j * rng.standard_normal((513, T))
    w = torch.hann_window(1024, periodic=True, dtype=torch.float64)
    for L in _lengths(T):
        got = lr.istft(X, hop_length=256, n_fft=1024, dtype=np.float64, length=L)
        ref = torch.istft(torch.from_numpy(X), 1024, 256, 1024, w, center=True, length=L).numpy()
        assert got.shape == ref.shape == (L,)
        assert np.abs(got - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max()), (T, L)
        if L > (T + 1) * 256:
            assert not got[(T + 1) * 256:].any()                 # zero padding past the last frame


def test_istft_length_zero_is_empty():
    rng = np.random.default_rng(0)
    X = (rng.standard_normal((2, 513, 5)) + 1j * rng.standard_normal((2, 513, 5))).astype(np.complex64)
    y = lr.istft(X, hop_length=256, n_fft=1024, length=0)
    assert y.shape == (2, 0) and y.dtype == np.float32


def test_griffinlim_length_loop_against_torchaudio(monkeypatch):
    """The loop with ``length`` against torchaudio's griffinlim(length=...), which also passes the length to every
    inner istft.  As in test_oracle.py's loop test, the re-analysis is swapped for a reflect-padded stft (torchaudio's
    padding) for this comparison only."""
    import torchaudio
    T, n_iter = 60, 8
    plain_stft = lr.stft

    def stft_reflect(y, *, n_fft=2048, hop_length=None, **kw):
        pad = [(0, 0)] * (np.ndim(y) - 1) + [(n_fft // 2, n_fft // 2)]
        return plain_stft(np.pad(y, pad, mode="reflect"), n_fft=n_fft, hop_length=hop_length, center=False)
    for L in ((T - 1) * 256, (T - 1) * 256 + 1, (T - 1) * 256 + 100, T * 256 - 1):
        y0 = synth.speechy(seed=78, n=L)
        S = np.abs(plain_stft(y0, n_fft=1024, hop_length=256)).astype(np.float32)
        assert S.shape == (513, T)
        monkeypatch.setattr(lr, "stft", stft_reflect)
        got = length_ref.griffinlim(S, n_iter=n_iter, init_phase=np.zeros(S.shape), length=L)
        monkeypatch.setattr(lr, "stft", plain_stft)
        ref = torchaudio.functional.griffinlim(torch.from_numpy(S).double(), torch.hann_window(1024, periodic=True, dtype=torch.float64),
                                               n_fft=1024, hop_length=256, win_length=1024, power=1.0, n_iter=n_iter,
                                               momentum=0.99, length=L, rand_init=False).numpy()
        assert got.shape == ref.shape == (L,)
        err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert err <= 1e-4, (L, err)


def test_griffinlim_length_of_whole_chunks_is_the_default():
    g = synth.speechy(seed=79, n=40 * 256)
    S = np.abs(lr.stft(g, n_fft=1024, hop_length=256)).astype(np.float32)        # [513, 41]
    ph = synth.init_phase(S.shape, seed=80)
    plain = lr.griffinlim(S, n_iter=4, hop_length=256, n_fft=1024, init_phase=ph)
    assert np.array_equal(length_ref.griffinlim(S, n_iter=4, init_phase=ph), plain)
    assert np.array_equal(length_ref.griffinlim(S, n_iter=4, init_phase=ph, length=40 * 256), plain)
    tail = length_ref.griffinlim(S, n_iter=4, init_phase=ph, length=40 * 256 + 200)
    assert tail.shape == (40 * 256 + 200,) and np.abs(tail[40 * 256:]).max() > 0
    assert not np.array_equal(tail[: 40 * 256], plain)         # the tail is re-analysed in every iteration


@pytest.fixture(scope="module")
def built():
    """The tile planners are the library's (spev_plan_*_tiles): build it first."""
    from spev_tts_b200 import build
    build.build()


def test_c_length_planner_covers_every_sample_once(built):
    rng = np.random.default_rng(5)
    for trial in range(20):
        n = int(rng.integers(1, 12))
        frames = rng.integers(1, 200, n)
        lens = rng.integers(0, 260 * 200, n) if trial % 2 else (frames - 1) * 256 + rng.integers(0, 256, n)
        if trial % 4 == 3:          # explicit, unaligned offsets with gaps
            gaps = rng.integers(0, 50, n)
            offs = np.cumsum(np.concatenate([[0], lens[:-1] + gaps[:-1]])) + gaps[0]
            off, L = B.out_layout(frames, lens, offs)
            assert np.array_equal(off, offs)
        else:
            off, L = B.out_layout(frames, lens)
            assert (off % 4 == 0).all() and off[0] == 0
        tiles = B.plan_chunk_tiles(frames, out_off=off, out_len=L)
        end = int((off + L).max(initial=0)) + 300
        count = np.zeros(end + 29 * 256, dtype=np.int64)
        for t in tiles:
            i = t["item"]
            assert t["lo"] == off[i] and t["hi"] == off[i] + L[i] and t["T"] == frames[i]
            assert t["src0"] == off[i] + 256 * t["t0"] and 1 <= t["n"] <= 29
            assert t["row0"] == frames[:i].sum() + t["t0"] - 1
            a = int(t["src0"])
            b = min(a + 256 * int(t["n"]), int(t["hi"]))
            assert b > a + 256 * (int(t["n"]) - 1)            # only the last chunk of an item may be partial
            count[a:b] += 1
        want = np.zeros_like(count)
        for i in range(n):
            want[off[i]: off[i] + L[i]] += 1
        assert np.array_equal(count, want), trial
        full = tiles["n"] == 29
        assert not (full[1:] & ~full[:-1]).any()               # full tiles first
        ft = B.plan_frame_tiles(frames, off, L)
        assert np.array_equal(ft["lo"], off[ft["item"]]) and np.array_equal(ft["hi"], (off + L)[ft["item"]])
    # the default layout: (T-1)*256 samples per item, bounded like any other
    frames = np.array([800, 33, 1, 2, 64])
    off, L = B.out_layout(frames)
    assert np.array_equal(L, (frames - 1) * 256) and np.array_equal(off, np.concatenate([[0], np.cumsum(L)[:-1]]))
    tiles = B.plan_chunk_tiles(frames, out_off=off, out_len=L)
    assert np.array_equal(tiles["lo"], off[tiles["item"]]) and np.array_equal(tiles["hi"], (off + L)[tiles["item"]])


def test_default_layout_of_items_without_frames(built):
    """Items with T = 0 take no output samples, leading or in the middle: every bound and chunk start is >= 0, the
    items are disjoint, and the buffer ends at the last item's end."""
    for frames in ([0, 5], [3, 0, 0, 40], [0, 0, 2, 0, 33, 0]):
        frames = np.array(frames)
        off, L = B.out_layout(frames)
        assert np.array_equal(L, np.maximum(frames - 1, 0) * 256)
        order = np.argsort(off, kind="stable")
        assert (off >= 0).all() and (off[order][1:] >= (off + L)[order][:-1]).all()
        ft = B.plan_frame_tiles(frames, off, L)
        ct = B.plan_chunk_tiles(frames, out_off=off, out_len=L)
        for t in (ft, ct):
            assert (t["lo"] >= 0).all() and np.array_equal(t["hi"], (off + L)[t["item"]])
        assert (ct["src0"] >= 0).all() and (ct["src0"] + 256 * ct["n"] <= ct["hi"]).all()
        assert set(ft["item"]) == set(np.flatnonzero(frames >= 1)) and set(ct["item"]) == set(np.flatnonzero(frames >= 2))
        assert int((off + L).max()) == int(L.sum())                # [0, 5]: the 1,024 samples item 1 needs


def test_out_layout_rejects_bad_layouts():
    with pytest.raises(ValueError):
        B.out_layout([3, 3], [-1, 5])
    with pytest.raises(ValueError):
        B.out_layout([3, 3], [600, 600], [0, 599])             # overlapping items
    with pytest.raises(ValueError):
        B.out_layout([3, 3], [600, 600], [0])
    assert B.out_layout([3, 3, 3], 513)[0].tolist() == [0, 516, 1032]


def test_output_items_of_the_flat_output_layout():
    """``FlatBatch.output_items``: a view of back-to-back items, a copy of items whose starts are padded to 4 samples,
    from a buffer of exactly ``n_out_samples``; unequal lengths or spacing are refused."""
    def host_batch(frames, out_len=None, out_off=None):
        frames = np.asarray(frames, dtype=np.int64)
        out_off, out_len = B.out_layout(frames, out_len, out_off)
        fo = np.concatenate([[0], np.cumsum(frames)])
        return B.FlatBatch(len(frames), int(fo[-1]), frames, None, fo, 0, 0, None, None, torch.device("cpu"),
                           out_off=out_off, out_len=out_len)
    for out_len, back_to_back in ((None, True), (99 * 256 + 8, True), (99 * 256 + 5, False), (0, True)):
        fb = host_batch([100] * 3, None if out_len is None else [out_len] * 3)
        L = 99 * 256 if out_len is None else out_len
        y = torch.arange(fb.n_out_samples, dtype=torch.float32)
        items = fb.output_items(y)
        pitch = L if back_to_back else (L + 3) // 4 * 4
        assert items.shape == (3, L) and items.is_contiguous()
        assert torch.equal(items, torch.stack([y[i * pitch: i * pitch + L] for i in range(3)]))
        assert (items.data_ptr() == y.data_ptr()) == back_to_back
    for fb in (host_batch([100, 99]), host_batch([100] * 3, [512] * 3, [0, 512, 1200])):
        with pytest.raises(ValueError, match="one length at one spacing"):
            fb.output_items(torch.zeros(fb.n_out_samples))
    fb = host_batch([100] * 2, [600] * 2)
    with pytest.raises(ValueError):
        fb.output_items(torch.zeros(fb.n_out_samples - 1))


def test_griffinlim_length_outside_the_frame_range_is_a_value_error():
    """librosa's loop needs the re-analysis to return T frames: 1 + length // 256 == T.  Checked before any device
    work, naming the valid range."""
    import spev_tts_b200 as sp
    S = np.zeros((513, 10), np.float32)
    for L in (9 * 256 - 1, 10 * 256, -1):
        with pytest.raises(ValueError, match="2304" if L >= 0 else "non-negative"):
            sp.griffinlim(S, n_iter=1, length=L)
        with pytest.raises(ValueError):
            sp.mel_to_audio(np.zeros((80, 10), np.float32), sr=22050, n_fft=1024, hop_length=256, length=L)
    with pytest.raises(ValueError):
        sp.istft(np.zeros((513, 4), np.complex64), length=-3)
