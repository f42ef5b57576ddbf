"""GPU: exact-length inverse transforms (librosa's ``length=``) for istft, griffinlim and mel_to_audio.
Chunk tiles bound each item's output by [lo, hi); the ISTFT kernels (k_istft, k_ola_pairs) write every sample of it
and nothing else, and the fused Griffin-Lim iteration re-analyses exactly those samples."""
import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr
from tests import length_ref, synth

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FC0DEAD          # a NaN payload no kernel produces


def rel_l2(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _lengths(T):
    full = (T - 1) * 256
    out = [full - 300, full - 1, full, full + 1, full + 131, T * 256 - 1, T * 256, (T + 1) * 256 - 3, (T + 3) * 256 + 17]
    return sorted({L for L in out if L > 0})


@pytest.mark.parametrize("T", [1, 2, 3, 4, 5, 29, 30, 31, 33, 64, 100])
def test_istft_length_vs_oracle(cuda, T):
    import spev_tts_b200 as sp
    rng = np.random.default_rng(100 + T)
    X = (rng.standard_normal((2, 513, T)) + 1j * rng.standard_normal((2, 513, T))).astype(np.complex64)
    for L in _lengths(T):
        ref = lr.istft(X, hop_length=256, n_fft=1024, length=L)
        got = sp.istft(X, hop_length=256, n_fft=1024, length=L)
        assert got.shape == ref.shape == (2, L) and got.dtype == np.float32
        assert rel_l2(got, ref) <= 2e-6, (T, L, rel_l2(got, ref))
        if L > (T + 1) * 256:
            assert not got[:, (T + 1) * 256:].any()
    assert sp.istft(X, hop_length=256, n_fft=1024, length=0).shape == (2, 0)
    one = sp.istft(X[0], hop_length=256, n_fft=1024, length=(T - 1) * 256 + 77)      # no batch dimension
    assert one.shape == ((T - 1) * 256 + 77,)


def test_single_step_on_length_tables(cuda):
    """One Griffin-Lim iteration through spev_istft / spev_gl_phase_update on a batch with out_len: the ISTFT writes the
    tail samples and the phase update's STFT re-analyses them.  rel-L2 <= 1e-5 on every output."""
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    Bn, T = 2, 96
    L = (T - 1) * 256 + 131
    ys = [synth.speechy(seed=20 + b, n=L) for b in range(Bn)]
    S = np.stack([np.abs(lr.stft(y, n_fft=1024, hop_length=256)) for y in ys]).astype(np.float32)
    ph = synth.init_phase(S.shape, seed=21)
    ang0 = (lr.phasor(ph) * S).astype(np.complex64)
    a1, tprev1, _ = length_ref.griffinlim_step(ang0, None, S, length=L)
    a2, tprev2, inv2 = length_ref.griffinlim_step(a1, tprev1, S, length=L)

    ctx = sp.Context.get(cuda)
    fb = sp.make_batch(ctx, n_frames=[T] * Bn, with_chunks=True, out_len=[L] * Bn)
    off = fb.out_sample_off()

    def to_int(Z, dtype):
        t = torch.zeros((Bn * T, _lib.SPEC_LD), dtype=dtype, device=cuda)
        t[:, :513] = torch.from_numpy(np.ascontiguousarray(Z.transpose(0, 2, 1).reshape(Bn * T, 513))).to(cuda)
        return t

    def from_int(t):
        return t[:, :513].reshape(Bn, T, 513).permute(0, 2, 1).cpu().numpy()

    st = torch.cuda.current_stream(cuda).cuda_stream
    ang, tprev, Sd = to_int(a1, torch.complex64), to_int(tprev1, torch.complex64), to_int(S, torch.float32)
    y = torch.zeros(fb.n_out_samples, dtype=torch.float32, device=cuda)
    _lib.check(ctx.lib.spev_istft(ctx.handle, fb.desc, ang.data_ptr(), _lib.SPEC_LD, y.data_ptr(), st))
    yh = y.cpu().numpy()
    assert rel_l2(np.stack([yh[off[b]: off[b] + L] for b in range(Bn)]), inv2) <= 1e-5
    alpha = float(np.float32(0.99 / 1.99))
    _lib.check(ctx.lib.spev_gl_phase_update(ctx.handle, fb.desc, y.data_ptr(), Sd.data_ptr(), _lib.SPEC_LD,
                                            ang.data_ptr(), tprev.data_ptr(), _lib.SPEC_LD, alpha, 1, st))
    assert rel_l2(from_int(tprev), tprev2) <= 1e-5
    assert rel_l2(from_int(ang), a2) <= 1e-5


def _state(seed, T, L):
    y = synth.speechy(seed=seed, n=L)
    lm = lr.reference_logmel(y).T                                                # [80, T]
    assert lm.shape == (80, T)
    S = lr.mel_to_stft(np.exp(lm), sr=22050, n_fft=1024, fmin=0, fmax=8000, lbfgs=False)
    return lm, S


@pytest.mark.parametrize("n_iter", [0, 1, 8, 32])
def test_griffinlim_and_mel_to_audio_length_sc_delta(cuda, n_iter):
    """Shared initial phase: |SC_gpu - SC_oracle| <= 1e-3 for griffinlim(length=) and mel_to_audio(length=), waveform
    rel-L2 <= 1e-5 for n_iter <= 1."""
    import spev_tts_b200 as sp
    # an even and an odd frame count: at odd T the last chunk of k_ola_pairs sums the last pair's fifth chunk and the
    # lone last frame's segment, at even T only the last pair's
    for T, L in ((80, 79 * 256 + 1), (80, 79 * 256 + 200), (80, 80 * 256 - 1), (81, 80 * 256 + 1), (81, 81 * 256 - 1)):
        lm, S = _state(30, T, L)
        ph = synth.init_phase(S.shape, seed=31)
        ref = length_ref.griffinlim(S, n_iter=n_iter, init_phase=ph, length=L)
        sc_ref = lr.spectral_convergence(ref, S)
        # mel_to_audio's waveform is compared with the loop run on its own (tensor-core) magnitudes, so that the
        # tolerance measures Griffin-Lim alone; its SC is taken against the oracle's magnitudes like griffinlim's
        S_dev = sp.mel_to_stft(np.exp(lm), sr=22050, n_fft=1024, fmin=0, fmax=8000, nnls="pinv")
        assert rel_l2(S_dev, S) <= 1e-5
        outs = {"griffinlim": (sp.griffinlim(S, n_iter=n_iter, hop_length=256, n_fft=1024, init_phase=ph, length=L), ref),
                "mel_to_audio": (sp.mel_to_audio(np.exp(lm), sr=22050, n_fft=1024, hop_length=256, fmin=0, fmax=8000,
                                                 n_iter=n_iter, init_phase=ph, length=L, nnls="pinv"),
                                 length_ref.griffinlim(S_dev, n_iter=n_iter, init_phase=ph, length=L))}
        for name, (got, wref) in outs.items():
            assert got.shape == ref.shape == (L,), name
            sc = lr.spectral_convergence(got, S)
            assert abs(sc - sc_ref) <= 1e-3, (name, L, sc, sc_ref)
            if n_iter <= 1:
                assert rel_l2(got, wref) <= 1e-5, (name, L, rel_l2(got, wref))
            print(f"{name} n_iter={n_iter} L={L}: SC gpu {sc:.6f} oracle {sc_ref:.6f} rel-L2 {rel_l2(got, wref):.2e}")


def test_length_of_whole_chunks_is_bit_identical_to_default(cuda):
    import spev_tts_b200 as sp
    T = 70
    lm, S = _state(40, T, (T - 1) * 256)
    S2, lm2 = np.stack([S, S[:, ::-1]]), np.stack([lm, lm[:, ::-1]])
    ph = synth.init_phase(S2.shape, seed=41)
    L = (T - 1) * 256
    for n_iter in (0, 5):
        a = sp.griffinlim(S2, n_iter=n_iter, init_phase=ph, n_fft=1024)
        b = sp.griffinlim(S2, n_iter=n_iter, init_phase=ph, n_fft=1024, length=L)
        assert a.shape == b.shape == (2, L) and np.array_equal(a, b)
    kw = dict(sr=22050, n_fft=1024, hop_length=256, fmin=0, fmax=8000, n_iter=5, init_phase=ph, is_log=True)
    assert np.array_equal(sp.mel_to_audio(lm2, **kw), sp.mel_to_audio(lm2, length=L, **kw))
    X = sp.stft(synth.white(seed=42, n=L), n_fft=1024, hop_length=256)
    assert np.array_equal(sp.istft(X, n_fft=1024), sp.istft(X, n_fft=1024, length=L))


RAGGED = [800, 33, 1, 2, 64, 517, 95]
TAILS = [255, 0, 37, 1, 128, 3, 254]


def _ragged(ctx, cuda, seed, out_off=None):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    lens = [(T - 1) * 256 + k for T, k in zip(RAGGED, TAILS)]
    fb = sp.make_batch(ctx, n_frames=RAGGED, with_chunks=True, out_len=lens, out_off=out_off)
    g = torch.Generator(device=cuda).manual_seed(seed)
    S = torch.rand(fb.n_frames, _lib.SPEC_LD, generator=g, device=cuda)
    ph = torch.rand(fb.n_frames, 513, generator=g, device=cuda) * 6.2831853
    return fb, lens, S, ph


def _items(fb, y):
    """The samples of every item of a flat output, concatenated.  The <= 3 filler samples between items of the default
    layout are never written (the buffer may come from torch.empty): nothing is asserted about them."""
    off, lens = fb.out_sample_off(), fb.out_lengths()
    return torch.cat([y[o: o + n] for o, n in zip(off, lens)])


def test_ragged_length_batch_matches_per_item_calls(cuda):
    import spev_tts_b200 as sp
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    fb, lens, S, ph = _ragged(ctx, cuda, 5)
    flat = sp.griffinlim_flat(S, fb, ctx, n_iter=7, init_phase=ph)
    assert torch.isfinite(_items(fb, flat)).all()
    off, fo = fb.out_sample_off(), fb.frame_off
    for i, (T, L) in enumerate(zip(RAGGED, lens)):
        one = sp.make_batch(ctx, n_frames=[T], with_chunks=True, out_len=[L])
        y = sp.griffinlim_flat(S[fo[i]: fo[i + 1]].contiguous(), one, ctx, n_iter=7, init_phase=ph[fo[i]: fo[i + 1]].contiguous())
        assert torch.equal(y[:L], flat[off[i]: off[i] + L]), (T, L)


def test_length_static_and_dynamic_pair_tickets_agree(cuda):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    n_sms = torch.cuda.get_device_properties(cuda).multi_processor_count
    limits = (0, 1, 3, 16)
    fb, _, S, ph = _ragged(ctx, cuda, 6)
    grids = [min(fb.n_ftiles, lim or n_sms) for lim in limits]
    assert fb.n_ftiles < 8 * grids[0] and any(fb.n_ftiles >= 8 * g for g in grids[1:])
    outs = []
    try:
        for lim in limits:
            _lib.check(ctx.lib.spev_set_sm_limit(ctx.handle, lim))
            outs.append(sp.griffinlim_flat(S, fb, ctx, n_iter=7, init_phase=ph).clone())
    finally:
        _lib.check(ctx.lib.spev_set_sm_limit(ctx.handle, 0))   # the ctx is cached and shared
    ref = _items(fb, outs[0])
    assert torch.isfinite(ref).all()
    for lim, out in zip(limits[1:], outs[1:]):
        assert torch.equal(ref, _items(fb, out)), lim


def test_length_outputs_stay_inside_their_bounds(cuda):
    """Items at explicit offsets with gaps between them (some offsets not multiples of 4: the unaligned load / store
    paths): spev_istft and spev_griffinlim write every sample of each item's [lo, hi) and nothing else."""
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    lens = [(T - 1) * 256 + k for T, k in zip(RAGGED, TAILS)]
    gaps = [5, 64, 3, 1, 300, 7, 16]
    offs = np.cumsum([gaps[0]] + [L + g for L, g in zip(lens[:-1], gaps[1:])]).astype(np.int64)
    fb, _, S, ph = _ragged(ctx, cuda, 7, out_off=offs)
    # the plain ISTFT takes any length: longer than the signal too
    ilens = [L + (600 if i % 2 else 0) for i, L in enumerate(lens)]
    ioffs = np.cumsum([gaps[0]] + [L + g for L, g in zip(ilens[:-1], gaps[1:])]).astype(np.int64)
    fbi = sp.make_batch(ctx, n_frames=RAGGED, with_chunks=True, out_len=ilens, out_off=ioffs)
    st = torch.cuda.current_stream(cuda).cuda_stream
    X = torch.view_as_complex(torch.randn(fb.n_frames, _lib.SPEC_LD, 2, device=cuda))

    def check(y, off, L, what):
        bits = y.view(torch.int32).cpu().numpy()
        inside = np.zeros(len(bits), bool)
        for o, n in zip(off, L):
            inside[o: o + n] = True
        assert (bits[~inside] == SENTINEL).all(), f"{what}: written outside the items"
        assert (bits[inside] != SENTINEL).all(), f"{what}: sample inside an item not written"

    for batch, off, L in ((fbi, ioffs, ilens), (fb, offs, lens)):
        y = torch.full((batch.n_out_samples + 700,), SENTINEL, dtype=torch.int32, device=cuda).view(torch.float32)
        _lib.check(ctx.lib.spev_istft(ctx.handle, batch.desc, X.data_ptr(), _lib.SPEC_LD, y.data_ptr(), st))
        check(y, off, L, "spev_istft")
    y = torch.full((fb.n_out_samples + 700,), SENTINEL, dtype=torch.int32, device=cuda).view(torch.float32)
    sp.griffinlim_flat(S, fb, ctx, n_iter=4, init_phase=ph, out=y)
    check(y, offs, lens, "spev_griffinlim")
    # the same items packed at the default (4-aligned) offsets give the same samples
    fbd, _, _, _ = _ragged(ctx, cuda, 7)
    yd = sp.griffinlim_flat(S, fbd, ctx, n_iter=4, init_phase=ph)
    od = fbd.out_sample_off()
    for i, L in enumerate(lens):
        assert torch.equal(yd[od[i]: od[i] + L], y[offs[i]: offs[i] + L]), i


def test_length_call_is_graph_capturable(cuda):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    fb = sp.make_batch(ctx, n_frames=[120, 33, 64], with_chunks=True, out_len=[119 * 256 + 255, 32 * 256 + 1, 63 * 256 + 100])
    g = torch.Generator(device=cuda).manual_seed(17)
    S = torch.rand(fb.n_frames, _lib.SPEC_LD, generator=g, device=cuda)
    ph = torch.rand(fb.n_frames, 513, generator=g, device=cuda) * 6.2831853
    ws = torch.empty(ctx.lib.spev_griffinlim_workspace_bytes(fb.n_frames), dtype=torch.uint8, device=cuda)
    eager = sp.griffinlim_flat(S, fb, ctx, n_iter=5, init_phase=ph, workspace=ws).clone()
    y = torch.zeros(fb.n_out_samples, device=cuda)
    s = torch.cuda.Stream(cuda)
    s.wait_stream(torch.cuda.current_stream(cuda))
    with torch.cuda.stream(s):
        sp.griffinlim_flat(S, fb, ctx, n_iter=5, init_phase=ph, out=y, workspace=ws)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            sp.griffinlim_flat(S, fb, ctx, n_iter=5, init_phase=ph, out=y, workspace=ws)
    torch.cuda.current_stream(cuda).wait_stream(s)
    off, lens = fb.out_sample_off(), fb.out_lengths()
    for _ in range(2):
        y.zero_()
        graph.replay()
        torch.cuda.synchronize(cuda)
        for o, n in zip(off, lens):                 # the <= 3 filler samples between items are never written
            assert torch.equal(y[o: o + n], eager[o: o + n])
