"""GPU parity of the SURVEY 8(f) row-1 kernels: RMS energy, spectral centroid (2048-point STFT) and
per-phoneme pooling, against the restated librosa calls of spev_real_metrics.py:370-371, :400-417, and against
plain float64 references of the same operations.

float64 framing (librosa ``center=True``): 1024 zero samples on each side, frame t at sample 256 t, periodic
Hann-2048, ``np.fft.rfft``, f_k = k sr / 2048.  Kernel results are held to per-frame error bounds built from the
float64 values, not to blanket tolerances."""
import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr
from tests import synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n", [132300, 256 * 40, 255, 4000, 70001])
def test_rms_and_centroid_vs_oracle(cuda, n):
    import spev_tts_b200 as sp
    y = synth.speechy(seed=n % 97, n=n)
    r_ref = lr.rms(y=y, hop_length=256)[0]
    c_ref = lr.spectral_centroid(y=y, sr=22050, hop_length=256)[0]
    r = sp.rms(y=y, hop_length=256)
    c = sp.spectral_centroid(y=y, sr=22050, hop_length=256)
    assert r.shape == (1, 1 + n // 256) and c.shape == (1, 1 + n // 256)
    assert np.abs(r[0] - r_ref).max() <= 2e-6 * max(1.0, r_ref.max()) + 1e-7
    # the reference uses the logs (:370, :397): compare there too
    assert np.abs(np.log(r[0] + 1e-6) - np.log(r_ref + 1e-6)).max() <= 2e-5
    assert np.abs(np.log(c[0] + 1e-8) - np.log(c_ref + 1e-8)).max() <= 2e-5
    # stats pass (:316) calls spectral_centroid with librosa's default hop 512 = every second frame
    c512 = sp.spectral_centroid(y=y, sr=22050)
    c512_ref = lr.spectral_centroid(y=y, sr=22050)[0]
    assert c512.shape == (1, 1 + n // 512)
    assert np.abs(np.log(c512[0] + 1e-8) - np.log(c512_ref + 1e-8)).max() <= 2e-5


def test_silence_and_ragged_batch(cuda):
    import spev_tts_b200 as sp
    lens = [0, 100, 2048, 5000, 256 * 33 + 1, 30000]
    rng = np.random.default_rng(3)
    ys = [(0.1 * rng.standard_normal(n)).astype(np.float32) for n in lens]
    ys[2][:] = 0.0                                             # all-zero utterance: centroid 0, rms 0
    flat = torch.from_numpy(np.concatenate(ys)).to(cuda)
    r, c, fb = sp.frame_features_flat(flat, lens)
    r, c = r.cpu().numpy(), c.cpu().numpy()
    for i, y in enumerate(ys):
        sl = slice(fb.frame_off[i], fb.frame_off[i + 1])
        r_ref = lr.rms(y=y, hop_length=256)[0] if len(y) else np.zeros(1, np.float32)
        c_ref = lr.spectral_centroid(y=y, sr=22050, hop_length=256)[0] if len(y) else np.zeros(1)
        assert np.abs(r[sl] - r_ref).max() <= 1e-6, i
        assert np.abs(c[sl] - c_ref).max() <= 2e-5 * max(1.0, np.abs(c_ref).max()), i
    assert np.all(r[fb.frame_off[2]: fb.frame_off[3]] == 0) and np.all(c[fb.frame_off[2]: fb.frame_off[3]] == 0)


def test_segment_pool_vs_reference_lines(cuda):
    import spev_tts_b200 as sp
    rng = np.random.default_rng(4)
    U = 9
    frames = rng.integers(20, 400, U)
    fo = np.concatenate([[0], np.cumsum(frames)])
    curve = rng.standard_normal(fo[-1]).astype(np.float32)
    durs, po, ref = [], [0], []
    for u in range(U):
        k = int(rng.integers(1, 40))
        d = rng.multinomial(frames[u] - k, np.ones(k) / k) + 1      # >= 1 each, sums to frames[u]
        durs.append(d); po.append(po[-1] + k)
        ref.append(lr.phoneme_pool(curve[fo[u]: fo[u + 1]], d, 0.3, 1.7, -2.5, 2.5))
    durs = np.concatenate(durs).astype(np.int64)
    got = sp.segment_pool(torch.from_numpy(curve).to(cuda), fo, torch.from_numpy(durs).to(cuda), np.array(po),
                          mu=0.3, sigma=1.7, lo=-2.5, hi=2.5).cpu().numpy()
    assert np.abs(got - np.concatenate(ref)).max() <= 2e-6
    # breathiness line: clip(1 - mean(voiced_prob), 0, 0.8) == pool with mu=1, sigma=-1
    vp = rng.random(fo[-1]).astype(np.float32)
    got = sp.segment_pool(torch.from_numpy(vp).to(cuda), fo, torch.from_numpy(durs).to(cuda), np.array(po),
                          mu=1.0, sigma=-1.0, lo=0.0, hi=0.8).cpu().numpy()
    ref = np.concatenate([np.clip(1.0 - np.array([vp[fo[u]: fo[u + 1]][s: s + d].mean() for s, d in
                          zip(np.cumsum(dd) - dd, dd)]), 0.0, 0.8) for u, dd in
                          enumerate(np.split(durs, po[1:-1]))]).astype(np.float32)
    assert np.abs(got - ref).max() <= 2e-6


def test_segment_pool_log_mode(cuda):
    """spev_segment_pool_log == pooling the per-frame log, the way :370 / :397 / :404 / :408 do it in numpy."""
    import spev_tts_b200 as sp
    rng = np.random.default_rng(9)
    frames = np.array([40, 7, 123])
    fo = np.concatenate([[0], np.cumsum(frames)])
    curve = (rng.random(fo[-1]) * 0.2).astype(np.float32)
    durs = [np.array([10, 0, 30]), np.array([7]), np.array([100, 20, 3])]
    po = np.concatenate([[0], np.cumsum([len(d) for d in durs])])
    want = []
    for u, d in enumerate(durs):
        logc = np.log(curve[fo[u]: fo[u + 1]] + 1e-6)                       # float32, like np.log(rms + 1e-6)
        cur = 0
        for dd in d:
            m = np.mean(logc[cur: cur + dd]) if dd else np.float32(np.nan)     # numpy: mean of an empty slice is NaN
            want.append(np.clip((m - (-3.0)) / 1.5, -2.5, 2.5))
            cur += dd
    got = sp.segment_pool(torch.from_numpy(curve).to(cuda), fo, torch.from_numpy(np.concatenate(durs)).to(cuda), po,
                          mu=-3.0, sigma=1.5, lo=-2.5, hi=2.5, log_eps=1e-6).cpu().numpy()
    want = np.array(want, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.abs(got[ok] - want[ok]).max() <= 2e-6          # float32 sums of up to 100 logs, sequential vs pairwise


# ---- k_frame_features against float64, frame by frame ------------------------------------------------------------

U32 = 2.0 ** -24
N_WIN = 2048
HANN64 = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N_WIN) / N_WIN)          # periodic Hann-2048
TINY32 = float(np.finfo(np.float32).tiny)
# The float32 FFT's error is modelled as a noise floor on every bin's magnitude:
#   eps = K_FFT * u * log2(2048) * ||X||_2 / sqrt(1025),   u = 2^-24.
# On a B200 (1,000 W power limit) the kernel's centroids over every signal of this file need at most K = 0.10, so
# K_FFT = 1 leaves a margin of ten.
K_FFT = 1.0


def _gamma(n):
    return n * U32 / (1 - n * U32)


def _ref_frames(y, sr, chunk=256):
    """float64 RMS and centroid of every frame of the float32 signal ``y`` and their error bounds:
    -> (rms, rms_bound, centroid, centroid_bound_fft, centroid_bound_rest), each ``[1 + len(y) // 256]``.

    RMS: the kernel sums x^2 with 64 sequential fmaf per lane and a 5-level butterfly (depth 69), scales by 1/2048
    (exact) and takes sqrtf: |dr| <= r (gamma_69 / 2 + 2u).
    Centroid c = sum f_k m_k / M, M = sum m_k: a magnitude error d_k moves it by sum (f_k - c) d_k / M.
    ``centroid_bound_fft`` is that sum for the FFT noise floor eps; ``centroid_bound_rest`` adds 2u per magnitude (fmaf + sqrtf), gamma_40 on each of the two
    float32 sums (32 terms per lane, one more on lane 0, 5 butterfly levels), the division and the product with
    sr / 2048 (exact in float32 for the rates used here)."""
    T = 1 + len(y) // 256
    yp = np.pad(y.astype(np.float64), 1024)
    f = np.arange(1025) * (sr / N_WIN)
    r, rb, c, cb_fft, cb_rest = (np.empty(T) for _ in range(5))
    for t0 in range(0, T, chunk):
        t = np.arange(t0, min(T, t0 + chunk))
        fr = yp[t[:, None] * 256 + np.arange(N_WIN)]
        r[t] = np.sqrt(np.sum(fr * fr, axis=1) / N_WIN)
        m = np.abs(np.fft.rfft(fr * HANN64, axis=1))
        M = m.sum(axis=1)
        L = np.where(M < TINY32, 1.0, M)                       # librosa.util.normalize(norm=1) keeps tiny columns
        c[t] = (m @ f) / L
        dev = np.abs(f[None, :] - c[t][:, None])
        eps = K_FFT * U32 * np.log2(N_WIN) * np.linalg.norm(m, axis=1) / np.sqrt(1025)
        cb_fft[t] = eps * dev.sum(axis=1) / L
        cb_rest[t] = 2 * U32 * (dev * m).sum(axis=1) / L + c[t] * (2 * _gamma(40) + 4 * U32)
    rb[:] = r * (_gamma(69) / 2 + 2 * U32)
    return r, rb, c, cb_fft, cb_rest


def _worst(err, bound):
    return float(np.max(np.divide(err, bound, out=np.zeros_like(err), where=bound > 0), initial=0.0))


def _check_frames(rms, cent, y, sr, what):
    """Kernel RMS / centroid of every frame of ``y`` within the float64 bounds (a silent frame: exactly 0).
    -> the float64 (rms, centroid, centroid bound)."""
    r, rb, c, cb_fft, cb_rest = _ref_frames(y, sr)
    assert rms.shape == r.shape and cent.shape == c.shape, what
    er, ec = np.abs(rms - r), np.abs(cent - c)
    cb = cb_fft + cb_rest
    assert (er <= rb).all(), f"{what}: rms err / bound {_worst(er, rb):.3g} (frame {int(np.argmax(er - rb))})"
    assert (ec <= cb).all(), f"{what}: centroid err / bound {_worst(ec, cb):.3g} (frame {int(np.argmax(ec - cb))})"
    return r, c, cb


def _pack(items, packing):
    """Flat float32 buffer holding ``items`` with NaN everywhere else (before, between and after them).
    ``aligned``: starts from ``aligned_offsets`` (+4), 16-byte cp.async path;  ``gaps``: 1-3 filler samples before
    every item and no start a multiple of 4, 4-byte path;  ``shifted``: the aligned starts on a base one element off
    (the kernel sees ``buf[1:]``), 4-byte path with every start a multiple of 4.  -> (buf, sample_off, base)."""
    from spev_tts_b200.batch import aligned_offsets
    lens = [len(y) for y in items]
    if packing == "gaps":
        off, pos = [], 0
        for i, n in enumerate(lens):
            g = 1 + i % 3
            if (pos + g) % 4 == 0:
                g = g % 3 + 1
            off.append(pos + g)
            pos += g + n
        off = np.array(off, dtype=np.int64)
    else:
        off = 4 + aligned_offsets(lens)[:-1]
    base = 1 if packing == "shifted" else 0
    buf = np.full(base + int((off + lens).max()) + 64, np.nan, dtype=np.float32)
    for o, y in zip(off, items):
        buf[base + o: base + o + len(y)] = y
    return buf, off, base


def _features(items, sr, dev, packing="aligned"):
    """One k_frame_features launch over ``items`` packed per ``_pack`` -> (rms, centroid, frame_off), numpy."""
    import spev_tts_b200 as sp
    buf, off, base = _pack(items, packing)
    samples = torch.from_numpy(buf).to(dev)[base:]
    assert (samples.data_ptr() % 16 == 0) == (packing != "shifted")
    r, c, fb = sp.frame_features_flat(samples, [len(y) for y in items], sr=sr, sample_off=off)
    return r.cpu().numpy(), c.cpu().numpy(), fb.frame_off


def _signal_families(sr):
    """speech-like, white noise, tone + -80 dB noise, speech with silent stretches (whole frames of exact zeros)"""
    rng = np.random.default_rng(sr)
    n = int(1.3 * sr)
    t = np.arange(n + 777) / sr
    tone = (0.5 * np.sin(2 * np.pi * 1234.5 * t) + 5e-5 * rng.standard_normal(len(t))).astype(np.float32)
    gappy = synth.speechy(seed=7, n=n + 3001, sr=sr)
    gappy[:5000] = 0.0
    gappy[9000:17000] = 0.0
    gappy[-4500:] = 0.0
    return {"speechy": synth.speechy(seed=sr % 89, n=n, sr=sr), "white": synth.white(seed=sr % 83, n=n - 1000, sigma=0.1),
            "tone_80dB": tone, "silences": gappy}


@pytest.mark.parametrize("sr", [16000, 22050, 24000])
def test_frame_features_vs_float64(cuda, sr):
    """Every frame of four signal families in one ragged launch against float64, at the centroid scale of each rate."""
    fam = _signal_families(sr)
    items = list(fam.values())
    rms, cent, fo = _features(items, sr, cuda)
    for i, (name, y) in enumerate(fam.items()):
        r, _, _ = _check_frames(rms[fo[i]: fo[i + 1]], cent[fo[i]: fo[i + 1]], y, sr, f"{name} @ {sr}")
        if name == "silences":
            assert (r == 0).sum() >= 20                       # the exact-zero frames were checked for exactly 0


KNOWN_TONES = (2, 3, 100, 511, 512, 513, 1021, 1022)
KNOWN_LEVELS = (1e-6, 1e-3, 1.0)


@pytest.mark.parametrize("sr", [16000, 22050, 24000])
def test_centroid_known_answers(cuda, sr):
    """Signals whose centroid is known in closed form and together reach every arm of the packed real-FFT split:
    the mirror pairs (k, 1024 - k), bin 0 with bin 1024, and bin 512 that lane 0 adds.
    A cosine on bin k has |X| at k-1, k, k+1 in the ratio 1:2:1 -> k sr / 2048; a constant -> sr / 2048 / 3; (-1)^n ->
    (2 * 1024 + 1023) / 3 * sr / 2048.  Checked on the frames whose window lies inside the signal (t = 4 .. 10)."""
    n = np.arange(N_WIN + 6 * 256)
    inside = slice(4, 11)
    # (name, signal, centroid in bins, tolerance of the float64 closed form, RMS of a window at level 1).  Rounding a
    # general tone to float32 spreads a noise floor over all bins, which moves its float64 centroid by up to 8.6e-5
    # relative (k = 2, level 1e-6); samples exact in float32 (0, +-1) keep the closed form to float64 roundoff (3.6e-12 at DC)
    cases = [(f"bin{k}", np.cos(2 * np.pi * k * n / N_WIN), k, 1e-4, np.sqrt(0.5)) for k in KNOWN_TONES if k != 512]
    cases += [("bin512", np.cos(np.pi * n / 2).round(), 512, 1e-11, np.sqrt(0.5)),
              ("dc", np.ones(len(n)), 1 / 3, 1e-11, 1.0), ("nyquist", (-1.0) ** n, (2 * 1024 + 1023) / 3, 1e-11, 1.0)]
    items, want = [], []
    for name, x, k, tol, r0 in cases:
        for level in KNOWN_LEVELS:
            level = float(np.float32(level))
            items.append((level * x).astype(np.float32))
            want.append((f"{name} x {level:.3g}", k * sr / N_WIN, tol, level * r0))
    rms, cent, fo = _features(items, sr, cuda)
    for i, (y, (what, c0, tol, r0)) in enumerate(zip(items, want)):
        r_k, c_k = rms[fo[i]: fo[i + 1]], cent[fo[i]: fo[i + 1]]
        _, c, cb = _check_frames(r_k, c_k, y, sr, what)
        assert np.abs(c[inside] / c0 - 1).max() <= tol, what
        # so the kernel's centroid does not depend on the level, and its RMS scales with it
        assert (np.abs(c_k[inside] - c0) <= tol * c0 + cb[inside]).all(), what
        assert np.abs(r_k[inside] / r0 - 1).max() <= 1e-6, what


@pytest.mark.parametrize("n", [256 * 40, 256 * 41 + 3, 511, 100000])
def test_hop512_is_every_second_frame(cuda, n):
    """rms / spectral_centroid at hop 512 are exactly every second frame of the hop-256 launch: 1 + n // 512 frames."""
    import spev_tts_b200 as sp
    y = np.stack([synth.speechy(seed=n % 31, n=n), synth.white(seed=n % 29, n=n)])
    for fn in (sp.rms, sp.spectral_centroid):
        a, b = fn(y=y, hop_length=512), fn(y=y, hop_length=256)
        assert a.shape == (2, 1, 1 + n // 512) and b.shape == (2, 1, 1 + n // 256)
        assert np.array_equal(a, b[..., ::2])


def _edge_items():
    """lengths where the window overhangs both ends of the item, and T = 31 .. 65 frames around the 32-frame tiles"""
    rng = np.random.default_rng(11)
    lens = [0, 1, 255, 1023, 1024, 2047, 2048, 2049] + [256 * (T - 1) + r for T, r in
                                                       zip((31, 32, 33, 63, 64, 65), (0, 255, 17, 100, 1, 200))]
    items = [(0.1 * rng.standard_normal(n) + 0.2 * np.sin(0.05 * np.arange(n))).astype(np.float32) for n in lens]
    items[9] = synth.speechy(seed=3, n=lens[9])
    return items


def test_staging_edges_packings_and_poisoned_filler(cuda):
    """Items of 0 .. 2049 samples and of 31 .. 65 frames, packed three ways (16-byte path, 4-byte path with ragged
    starts, 4-byte path on a base one element off) with NaN filler around every item: every frame matches float64,
    and the three packings are bit-identical."""
    items = _edge_items()
    got = {p: _features(items, 22050, cuda, p) for p in ("aligned", "gaps", "shifted")}
    rms, cent, fo = got["aligned"]
    assert list(np.diff(fo)) == [1 + len(y) // 256 for y in items]
    for p in ("gaps", "shifted"):
        assert np.array_equal(got[p][0], rms) and np.array_equal(got[p][1], cent), p
    for i, y in enumerate(items):
        _check_frames(rms[fo[i]: fo[i + 1]], cent[fo[i]: fo[i + 1]], y, 22050, f"item {i} ({len(y)} samples)")
    assert rms[0] == 0 and cent[0] == 0                            # the empty item: one all-zero frame


def test_ring_wrap_and_determinism(cuda):
    """One CTA (or three) walking all 40+ tiles wraps the 4-slot descriptor ring many times; the result is
    bit-identical to the default grid, and two launches are bit-identical."""
    import spev_tts_b200 as sp
    items = [synth.speechy(seed=s, n=40000 + 3001 * s) for s in range(8)] + _edge_items()
    buf, off, _ = _pack(items, "aligned")
    samples = torch.from_numpy(buf).to(cuda)
    lens = [len(y) for y in items]
    ctx = sp.Context.get(cuda, sr=22050)

    def run():
        r, c, fb = sp.frame_features_flat(samples, lens, sample_off=off)
        return r.cpu().numpy(), c.cpu().numpy(), fb.n_ftiles
    r0, c0, n_tiles = run()
    assert n_tiles >= 40
    r1, c1, _ = run()
    assert np.array_equal(r0, r1) and np.array_equal(c0, c1)
    try:
        for limit in (1, 3):
            from spev_tts_b200 import _lib
            _lib.check(ctx.lib.spev_set_sm_limit(ctx.handle, limit), "spev_set_sm_limit")
            r, c, _ = run()
            assert np.array_equal(r, r0) and np.array_equal(c, c0), limit
    finally:
        ctx.lib.spev_set_sm_limit(ctx.handle, 0)


# ---- the per-phoneme duration walk: spev_segment_pool(_log), spev_pitch_pool ----------------------------------------

def _pool_items(seed=12):
    """-> [(T, durations)]: phone counts 1 .. 100 (across the 32-phone carry) filling their item, an item without
    phones, one without frames, zero-length and negative durations, durations that run past T (a phone straddling T,
    phones starting at and after T, also across the carry), then enough small items (> 148 * 16 * 4 = 9472 warps)
    that warps take the grid-stride step."""
    rng = np.random.default_rng(seed)
    items = []
    for k in (1, 31, 32, 33, 64, 65, 100):
        T = int(rng.integers(k, 3 * k + 20))
        cuts = np.sort(rng.integers(0, T + 1, k - 1))
        items.append((T, np.diff(np.concatenate([[0], cuts, [T]]))))
    items += [(50, np.zeros(0)), (0, np.array([0, 3, 1])), (40, np.array([5, -3, 10, -1, 0, 25])),
              (40, np.array([10, 20, 15, 5])), (40, np.array([10, 30, 4, 2])), (1, np.array([-7, 2, 1]))]
    d = rng.integers(-2, 7, 70)
    items.append((int(np.maximum(d, 0)[:40].sum()), d))                 # past T from phone 40 on, across two carries
    for _ in range(9600):
        items.append((int(rng.integers(0, 12)), rng.integers(-1, 6, int(rng.integers(0, 4)))))
    return [(T, np.asarray(d, dtype=np.int64)) for T, d in items]


def _walk(items):
    """spev_real_metrics.py:400-417's walk: phone p covers [curr, curr + d) of its item, curr += d.  Negative durations
    count as 0 (numpy would move curr backwards); the mean covers the frames inside the item.
    -> per phone (item, first frame, end frame) with the slice already cut at T."""
    out = []
    for u, (T, durs) in enumerate(items):
        curr = 0
        for d in durs:
            d = max(int(d), 0)
            out.append((u, min(curr, T), min(curr + d, T)))
            curr += d
    return out


def _layout(items):
    fo = np.concatenate([[0], np.cumsum([T for T, _ in items])]).astype(np.int64)
    po = np.concatenate([[0], np.cumsum([len(d) for _, d in items])]).astype(np.int64)
    durs = np.concatenate([d for _, d in items]).astype(np.int64)
    return fo, po, durs


def _segment_ref(curve, log_eps, items, mu, sigma, lo, hi):
    """float64 clip((mean - mu) / sigma, lo, hi) per phone (NaN without frames) and its bound: the float32 sequential
    sum of n terms (gamma_{n+1} with the division by n), 2 ulp for every logf, and u for each of the subtraction and
    the division by sigma.  mu, sigma, lo, hi: as float32 values, the way the kernel receives them."""
    fo, _, _ = _layout(items)
    mu, sigma, lo, hi = (float(np.float32(v)) for v in (mu, sigma, lo, hi))
    if log_eps is None:
        terms, slack = curve.astype(np.float64), np.zeros(len(curve))
    else:
        v = curve + np.float32(log_eps)                                  # float32, like np.log(rms + 1e-6)
        terms = np.log(v.astype(np.float64))
        slack = 2 * np.spacing(np.abs(terms).astype(np.float32)).astype(np.float64)
    want, bound = [], []
    for u, s, e in _walk(items):
        n = e - s
        if n == 0:
            want.append(np.nan)
            bound.append(0.0)
            continue
        seg = slice(fo[u] + s, fo[u] + e)
        z = (terms[seg].mean() - mu) / sigma
        want.append(np.clip(z, lo, hi))
        bound.append((_gamma(n + 1) * np.abs(terms[seg]).sum() / n + slack[seg].mean()) / abs(sigma) + 3 * U32 * abs(z))
    return np.array(want), np.array(bound)


def _pitch_ref(states, logf, items, pm, ps, lo, hi, rough_hi):
    """float64 lines :399-414: masked mean / population std of the voiced log-f0 per phone; pitch clip(0) and rough 0
    without voiced frames.  The kernel is float64 too: bound 1 float32 ulp of the result (+1e-12 for the std)."""
    fo, _, _ = _layout(items)
    n_bins = len(logf)
    lo, hi, rough_hi = (float(np.float32(v)) for v in (lo, hi, rough_hi))
    pitch, rough = [], []
    for u, s, e in _walk(items):
        st = states[fo[u] + s: fo[u] + e]
        v = logf[st[st < n_bins]]
        pitch.append(np.clip((v.mean() - pm) / ps if v.size else 0.0, lo, hi))
        rough.append(np.clip(v.std() if v.size else 0.0, 0.0, rough_hi))
    pitch, rough = np.array(pitch), np.array(rough)
    return pitch, rough, (np.spacing(np.abs(pitch).astype(np.float32)).astype(np.float64),
                          np.spacing(rough.astype(np.float32)).astype(np.float64) + 1e-12)


def _assert_pooled(got, want, bound, what):
    assert got.shape == want.shape, what
    assert np.array_equal(np.isnan(got), np.isnan(want)), \
        f"{what}: NaN mismatch at phones {np.flatnonzero(np.isnan(got) != np.isnan(want))[:8]}"
    ok = ~np.isnan(want)
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    assert (err <= bound[ok]).all(), \
        f"{what}: err / bound {_worst(err, bound[ok]):.3g} at phone {np.flatnonzero(ok)[int(np.argmax(err - bound[ok]))]}"


SEGMENT_LINES = [(0.25, 0.5, -0.5, 0.75), (1.0, -1.0, 0.0, 0.8)]          # (mu, sigma, lo, hi); sigma = -1: breathiness


@pytest.mark.parametrize("entry", ["spev_segment_pool", "spev_segment_pool_log", "spev_pitch_pool"])
def test_duration_walk_vs_float64(cuda, entry):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    from spev_tts_b200.batch import stream_ptr
    items = _pool_items()
    fo, po, durs = _layout(items)
    assert len(items) > 148 * 16 * 4
    rng = np.random.default_rng(13)
    d_durs = torch.from_numpy(durs).to(cuda)
    if entry != "spev_pitch_pool":
        log_eps = 1e-6 if entry == "spev_segment_pool_log" else None
        curve = (rng.random(fo[-1]) if log_eps else rng.standard_normal(fo[-1])).astype(np.float32)
        curve[::7] = 0.0
        lines = SEGMENT_LINES if log_eps is None else [(-5.0, 1.5, -2.5, 2.5), (-2.0, -1.0, -1.0, 1.0)]
        for mu, sigma, lo, hi in lines:
            got = sp.segment_pool(torch.from_numpy(curve).to(cuda), fo, d_durs, po, mu=mu, sigma=sigma, lo=lo, hi=hi,
                                  log_eps=log_eps).cpu().numpy()
            want, bound = _segment_ref(curve, log_eps, items, mu, sigma, lo, hi)
            _assert_pooled(got, want, bound, f"{entry} mu={mu} sigma={sigma}")
            assert (got == np.float32(lo)).any() and (got == np.float32(hi)).any()     # both clip ends reached
        return
    from spev_tts_b200.pitch import PyinContext
    p = PyinContext.get(cuda)
    logf = np.log(p.host_tables()[1] + 1e-8)
    states = np.where(rng.random(fo[-1]) < 0.6, rng.integers(0, p.n_bins, fo[-1]),
                      p.n_bins + rng.integers(0, p.n_bins, fo[-1])).astype(np.int32)
    pm, ps, lo, hi, rough_hi = 5.2, 0.31, -2.5, 2.5, 0.4
    pitch = torch.full((len(durs),), float("nan"), dtype=torch.float32, device=cuda)
    rough = torch.full_like(pitch, float("nan"))
    d_fo, d_po = torch.from_numpy(fo).to(cuda), torch.from_numpy(po).to(cuda)
    _lib.check(p.lib.spev_pitch_pool(p.handle, torch.from_numpy(states).to(cuda).data_ptr(), d_fo.data_ptr(),
                                     d_durs.data_ptr(), d_po.data_ptr(), len(items), pm, ps, lo, hi, rough_hi,
                                     pitch.data_ptr(), rough.data_ptr(), stream_ptr(cuda)), "spev_pitch_pool")
    want_p, want_r, (bp, br) = _pitch_ref(states, logf, items, pm, ps, lo, hi, rough_hi)
    got_p, got_r = pitch.cpu().numpy(), rough.cpu().numpy()
    _assert_pooled(got_p, want_p, bp, "pitch")
    _assert_pooled(got_r, want_r, br, "rough")
    assert (got_p == lo).any() and (got_p == hi).any() and (got_r == np.float32(rough_hi)).any()
