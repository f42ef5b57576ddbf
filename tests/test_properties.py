"""Property tests (hypothesis) of the host logic and the oracle: tile planning covers every
frame / chunk exactly once; the vectorised LengthRegulator restatement equals a literal
transcription of the reference loop for arbitrary durations."""
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import librosa_restated as lr


@pytest.fixture(scope="module")
def planners():
    """The tile planners are the library's (spev_plan_*_tiles): build it first."""
    from spev_tts_b200 import batch, build
    build.build()
    return batch


def literal_lr(x, dur):
    """Line-by-line transcription of spev_real_metrics.py:122-146 in numpy (slow, obvious)."""
    out, lens = [], []
    for b in range(x.shape[0]):
        rows = []
        for t in range(x.shape[1]):
            d = dur[b, t].item()
            if not np.isfinite(d) or d < 0 or d > 1000:
                d = 0
            n = int(d)
            if n > 0:
                rows.append(np.repeat(x[b, t:t + 1], n, axis=0))
        if not rows:
            out.append(np.zeros((1, x.shape[2]), x.dtype)); lens.append(1)
        else:
            out.append(np.concatenate(rows)); lens.append(out[-1].shape[0])
    m = max(lens)
    return np.stack([np.pad(o, ((0, m - o.shape[0]), (0, 0))) for o in out]), np.array(lens, np.int64)


@settings(max_examples=60, deadline=None)
@given(st.integers(1, 4), st.integers(1, 12), st.integers(1, 5), st.integers(0, 2 ** 31 - 1), st.booleans())
def test_lr_restatement_equals_literal_loop(B, T, H, seed, as_float):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, T, H)).astype(np.float32)
    d = rng.integers(-2, 7, (B, T)).astype(np.float64)
    if as_float:
        d = d + rng.choice([0.0, 0.3, 0.999], (B, T))
        d[rng.random((B, T)) < 0.1] = np.nan
        d[rng.random((B, T)) < 0.05] = 1000.5
    else:
        d = d.astype(np.int64)
    o, l = lr.length_regulator(x, d)
    ro, rl = literal_lr(x, d)
    assert np.array_equal(o, ro) and np.array_equal(l, rl)


@settings(max_examples=80, deadline=None)
@given(st.lists(st.integers(0, 40000), min_size=1, max_size=30))
def test_c_planned_tiles_cover_everything_once_in_order(planners, n_samples):
    B = planners
    ns = np.asarray(n_samples, dtype=np.int64)
    frames = 1 + ns // 256
    starts = np.concatenate([[0], np.cumsum((ns + 3) // 4 * 4)])[:-1]
    ft = B.plan_frame_tiles(frames, starts, ns)
    fo = np.concatenate([[0], np.cumsum(frames)])
    # item order, 32-frame steps within an item
    assert np.array_equal(ft["item"], np.repeat(np.arange(len(frames)), (frames + 31) // 32))
    assert (np.diff(ft["row0"]) > 0).all()
    covered = np.zeros(fo[-1], dtype=np.int32)
    for t in ft:
        assert 1 <= t["n"] <= 32 and t["T"] == frames[t["item"]] and t["t0"] % 32 == 0
        assert t["row0"] == fo[t["item"]] + t["t0"]
        assert t["src0"] == starts[t["item"]] + 256 * t["t0"] - 512
        assert t["lo"] == starts[t["item"]] and t["hi"] == t["lo"] + ns[t["item"]]
        covered[t["row0"]: t["row0"] + t["n"]] += 1
    assert np.all(covered == 1)
    # the default ISTFT output layout: (T-1)*256 samples per item, back to back
    off, L = B.out_layout(frames)
    yo = (fo - np.arange(len(fo))) * 256
    assert np.array_equal(off, yo[:-1]) and np.array_equal(L, np.diff(yo))
    ct = B.plan_chunk_tiles(frames, out_off=off, out_len=L)
    cov = np.zeros(yo[-1] // 256, dtype=np.int32)
    for t in ct:
        assert 1 <= t["n"] <= 29 and t["t0"] % 29 == 0
        assert t["lo"] == yo[t["item"]] and t["hi"] == yo[t["item"] + 1] and t["T"] == frames[t["item"]]
        assert t["src0"] == yo[t["item"]] + 256 * t["t0"] and t["row0"] == fo[t["item"]] + t["t0"] - 1
        cov[t["src0"] // 256: t["src0"] // 256 + t["n"]] += 1
    assert np.all(cov == 1)
    # full tiles first, then the partial ones; each group in item order
    full = ct["n"] == 29
    assert not (full[1:] & ~full[:-1]).any()
    for group in (ct[full], ct[~full]):
        assert (np.lexsort((group["t0"], group["item"])) == np.arange(len(group))).all()
