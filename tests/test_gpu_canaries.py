"""Out-of-bounds write detection without compute-sanitizer (closed on this pool): every output
buffer handed to the C ABI sits between canary regions that must survive the launch, for odd and
ragged sizes."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
CANARY = 1.2345678e30
PAD = 4096


class Guarded:
    """float32 buffer of n elements between two PAD-element canary regions (16-byte aligned payload)."""

    def __init__(self, n, dev, dtype=torch.float32, words_per_elem=1):
        self.n = n * words_per_elem
        self.raw = torch.full((self.n + 2 * PAD,), CANARY, dtype=torch.float32, device=dev)
        self.view = self.raw[PAD: PAD + self.n]
        self.view.fill_(float("nan"))

    def ptr(self):
        return self.view.data_ptr()

    def check(self, what):
        head, tail = self.raw[:PAD], self.raw[PAD + self.n:]
        assert bool((head == CANARY).all()) and bool((tail == CANARY).all()), f"{what}: canary overwritten"
        return self.view


@pytest.mark.parametrize("lens", [[1], [255, 256, 257], [8191, 8192, 8193, 5], [33 * 256 + 5, 0, 70001]])
def test_forward_kernels_stay_in_bounds(cuda, lens):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    rng = np.random.default_rng(len(lens))
    flat = torch.from_numpy(np.concatenate([(0.1 * rng.standard_normal(n)).astype(np.float32) for n in lens])).to(cuda) \
        if sum(lens) else torch.zeros(1, device=cuda)
    ctx = sp.Context.get(cuda)
    fb = sp.make_batch(ctx, n_samples=lens)
    st = torch.cuda.current_stream(cuda).cuda_stream
    F = fb.n_frames
    out = Guarded(F * 80, cuda)
    _lib.check(ctx.lib.spev_logmel(ctx.handle, fb.desc, flat.data_ptr(), out.ptr(), 1, 1e-5, -10.0, 2.0, st))
    v = out.check("spev_logmel")
    assert bool(torch.isfinite(v).all())                      # every element written
    pw = Guarded(F * 520, cuda)
    _lib.check(ctx.lib.spev_stft_power(ctx.handle, fb.desc, flat.data_ptr(), pw.ptr(), st))
    assert bool(torch.isfinite(pw.check("spev_stft_power")).all())
    mo = Guarded(F * 80, cuda)
    _lib.check(ctx.lib.spev_mel_project(ctx.handle, pw.ptr(), F, mo.ptr(), 1, 1e-5, -10.0, 2.0, st))
    assert bool(torch.isfinite(mo.check("spev_mel_project")).all())
    r, c = Guarded(F, cuda), Guarded(F, cuda)
    _lib.check(ctx.lib.spev_frame_features(ctx.handle, fb.desc, flat.data_ptr(), r.ptr(), c.ptr(), st))
    assert bool(torch.isfinite(r.check("rms")).all()) and bool(torch.isfinite(c.check("centroid")).all())


@pytest.mark.parametrize("frames", [[1], [2, 3], [29, 30, 31, 32, 33], [100, 1, 64], [0, 5], [3, 0, 0, 40]])
def test_griffinlim_kernels_stay_in_bounds(cuda, frames):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    fb = sp.make_batch(ctx, n_frames=frames, with_chunks=True)
    st = torch.cuda.current_stream(cuda).cuda_stream
    F = fb.n_frames
    g = torch.Generator(device=cuda).manual_seed(1)
    lm = (-4 + 2 * torch.randn(F, 80, generator=g, device=cuda)).clamp(-10, 2)
    S = Guarded(F * 520, cuda)
    for tc in (1, 0):                                           # tcgen05 and FFMA variants
        ctx.set_tensor_core(bool(tc))
        _lib.check(ctx.lib.spev_mel_to_mag(ctx.handle, fb.desc, lm.data_ptr(), 0, 1, S.ptr(), 520, st))
        Sv = S.check("spev_mel_to_mag")
        assert bool(torch.isfinite(Sv.view(F, 520)[:, :513]).all())
    ctx.set_tensor_core(True)
    y = Guarded(max(fb.n_out_samples, 1), cuda)
    ws_bytes = ctx.lib.spev_griffinlim_workspace_bytes(F)
    ws = Guarded((ws_bytes + 3) // 4, cuda)
    _lib.check(ctx.lib.spev_griffinlim(ctx.handle, fb.desc, S.ptr(), 520, None, 7, 3, 0.99, y.ptr(), ws.ptr(), ws_bytes, st))
    yv = y.check("spev_griffinlim y")
    ws.check("spev_griffinlim workspace")
    if fb.n_out_samples:
        assert bool(torch.isfinite(yv[: fb.n_out_samples]).all())


def test_lr_and_bucketize_stay_in_bounds(cuda):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    lib = sp.load()
    st = torch.cuda.current_stream(cuda).cuda_stream
    B, T, H = 5, 37, 13
    g = torch.Generator(device=cuda).manual_seed(2)
    x = torch.randn(B, T, H, generator=g, device=cuda)
    d = torch.randint(0, 9, (B, T), generator=g, device=cuda)
    p = sp.plan(d)
    out = Guarded(B * p.max_len * H, cuda)
    fo = Guarded(5 * B * p.max_len, cuda)
    feats = torch.randn(5, B, T, generator=g, device=cuda)
    _lib.check(lib.spev_lr_expand_fused(x.data_ptr(), H * 4, feats.data_ptr(), 5, None, None, p.cumsum.data_ptr(), B, T,
                                        out.ptr(), fo.ptr(), p.max_len, st))
    assert bool(torch.isfinite(out.check("lr out")).all()) and bool(torch.isfinite(fo.check("lr feats")).all())
    n, Hh = 77, 10
    v = torch.randn(n, generator=g, device=cuda)
    bnd = torch.linspace(-3, 3, 255, device=cuda)
    tab = torch.randn(256, Hh, generator=g, device=cuda)
    emb = Guarded(n * Hh, cuda)
    _lib.check(lib.spev_bucketize_embed(v.data_ptr(), n, bnd.data_ptr(), 255, 0, tab.data_ptr(), Hh, None, emb.ptr(), 0, st))
    assert bool(torch.isfinite(emb.check("bucketize")).all())


@pytest.mark.parametrize("lens", [[1], [255, 256, 257], [8191, 8192, 8193, 5], [33 * 256 + 5, 0, 70001]])
def test_pyin_kernels_stay_in_bounds(cuda, lens):
    """Every pYIN stage writes all of its output and nothing else (guarded buffers, ragged sizes)."""
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib
    from spev_tts_b200.pitch import PyinContext
    from tests import synth
    ys = [synth.voiced_unvoiced(seed=3 + i, n=max(n, 1))[0][:n] for i, n in enumerate(lens)]
    flat = torch.from_numpy(np.concatenate(ys)).to(cuda) if sum(lens) else torch.zeros(1, device=cuda)
    ctx = sp.Context.get(cuda)
    p = PyinContext.get(cuda)
    fb = sp.make_batch(ctx, n_samples=lens)
    st = torch.cuda.current_stream(cuda).cuda_stream
    F = fb.n_frames
    yin = Guarded(F * p.n_lags, cuda)
    _lib.check(p.lib.spev_pyin_cmnd(p.handle, fb.desc, flat.data_ptr(), yin.ptr(), st))
    assert bool(torch.isfinite(yin.check("spev_pyin_cmnd")).all())
    lo, lu, vp = Guarded(F * p.n_bins, cuda), Guarded(F, cuda), Guarded(F, cuda)
    _lib.check(p.lib.spev_pyin_observe(p.handle, yin.ptr(), F, lo.ptr(), lu.ptr(), vp.ptr(), st))
    for g, name in ((lo, "logobs"), (lu, "log_unvoiced"), (vp, "voiced_prob")):
        assert bool(torch.isfinite(g.check(name)).all())
    nbytes = p.lib.spev_pyin_decode_workspace_bytes(p.handle, F)
    ws = Guarded((nbytes + 3) // 4, cuda)
    states, f0, flag = Guarded(F, cuda), Guarded(F, cuda), Guarded((F + 3) // 4, cuda)
    fo = torch.from_numpy(fb.frame_off).to(cuda)
    _lib.check(p.lib.spev_pyin_decode(p.handle, lo.ptr(), lu.ptr(), fo.data_ptr(), len(lens), F, states.ptr(), f0.ptr(),
                                      flag.ptr(), ws.ptr(), nbytes, st))
    ws.check("viterbi workspace")
    s = states.check("states").view(torch.int32)
    assert bool(((s >= 0) & (s < 2 * p.n_bins)).all())
    f0v = f0.check("f0")
    voiced = flag.check("voiced_flag").view(torch.uint8)[:F]
    assert bool(((voiced == 1) == (s < p.n_bins)).all()) and bool((torch.isnan(f0v) == (voiced == 0)).all())
    # pooling over arbitrary phone cuts
    durs = torch.tensor([max(1, int(t) // 2) for t in fb.frames for _ in range(2)], dtype=torch.int64, device=cuda)
    po = torch.arange(0, 2 * len(lens) + 1, 2, dtype=torch.int64, device=cuda)
    pitch, rough = Guarded(2 * len(lens), cuda), Guarded(2 * len(lens), cuda)
    _lib.check(p.lib.spev_pitch_pool(p.handle, states.ptr(), fo.data_ptr(), durs.data_ptr(), po.data_ptr(), len(lens),
                                     5.2, 0.3, -2.5, 2.5, 1.5, pitch.ptr(), rough.ptr(), st))
    assert bool(torch.isfinite(pitch.check("pitch")).all()) and bool(torch.isfinite(rough.check("rough")).all())


@pytest.mark.parametrize("B,T,H,n_feat", [(1, 1, 1, 0), (3, 7, 5, 2), (4, 33, 256, 5), (2, 50, 12, 5)])
def test_backward_kernels_stay_in_bounds(cuda, B, T, H, n_feat):
    """spev_lr_expand_backward / spev_variance_fuse_backward: every gradient buffer fully written, nothing around it."""
    from spev_tts_b200 import _lib
    from spev_tts_b200.length_regulator import plan
    lib = _lib.load()
    rng = np.random.default_rng(B * 100 + T)
    dur = torch.from_numpy(rng.integers(0, 6, (B, T))).to(cuda)
    p = plan(dur)
    st = torch.cuda.current_stream(cuda).cuda_stream
    go = torch.randn(B, p.max_len, H, device=cuda)
    gx = Guarded(B * T * H, cuda)
    gfo = torch.randn(max(n_feat, 1), B, p.max_len, device=cuda)
    feats = torch.randn(max(n_feat, 1), B, T, device=cuda) * 2
    gf = Guarded(max(n_feat, 1) * B * T, cuda)
    lo = (C.c_float * 5)(-3, -3, 0, 0, -3); hi = (C.c_float * 5)(3, 3, 1, 2, 3)
    _lib.check(lib.spev_lr_expand_backward(go.data_ptr(), 0, H, gfo.data_ptr() if n_feat else None, n_feat,
                                           feats.data_ptr() if n_feat else None, C.cast(lo, C.c_void_p) if n_feat else None,
                                           C.cast(hi, C.c_void_p) if n_feat else None, p.cumsum.data_ptr(), B, T, p.max_len,
                                           gx.ptr(), gf.ptr() if n_feat else None, st))
    assert bool(torch.isfinite(gx.check("grad_x")).all())
    if n_feat:
        assert bool(torch.isfinite(gf.check("grad_feats")[: n_feat * B * T]).all())
    if n_feat:                                                   # fused variance adaptor backward
        w = torch.randn(n_feat, H, 3, device=cuda)
        gx2, gf2 = Guarded(B * T * H, cuda), Guarded(n_feat * B * T, cuda)
        gw, gb = Guarded(n_feat * H * 3, cuda), Guarded(n_feat * H, cuda)
        nws = lib.spev_variance_fuse_backward_workspace_bytes(n_feat, B, H, p.max_len)
        ws = Guarded((nws + 3) // 4, cuda)
        _lib.check(lib.spev_variance_fuse_backward(go.data_ptr(), feats.data_ptr(), n_feat, C.cast(lo, C.c_void_p),
                                                   C.cast(hi, C.c_void_p), w.data_ptr(), p.cumsum.data_ptr(), B, T, H, p.max_len,
                                                   gx2.ptr(), gf2.ptr(), gw.ptr(), gb.ptr(), ws.ptr(), nws, st))
        ws.check("variance backward workspace")
        for g, name in ((gx2, "grad_x"), (gf2, "grad_feats"), (gw, "grad_w"), (gb, "grad_b")):
            assert bool(torch.isfinite(g.check(name)).all()), name
        assert torch.equal(gx2.view, gx.view)                    # same segment sums as the plain expand backward


def test_copy_segments_and_nnls_objective_stay_in_bounds(cuda):
    import spev_tts_b200 as sp
    from spev_tts_b200 import _lib, cache
    rng = np.random.default_rng(3)
    rows = rng.integers(0, 70, 23)                               # ragged runs of 7-float rows, some empty
    src = torch.randn(int(rows.sum()), 7, device=cuda)
    so = np.concatenate([[0], np.cumsum(rows)])[:-1]
    perm = rng.permutation(len(rows))
    do = np.zeros(len(rows), np.int64)
    do[perm] = np.concatenate([[0], np.cumsum(rows[perm])])[:-1]
    g = Guarded(src.numel(), cuda)
    dst = g.view.view(-1, 7)
    cache.copy_segments(src, dst, so, do, rows)
    out = g.check("spev_copy_segments").view(-1, 7)
    for i in range(len(rows)):
        assert torch.equal(out[do[i]: do[i] + rows[i]], src[so[i]: so[i] + rows[i]])
    # NNLS objective: per-column outputs and the gradient block
    ctx = sp.Context.get(cuda, fmin=0.0, fmax=8000.0)
    L, T, t0, tb = 3, 19, 4, 11
    mel = torch.rand(L * T, 80, device=cuda)
    x = torch.rand(L, 513, tb, device=cuda, dtype=torch.float64)
    val, pgm = Guarded(L * tb, cuda, words_per_elem=2), Guarded(L * tb, cuda, words_per_elem=2)
    grad = Guarded(L * 513 * tb, cuda, words_per_elem=2)
    _lib.check(ctx.lib.spev_nnls_objective(ctx.handle, x.data_ptr(), 0, 0, mel.data_ptr(), 0, L, T, t0, tb, 0, val.ptr(), grad.ptr(),
                                           pgm.ptr(), torch.cuda.current_stream(cuda).cuda_stream))
    for gd, name in ((val, "value_parts"), (pgm, "pg_max"), (grad, "grad")):
        v = gd.check(name).view(torch.float64)
        assert bool(torch.isfinite(v).all()), name
    # and the numbers: f = 0.5/size ||A x - B||^2, g = A^T (A x - B) / size, in float64
    A = torch.from_numpy(ctx.mel_basis()).to(cuda).double()
    Bm = mel.view(L, T, 80)[:, t0: t0 + tb].permute(0, 2, 1).double()          # [L, 80, tb]
    r = torch.einsum("mf,lft->lmt", A, x) - Bm
    size = L * 80 * tb
    assert abs(float(val.view.view(torch.float64).sum()) - float(0.5 / size * (r ** 2).sum())) <= 1e-12
    gref = torch.einsum("mf,lmt->lft", A, r) / size
    assert float((grad.view.view(torch.float64).view(L, 513, tb) - gref).abs().max()) <= 1e-14
