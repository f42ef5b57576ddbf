"""The mel -> linear inversion, kernel by kernel, against float64: the NNLS objective (``spev_nnls_objective``, all four
device paths), the float32 screening pass and the decisions ``nnls_refine`` takes from it, and the warm start
``spev_mel_to_mag`` in both input layouts.

Reference for one column ``(l, t)`` (librosa.util.nnls's objective, scipy's ``projgr`` for the bound ``x >= 0``):
    r = A x - B,   g = A^T r / size,   value = 0.5 |r|^2 / size,   pg = max_k (g_k < 0 ? -g_k : min(x_k, g_k))
with ``size = L * n_mels * (size_cols or tb)``, all in float64.  Kernel results are held to an error bound built from
the magnitudes that enter each sum, not to a blanket tolerance."""
import functools

import numpy as np
import pytest
import torch

from oracle import librosa_restated as lr
from tests import synth

pytestmark = pytest.mark.gpu

EPS64 = float(np.finfo(np.float64).eps)
EPS32 = float(np.finfo(np.float32).eps)
PGTOL = 1e-5                    # scipy.optimize.fmin_l_bfgs_b's default, librosa.util.nnls keeps it
NB = 513

# (name, x_mode, gradient buffer, unit roundoff of the arithmetic)
PATHS = [("f64", 0, True, EPS64), ("f64_rows", 1, True, EPS64), ("f32_dense", 2, True, EPS32), ("f32_banded", 2, False, EPS32)]

# Measured on a B200 (1,000 W power limit):
# largest relative error of the float32 screen's pg_max against float64 over the screening inputs below: 9.3e-6
# (banded kernel, log-mel input, scale 1e2), four orders of magnitude inside the +-10 % re-screen band of nnls_refine
SCREEN_REL = 5e-5
# largest relative difference between the float64 pg of the product's warm start (3xTF32 pinv, x0 = (sqrt x)^2) and
# that of the oracle's float32 warm start, per librosa block: 8.4e-6.  Decisions may differ only for blocks this close
# to pgtol; none of the cases below comes that close, and no decision differs
DECISION_BAND = 1e-4


def _st(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _ctx(cuda, n_mels=80, fmin=0.0, fmax=8000.0):
    import spev_tts_b200 as sp
    return sp.Context.get(cuda, sr=22050, n_mels=n_mels, fmin=fmin, fmax=fmax)


def _nnz(A):
    """non-zeros of the longest band plus those of the most covered bin: the length of the longest sum a kernel forms"""
    nz = A != 0
    return int(nz.sum(1).max()) + int(nz.sum(0).max())


@functools.lru_cache(maxsize=None)
def _power():
    """|STFT|^2 of 601 frames of harmonic speech-like signal: [513, 601] float64"""
    y = synth.speechy(seed=21, n=600 * 256)
    return np.abs(lr.stft(y, n_fft=1024, hop_length=256)).astype(np.float64) ** 2


def _objective(ctx, x, x_mode, ld_x, mel, is_log, L, T, t0, tb, size_cols=0, want_grad=False):
    """One spev_nnls_objective launch -> (value_parts [L*tb], pg_max [L*tb], grad [L*tb, 513] or None), numpy.
    Outputs start as NaN so an unwritten column shows."""
    from spev_tts_b200 import _lib
    dev = mel.device
    n = L * tb
    val = torch.full((n,), float("nan"), dtype=torch.float64, device=dev)
    pg = torch.full((n,), float("nan"), dtype=torch.float64, device=dev)
    grad = torch.full((L, NB, tb), float("nan"), dtype=torch.float64, device=dev) if want_grad else None
    _lib.check(ctx.lib.spev_nnls_objective(ctx.handle, x.data_ptr(), x_mode, ld_x, mel.data_ptr(), int(is_log), L, T, t0, tb,
                                           size_cols, val.data_ptr(), grad.data_ptr() if want_grad else None, pg.data_ptr(),
                                           _st(dev)), "spev_nnls_objective")
    g = grad.cpu().numpy().transpose(0, 2, 1).reshape(n, NB) if want_grad else None
    return val.cpu().numpy(), pg.cpu().numpy(), g


def _expf_ulps(lm):
    """2 float32 ulp of exp(lm): CUDA's expf is within 2 ulp of the exact value (the reference takes exp in float64)"""
    return 2.0 * np.spacing(np.exp(lm.astype(np.float32))).astype(np.float64)


def _reference(A, X, B, dB, inv_size, eps, nnz):
    """float64 value, g, pg per column (X [C, 513], B [C, n_mels]) and bounds on what a kernel working in unit roundoff
    ``eps`` may differ by: every r_m is off by at most gamma (sum_j |A_mj| x_j + |B_m|) + dB_m (dB: the uncertainty of
    B itself, expf), every g_k by inv_size * sum_m |A_mk| times that, pg by the largest of those (both arms of projgr
    are 1-Lipschitz in g) plus the rounding of x."""
    gamma = (64 + nnz) * eps
    absA = np.abs(A)
    r = X @ A.T - B
    g = (r @ A) * inv_size
    value = 0.5 * inv_size * np.einsum("cm,cm->c", r, r)
    pg = np.where(g < 0, -g, np.minimum(X, g)).max(axis=1, initial=0.0)
    e = gamma * (X @ absA.T + np.abs(B)) + dB
    g_tol = (e @ absA) * inv_size
    v_tol = inv_size * ((np.abs(r) + e) * e).sum(1) + gamma * value
    pg_tol = g_tol.max(axis=1, initial=0.0) + eps * X.max(axis=1, initial=0.0)
    return value, g, pg, v_tol, g_tol, pg_tol


class Problem:
    """One block [t0, t0+tb) of L stacked items of T columns: the warm-start rows S [L*T, ld_x] (float32) and mel rows
    [L*T, n_mels] on the device with NaN everywhere outside the block (other items' rows, columns 513..ld_x-1), the
    same x as float64 [L, 513, tb] (x_mode 0), and the float64 columns the reference takes."""

    def __init__(self, ctx, L, T, t0, tb, ld_x, is_log, seed, scale=1.0, S=None, mel=None):
        dev = torch.device("cuda", ctx.device)
        self.L, self.T, self.t0, self.tb, self.ld_x, self.is_log = L, T, t0, tb, ld_x, int(is_log)
        A = ctx.mel_basis()
        self.A = A.astype(np.float64)
        n_mels = A.shape[0]
        rng = np.random.default_rng(seed)
        if mel is None:                                        # mel power of speech-like spectra, one gain per item
            P = _power()
            cols = (np.arange(L)[:, None] * 37 + t0 + np.arange(tb)[None, :]) % P.shape[1]
            gain = scale * np.exp(rng.standard_normal(L))[:, None, None]
            M = (np.einsum("mf,flt->ltm", self.A, P[:, cols]) * gain).astype(np.float32)      # [L, tb, n_mels]
            mel = np.log(np.maximum(M, 1e-30)).astype(np.float32) if is_log else M
        if S is None:                                          # pinv warm start, jittered so the residual is not tiny
            Bm = np.exp(mel) if is_log else mel
            z = np.einsum("fm,ltm->ltf", ctx.mel_pinv().astype(np.float64), Bm.astype(np.float64))
            S = (np.sqrt(np.maximum(z, 0)) * np.abs(1 + 0.1 * rng.standard_normal(z.shape))).astype(np.float32)
        self.mel_blk, self.S_blk = mel, S                      # [L, tb, n_mels], [L, tb, 513]
        S_buf = np.full((L, T, ld_x), np.nan, np.float32)
        S_buf[:, t0: t0 + tb, :NB] = S
        mel_buf = np.full((L, T, n_mels), np.nan, np.float32)
        mel_buf[:, t0: t0 + tb] = mel
        self.S = torch.from_numpy(S_buf.reshape(L * T, ld_x)).to(dev)
        self.mel = torch.from_numpy(mel_buf.reshape(L * T, n_mels)).to(dev)
        self.X = S.reshape(L * tb, NB).astype(np.float64) ** 2                              # exact in float64
        self.x0 = torch.from_numpy(np.ascontiguousarray(self.X.reshape(L, tb, NB).transpose(0, 2, 1))).to(dev)
        self.B = (np.exp(mel.astype(np.float64)) if is_log else mel.astype(np.float64)).reshape(L * tb, n_mels)
        self.dB = _expf_ulps(mel).reshape(L * tb, n_mels) if is_log else np.zeros_like(self.B)

    def run(self, ctx, x_mode, want_grad, size_cols=0, t0=None, tb=None):
        t0 = self.t0 if t0 is None else t0
        tb = self.tb if tb is None else tb
        if x_mode == 0:
            x = self.x0[:, :, t0 - self.t0: t0 - self.t0 + tb].contiguous()
            return _objective(ctx, x, 0, 0, self.mel, self.is_log, self.L, self.T, t0, tb, size_cols, want_grad)
        return _objective(ctx, self.S, x_mode, self.ld_x, self.mel, self.is_log, self.L, self.T, t0, tb, size_cols, want_grad)

    def reference(self, eps, size_cols=0):
        inv_size = 1.0 / (self.L * self.A.shape[0] * (size_cols or self.tb))
        return _reference(self.A, self.X, self.B, self.dB, inv_size, eps, _nnz(self.A))


def _check_against_reference(ctx, prob, path):
    name, x_mode, want_grad, eps = path
    val, pg, g = prob.run(ctx, x_mode, want_grad)
    assert np.isfinite(val).all() and np.isfinite(pg).all(), f"{name}: a column was not written (or read NaN)"
    value_r, g_r, pg_r, v_tol, g_tol, pg_tol = prob.reference(eps)
    assert (np.abs(val - value_r) <= v_tol).all(), (name, float(np.max(np.abs(val - value_r) / np.maximum(v_tol, 1e-300))))
    assert (np.abs(pg - pg_r) <= pg_tol).all(), (name, float(np.max(np.abs(pg - pg_r) / np.maximum(pg_tol, 1e-300))))
    if want_grad:
        assert np.isfinite(g).all(), name
        assert (np.abs(g - g_r) <= g_tol).all(), (name, float(np.max(np.abs(g - g_r) / np.maximum(g_tol, 1e-300))))
    again = prob.run(ctx, x_mode, want_grad)                                               # determinism
    assert again[0].tobytes() == val.tobytes() and again[1].tobytes() == pg.tobytes(), f"{name}: not deterministic"
    if want_grad:
        assert again[2].tobytes() == g.tobytes(), f"{name}: gradient not deterministic"
    return val, pg


# n_mels from 4 to 256; (40, 300, 4000) leaves 341 bins no band covers, (256, 0, 4000) has 18 empty Slaney filters too
BASES = [(4, 0.0, None), (40, 300.0, 4000.0), (80, 0.0, 8000.0), (128, 50.0, None), (160, 0.0, 11025.0),
         (256, 0.0, 4000.0), (256, 0.0, None)]
# (L, T, t0, tb, ld_x): single columns, t0 > 0, tb = T, remainder-sized and long blocks; ld_x 513, 520 and 1000
SHAPES = [(1, 1, 0, 1, 513), (3, 2, 1, 1, 520), (3, 51, 7, 40, 1000), (16, 120, 0, 120, 520), (1, 820, 0, 820, 513),
          (16, 51, 50, 1, 1000), (3, 820, 17, 800, 520)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "L%d_T%d_t0%d_tb%d_ld%d" % s)
@pytest.mark.parametrize("basis", BASES, ids=lambda b: "m%d_%g_%s" % (b[0], b[1], b[2]))
def test_objective_paths_match_float64(cuda, basis, shape):
    """value_parts, grad and pg_max of all four device paths against the float64 reference within the error bound,
    reading nothing outside the block (NaN there), and bit-identical from one call to the next.  The float64 re-screen
    (x_mode 1, no gradient: nnls_refine's call) equals the same launch with a gradient buffer."""
    n_mels, fmin, fmax = basis
    L, T, t0, tb, ld_x = shape
    ctx = _ctx(cuda, n_mels, fmin, fmax)
    is_log = (SHAPES.index(shape) + BASES.index(basis)) % 2
    prob = Problem(ctx, L, T, t0, tb, ld_x, is_log, seed=7 * n_mels + T)
    out = {p[0]: _check_against_reference(ctx, prob, p) for p in PATHS}
    v1, p1, _ = prob.run(ctx, 1, False)
    assert v1.tobytes() == out["f64_rows"][0].tobytes() and p1.tobytes() == out["f64_rows"][1].tobytes()


def test_basis_tables_cover_empty_bands_and_uncovered_bins(cuda):
    """The shapes above do reach the banded kernel's degenerate table entries: zero-count bands and (0, -1) bins."""
    for n_mels, fmin, fmax, band, bins in ((256, 0.0, 4000.0, True, True), (40, 300.0, 4000.0, False, True)):
        nz = _ctx(cuda, n_mels, fmin, fmax).mel_basis() != 0
        assert bool((nz.sum(1) == 0).any()) == band and bool((nz.sum(0) == 0).any()) == bins


@pytest.mark.parametrize("x_mode,want_grad", [(0, True), (1, False), (1, True), (2, True), (2, False)])
def test_size_cols_launch_equals_per_block_launches(cuda, x_mode, want_grad):
    """nnls_refine screens all of librosa's equal blocks in one launch with size_cols = one block: every column's
    value_parts and pg_max (and gradient) are bit-identical to launching each block on its own."""
    ctx = _ctx(cuda)
    L, n, k, t0 = 16, 51, 3, 2                                   # b = 16: librosa's blocks hold 51 columns
    T = t0 + n * k + 5
    prob = Problem(ctx, L, T, t0, n * k, 520, 1, seed=11)
    val, pg, g = prob.run(ctx, x_mode, want_grad, size_cols=n)
    val, pg = val.reshape(L, n * k), pg.reshape(L, n * k)
    for i in range(k):
        vb, pb, gb = prob.run(ctx, x_mode, want_grad, t0=t0 + i * n, tb=n)
        assert vb.tobytes() == np.ascontiguousarray(val[:, i * n: (i + 1) * n]).tobytes(), f"block {i}: value_parts"
        assert pb.tobytes() == np.ascontiguousarray(pg[:, i * n: (i + 1) * n]).tobytes(), f"block {i}: pg_max"
        if want_grad:
            gs = g.reshape(L, n * k, NB)[:, i * n: (i + 1) * n]
            assert gb.tobytes() == np.ascontiguousarray(gs).reshape(L * n, NB).tobytes(), f"block {i}: grad"
    # and the scale is one block's: the reference with size = L * n_mels * n
    value_r, _, pg_r, v_tol, _, pg_tol = prob.reference(EPS64 if x_mode < 2 else EPS32, size_cols=n)
    assert (np.abs(val.reshape(-1) - value_r) <= v_tol).all() and (np.abs(pg.reshape(-1) - pg_r) <= pg_tol).all()


@pytest.mark.parametrize("path", PATHS, ids=[p[0] for p in PATHS])
def test_projected_gradient_arms(cuda, path):
    """Columns built so that each arm of projgr decides, with results known exactly where the arithmetic allows:
    x = 0, B = 0 -> pg = 0 and value = 0 exactly; B < 0 with tiny x (g > x everywhere a band covers) -> pg = max x
    exactly, the min(x, g) arm; x = 0, B > 0 (g <= 0) -> pg = max |g|, the -g arm; and a warm-start column where the
    reference decides between arms."""
    name, x_mode, want_grad, eps = path
    ctx = _ctx(cuda)
    A = ctx.mel_basis()
    covered = (A != 0).any(0)
    n_mels = A.shape[0]
    tb = 4
    S = np.zeros((1, tb, NB), np.float32)
    S[0, 1] = 2.0 ** -20 * (1024 + np.arange(NB)) / 1024        # 11-bit mantissas: S^2 exact in float32
    mel = np.zeros((1, tb, n_mels), np.float32)
    mel[0, 1] = -1.0
    mel[0, 2] = np.linspace(0.5, 2.0, n_mels)
    M = np.exp(lr.reference_logmel(synth.speechy(seed=5, n=256 * 40))[20])
    mel[0, 3] = M
    S[0, 3] = np.sqrt(np.maximum(ctx.mel_pinv().astype(np.float64) @ M, 0)) * np.where(np.arange(NB) % 3 == 0, 0, 1)
    prob = Problem(ctx, 1, tb, 0, tb, 520, 0, seed=0, S=S, mel=mel)
    val, pg = _check_against_reference(ctx, prob, path)
    _, g_r, pg_r, _, _, pg_tol = prob.reference(eps)
    assert pg[0] == 0.0 and val[0] == 0.0                                                  # x = 0, B = 0
    assert (g_r[1][covered] > prob.X[1][covered]).all()
    assert pg[1] == prob.X[1][covered].max()                                               # min(x, g) arm, exact
    assert (g_r[2] <= 0).all() and pg_r[2] > 1e3 * pg_tol[2]                               # -g arm
    neg = np.where(g_r[3] < 0, -g_r[3], 0).max()
    pos = np.where(g_r[3] >= 0, np.minimum(prob.X[3], g_r[3]), 0).max()
    assert abs(neg - pos) > 2 * pg_tol[3]                    # one arm decides column 3, clearly: the check above tells them apart


@functools.lru_cache(maxsize=None)
def _speech_mel(seed, n_frames):
    """reference-range log-mel ([-10, 2]) of speech-like signal, [80, n_frames] float32 (shared, read-only)"""
    lm = lr.reference_logmel(synth.speechy(seed=seed, n=(n_frames - 1) * 256)).T.copy()
    lm.setflags(write=False)
    return lm


@pytest.mark.parametrize("scale", [1e-3, 1.0, 1e2, 1e4])
@pytest.mark.parametrize("b,T", [(1, 820), (16, 51)])
@pytest.mark.parametrize("is_log", [0, 1])
def test_float32_screen_classifies_like_float64(cuda, is_log, b, T, scale):
    """The screening pass (x_mode 2: the banded kernel, and the dense float kernel behind a gradient buffer) on the
    oracle's warm start of reference-range log-mel times ``scale``: pg_max within the error bound and within
    SCREEN_REL of float64, and every column whose float64 pg lies outside [0.9, 1.1] * pgtol classified alike."""
    ctx = _ctx(cuda)
    lm = _speech_mel(40 + b, b * T + 40 * b)
    items = np.stack([lm[:, 40 * i: 40 * i + T] for i in range(b)])                           # [b, 80, T]
    M = (np.exp(items) * np.float32(scale)).astype(np.float32)
    x = lr.nnls(ctx.mel_basis(), M, lbfgs=False)                                              # clip(pinv(A) M, 0), float32
    S = np.sqrt(x).transpose(0, 2, 1)
    mel = (np.log(M) if is_log else M).transpose(0, 2, 1).astype(np.float32)
    prob = Problem(ctx, b, T, 0, T, 520, is_log, seed=0, S=np.ascontiguousarray(S), mel=np.ascontiguousarray(mel))
    _, _, pg64, _, _, _ = prob.reference(EPS64)
    report = []
    for path in PATHS[2:]:
        _, pg32 = _check_against_reference(ctx, prob, path)
        rel = np.abs(pg32 - pg64) / np.maximum(pg64, 1e-300)
        report.append((path[0], float(rel[pg64 > 0].max(initial=0.0))))
        assert rel[pg64 > 0].max(initial=0.0) <= SCREEN_REL, report
        outside = (pg64 < 0.9 * PGTOL) | (pg64 > 1.1 * PGTOL)
        assert ((pg32 > PGTOL) == (pg64 > PGTOL))[outside].all(), path[0]
    print(f"float32 screen rel error of pg_max (is_log={is_log}, b={b}, T={T}, scale={scale:g}):", report,
          f"pg/pgtol in [{pg64.min() / PGTOL:.3g}, {pg64.max() / PGTOL:.3g}]")


# ---------------------------------------------------------------------------------------------------------------------
# nnls_refine's decisions
# ---------------------------------------------------------------------------------------------------------------------
def _block_pg(A, x, M, blocks):
    """float64 pg of librosa's objective at x (float [b, 513, T]) for each block of M [b, n_mels, T]"""
    out = {}
    for t0, t1 in blocks:
        xb, Bb = x[..., t0:t1].astype(np.float64), M[..., t0:t1].astype(np.float64)
        r = np.einsum("mf,...ft->...mt", A, xb) - Bb
        g = np.einsum("mf,...mt->...ft", A, r) / Bb.size
        out[(t0, t1)] = float(np.where(g < 0, -g, np.minimum(xb, g)).max())
    return out


class Recorder:
    """Wraps scipy's fmin_l_bfgs_b (which nnls_refine imports at call time), the library's spev_nnls_objective and
    nnls_refine itself: records each block handed to L-BFGS-B (its x0), the x_mode of every screening launch and each
    returned count."""

    def __init__(self, monkeypatch, ctx):
        import scipy.optimize
        from spev_tts_b200 import spectral
        self.x0, self.modes, self.counts = [], [], []
        real_lbfgs, real_obj, real_refine = scipy.optimize.fmin_l_bfgs_b, ctx.lib.spev_nnls_objective, spectral.nnls_refine

        def lbfgs(func, x0, *a, **k):
            self.x0.append(np.array(x0, dtype=np.float64, copy=True))
            return real_lbfgs(func, x0, *a, **k)

        def obj(*a):
            if a[12] is None:                                      # screening launches pass no gradient buffer
                self.modes.append(a[2])
            return real_obj(*a)

        def refine(*a, **k):
            n = real_refine(*a, **k)
            self.counts.append(n)
            return n
        monkeypatch.setattr(scipy.optimize, "fmin_l_bfgs_b", lbfgs)
        monkeypatch.setattr(ctx.lib, "spev_nnls_objective", obj)
        monkeypatch.setattr(spectral, "nnls_refine", refine)

    def reset(self):
        self.x0.clear(), self.modes.clear(), self.counts.clear()

    def blocks(self, S_warm, blocks):
        """identify each recorded x0 with the block of the warm start S_warm [b, 513, T] it is closest to"""
        b = S_warm.shape[0]
        x_w = S_warm.astype(np.float64) ** 2
        got = []
        for x0 in self.x0:
            tb = x0.size // (b * NB)
            cand = [(t0, t1) for t0, t1 in blocks if t1 - t0 == tb]
            d = [np.linalg.norm(x0 - x_w[..., t0:t1].ravel()) / max(np.linalg.norm(x0), 1e-300) for t0, t1 in cand]
            assert cand and min(d) <= 1e-3, "L-BFGS-B was handed something that is no block of the warm start"
            got.append(cand[int(np.argmin(d))])
        assert len(set(got)) == len(got), "a block was iterated twice"
        return set(got)


# b = 1 slices start at column 400 (T <= 40) or 0 of one 1701-frame utterance; b = 16 items start 40 columns apart.
# Between them: blocks at 0.03, 0.5-0.6, 1.1 (the float64 re-screen), 1.3, 2-20 times pgtol.
DECISION_CASES = [(1, T, 400) for T in (1, 5, 20, 39, 40)] + [(1, T, 0) for T in (818, 819, 820, 1638, 1639)] + \
                 [(16, T, 0) for T in (50, 51, 52, 120, 153)]


def test_refine_decisions_follow_librosa_first_convergence_test(cuda, monkeypatch):
    """nnls_refine hands L-BFGS-B exactly the blocks whose float64 projected gradient at the oracle's float32 warm start
    exceeds pgtol (librosa's solver iterates there and returns x0 elsewhere), re-screens in float64 when the float32
    pass is within 10 % of pgtol, and returns the number of blocks it iterated.  mel_to_audio (log-mel input, the
    overlapped path) takes the same decisions as mel_to_stft, and when blocks iterate its waveform is bit-identical to
    griffinlim(mel_to_stft(...)) from the same phases."""
    import spev_tts_b200 as sp
    from spev_tts_b200.spectral import nnls_blocks
    ctx = _ctx(cuda)
    A = ctx.mel_basis()
    A64 = A.astype(np.float64)
    lm = _speech_mel(300, 1701)
    rec = Recorder(monkeypatch, ctx)
    seen, bands, report = [], [], []
    rescreened = False
    for b, T, s0 in DECISION_CASES:
        items = np.stack([lm[:, s0 + 40 * i: s0 + 40 * i + T] for i in range(b)])             # [b, 80, T] log-mel
        M = np.exp(items)
        _, blocks = nnls_blocks(b, T, 80)
        pg_or = _block_pg(A64, lr.nnls(A, M, lbfgs=False), M, blocks)
        S_warm = sp.mel_to_stft(M, sr=22050, n_fft=1024, fmin=0, fmax=8000, nnls="pinv").reshape(b, NB, T)
        pg_prod = _block_pg(A64, S_warm.astype(np.float64) ** 2, M, blocks)
        bands += [abs(pg_prod[k] - pg_or[k]) / pg_or[k] for k in blocks]
        rec.reset()
        sp.mel_to_stft(M, sr=22050, n_fft=1024, fmin=0, fmax=8000)
        got = rec.blocks(S_warm, blocks)
        assert rec.counts == [len(rec.x0)], (b, T, rec.counts, len(rec.x0))
        want = {k for k in blocks if pg_or[k] > PGTOL}
        for k in got ^ want:
            assert abs(pg_or[k] / PGTOL - 1) <= DECISION_BAND, (b, T, k, pg_or[k] / PGTOL)
        # the float64 re-screen runs iff a block's float32 pg lies within [0.9, 1.1] * pgtol (edges left out)
        near = [abs(pg_prod[k] / PGTOL - c) <= 1e-4 for k in blocks for c in (0.9, 1.1)]
        if not any(near):
            expect = any(0.9 <= pg_prod[k] / PGTOL <= 1.1 for k in blocks)
            assert (1 in rec.modes) == expect, (b, T, rec.modes, {k: pg_prod[k] / PGTOL for k in blocks})
            rescreened |= expect
        assert rec.modes[0] == 2, rec.modes                                                  # the float32 screen comes first
        seen += [pg_or[k] / PGTOL for k in blocks]
        report.append((b, T, sorted(got), {k: round(v / PGTOL, 4) for k, v in pg_or.items()}))
        # mel_to_audio: same decisions on log-mel input with the screen overlapped by Griffin-Lim
        rec.reset()
        sp.mel_to_audio(items, sr=22050, n_fft=1024, hop_length=256, fmin=0, fmax=8000, n_iter=1, is_log=True,
                        init_phase=np.zeros((b, NB, T), np.float32))
        got_audio = rec.blocks(S_warm, blocks)
        for k in got_audio ^ got:
            assert abs(pg_or[k] / PGTOL - 1) <= DECISION_BAND, ("mel_to_audio", b, T, k)
        assert rec.counts == [len(rec.x0)]
        if got and T > 1:                                                                    # re-run after refinement
            ph = synth.init_phase((b, NB, T), seed=T)
            y = sp.mel_to_audio(M, sr=22050, n_fft=1024, hop_length=256, fmin=0, fmax=8000, n_iter=3, init_phase=ph)
            S = sp.mel_to_stft(M, sr=22050, n_fft=1024, fmin=0, fmax=8000)
            y_ref = sp.griffinlim(S, n_iter=3, hop_length=256, n_fft=1024, init_phase=ph)
            assert np.array_equal(y, y_ref), (b, T)
    print("refine decisions (b, T, iterated blocks, oracle pg/pgtol per block):", report)
    print(f"decision band: max relative pg difference, product vs oracle warm start = {max(bands):.3g}")
    assert max(bands) <= DECISION_BAND
    seen = np.array(seen)
    assert (seen > 2).any() and (seen < 0.5).any() and rescreened, "the cases must straddle pgtol and re-screen once"


# ---------------------------------------------------------------------------------------------------------------------
# warm start: spev_mel_to_mag
# ---------------------------------------------------------------------------------------------------------------------
FRAMES = [1, 15, 16, 17, 32, 33, 100]                     # kMagFrames = 16 and 32-frame tile edges
SENT = -1234.5


def _mel_to_mag(ctx, fb, mel, layout, is_log, ld_s):
    """S [n_frames + 3, ld_s] pre-filled with a sentinel; the kernel must write [:n_frames, :513] only."""
    from spev_tts_b200 import _lib
    S = torch.full((fb.n_frames + 3, ld_s), SENT, dtype=torch.float32, device=mel.device)
    _lib.check(ctx.lib.spev_mel_to_mag(ctx.handle, fb.desc, mel.data_ptr(), layout, int(is_log), S.data_ptr(), ld_s,
                                       _st(mel.device)), "spev_mel_to_mag")
    return S.cpu().numpy()


def _warm_ref(ctx, items, is_log, terms):
    """float64 sqrt(max(pinv . M, 0)) per frame [F, 513] and its bound for a float32 sum of ``terms`` roundings per
    product; M = exp of the log-mel when is_log (2 ulp for expf)."""
    P = ctx.mel_pinv().astype(np.float64)
    M = np.concatenate([(np.exp(it.astype(np.float64)) if is_log else it).T for it in items]).astype(np.float64)
    dM = np.concatenate([_expf_ulps(it).T for it in items]) if is_log else 0
    z = M @ P.T
    dz = (terms * EPS32 * np.abs(M) + dM) @ np.abs(P).T
    S = np.sqrt(np.maximum(z, 0))
    tol = np.minimum(np.sqrt(dz), dz / np.maximum(S, 1e-300)) + EPS32 * S
    return S, tol


def _check_sentinels(S, F, what):
    assert (S[:F, NB:] == SENT).all(), f"{what}: pad columns written"
    assert (S[F:] == SENT).all(), f"{what}: rows outside the batch written"


@pytest.mark.parametrize("is_log", [0, 1])
def test_warm_start_layouts(cuda, is_log):
    """Layout 1 (per item [n_mels, T_i] at frame_off[i] * n_mels) on the FFMA kernel against float64; layout 0 on the
    FFMA kernel bit-identical to it; the tcgen05 (3xTF32) path within its bound of both.  The FFMA kernel leaves pad
    columns and rows outside the batch as they were."""
    import spev_tts_b200 as sp
    ctx = _ctx(cuda)
    fb = sp.make_batch(ctx, n_frames=FRAMES)
    F, n_mels = fb.n_frames, ctx.n_mels
    lm = _speech_mel(9, 300)
    items = [lm[:, 7 * i: 7 * i + T] for i, T in enumerate(FRAMES)]
    if not is_log:
        items = [np.exp(it) for it in items]
    l1 = torch.from_numpy(np.concatenate([it.ravel() for it in items])).to(cuda)
    l0 = torch.from_numpy(np.concatenate([it.T.ravel() for it in items])).to(cuda)
    S_ref, tol = _warm_ref(ctx, items, is_log, n_mels + 8)
    s1 = _mel_to_mag(ctx, fb, l1, 1, is_log, 520)
    _check_sentinels(s1, F, "layout 1")
    assert (np.abs(s1[:F, :NB] - S_ref) <= tol).all(), float(np.max(np.abs(s1[:F, :NB] - S_ref) / tol))
    try:
        ctx.set_tensor_core(False)
        s0 = _mel_to_mag(ctx, fb, l0, 0, is_log, 520)
    finally:
        ctx.set_tensor_core(True)
    assert np.array_equal(s0, s1), "FFMA layout 0 != layout 1"
    tc = _mel_to_mag(ctx, fb, l0, 0, is_log, 520)
    assert (tc[F:] == SENT).all(), "tcgen05: rows outside the batch written"
    # 3xTF32: three products per term (about 6 eps32 each for the dropped lo*lo and the split), all summed in float32
    _, tol_tc = _warm_ref(ctx, items, is_log, 3 * n_mels + 16)
    assert (np.abs(tc[:F, :NB] - S_ref) <= tol_tc).all(), float(np.max(np.abs(tc[:F, :NB] - S_ref) / tol_tc))
    assert (np.abs(tc[:F, :NB] - s1[:F, :NB]) <= tol_tc + tol).all()
    # ld_s = 513 (not a multiple of 4): the FFMA kernel with the tensor cores switched on
    s513 = _mel_to_mag(ctx, fb, l0, 0, is_log, NB)
    assert (s513[F:] == SENT).all() and np.array_equal(s513[:F], s1[:F, :NB])


@pytest.mark.parametrize("is_log", [0, 1])
def test_warm_start_n_mels_not_multiple_of_4(cuda, is_log):
    """n_mels = 42 takes the FFMA kernel for layout 0 even with the tensor cores on: bit-identical to layout 1, within
    the float64 bound, pads and outside rows untouched."""
    import spev_tts_b200 as sp
    ctx = _ctx(cuda, n_mels=42, fmin=0.0, fmax=None)
    fb = sp.make_batch(ctx, n_frames=FRAMES)
    F = fb.n_frames
    rng = np.random.default_rng(42)
    items = [np.clip(-4 + 2 * rng.standard_normal((42, T)), -10, 2).astype(np.float32) for T in FRAMES]
    if not is_log:
        items = [np.exp(it) for it in items]
    l1 = torch.from_numpy(np.concatenate([it.ravel() for it in items])).to(cuda)
    l0 = torch.from_numpy(np.concatenate([it.T.ravel() for it in items])).to(cuda)
    s1 = _mel_to_mag(ctx, fb, l1, 1, is_log, 520)
    s0 = _mel_to_mag(ctx, fb, l0, 0, is_log, 520)
    _check_sentinels(s0, F, "n_mels 42")
    assert np.array_equal(s0, s1)
    S_ref, tol = _warm_ref(ctx, items, is_log, 42 + 8)
    assert (np.abs(s0[:F, :NB] - S_ref) <= tol).all()
