// abi.cu -- extern "C" boundary (include/spev_b200.h) and ctx construction.
//
// ctx construction restates, in float64 -> float32 exactly as librosa does, the constants the
// reference path rebuilds on every call: scipy.signal.get_window('hann', 1024, fftbins=True)
// and librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax, norm='slaney') (reached from
// /root/reference/spev_real_metrics.py:363 with fmax=None and :730-733 with fmin=0,
// fmax=8000), plus np.linalg.pinv of the basis (librosa.util.nnls warm start).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>

#include "spev_internal.cuh"

namespace spev {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
    return SPEV_E_CUDA;
}

// launchers implemented in spectral.cu / lr.cu / gemm_tc.cu
int launch_stft_mel(spev_ctx*, const spev_batch*, const float*, float*, bool, int, float, float, float, cudaStream_t);
int launch_stft_phase(spev_ctx*, const spev_batch*, const float*, const float*, int64_t, void*, void*, int64_t, float, int, bool, cudaStream_t,
                      unsigned* counter = nullptr, unsigned base = 0, bool fuse = false);
int launch_ola_pairs(spev_ctx*, const spev_batch*, const void*, int64_t, float*, cudaStream_t);
int launch_istft(spev_ctx*, const spev_batch*, const void*, int64_t, float*, cudaStream_t);
int fft_grid(const spev_ctx*, int64_t);
int launch_nnls_objective(spev_ctx*, const void*, int, int64_t, const float*, int, int, int64_t, int64_t, int, int, double*, double*, double*, cudaStream_t);
int spectral_init(spev_ctx*);
int launch_gl_init(spev_ctx*, const float*, int64_t, const float*, uint64_t, void*, int64_t, int64_t, cudaStream_t);
int launch_mel_to_mag(spev_ctx*, const spev_batch*, const float*, int, int, float*, int64_t, cudaStream_t);
int launch_lr_plan(const void*, int, int, int, int32_t*, int64_t*, int64_t*, int64_t*, cudaStream_t);
int launch_lr_expand(const void*, int64_t, const float*, int, const float*, const float*, const int32_t*, int, int, void*, float*, int64_t, cudaStream_t);
int launch_duration_rule(const float*, int64_t, float, int64_t*, cudaStream_t);
int launch_lr_expand_backward(const void*, int, int, const float*, int, const float*, const float*, const float*, const int32_t*,
                              int, int, int64_t, void*, float*, cudaStream_t);
size_t variance_fuse_backward_workspace_bytes(int, int, int, int64_t);
int launch_variance_fuse_backward(const float*, const float*, int, const float*, const float*, const float*, const int32_t*, int,
                                  int, int, int64_t, float*, float*, float*, float*, void*, size_t, cudaStream_t);
int launch_variance_fuse(const float*, const float*, int, const float*, const float*, const float*, const float*, const int32_t*, int, int, int, float*, float*, int64_t, cudaStream_t);
int launch_pcm16_to_f32(const int16_t*, int64_t, float*, cudaStream_t);
int launch_collate(const spev_pad_array*, int, const int64_t*, const int64_t*, const int64_t*, int, int64_t, int64_t, cudaStream_t);
int launch_transpose(const void*, void*, int, int64_t, int, int, int64_t, int64_t, int64_t, int64_t, cudaStream_t);
int launch_copy_segments(const void*, void*, const int64_t*, const int64_t*, const int64_t*, const int64_t*, int, int64_t, cudaStream_t);
int launch_bucketize_embed(const float*, int64_t, const float*, int, int, const float*, int, int64_t*, float*, int, cudaStream_t);
int launch_frame_features(spev_ctx*, const spev_batch*, const float*, float*, float*, cudaStream_t);
int launch_segment_pool(const float*, const int64_t*, const int64_t*, const int64_t*, int, float, float, float, float, int, float,
                        float*, cudaStream_t);
int launch_mel_project_tc(spev_ctx*, const float*, int64_t, float*, int, float, float, float, cudaStream_t);
int launch_mel_to_mag_tc(spev_ctx*, const float*, int64_t, int, float*, int64_t, cudaStream_t);
int gemm_tc_init(spev_ctx*);
void gemm_tc_destroy(spev_ctx*);

// ---- Slaney mel scale (librosa.core.convert) -------------------------------------------------
static double hz_to_mel(double f) {
    const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
    const double logstep = std::log(6.4) / 27.0;
    return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz(double m) {
    const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
    const double logstep = std::log(6.4) / 27.0;
    return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

// librosa.filters.mel: rows computed in float64, stored to float32, Slaney-normalised in place.
static void build_mel_basis(int sr, int n_fft, int n_mels, double fmin, double fmax, std::vector<float>& w) {
    const int nb = 1 + n_fft / 2;
    w.assign(static_cast<size_t>(n_mels) * nb, 0.f);
    std::vector<double> fftfreqs(nb), mel_f(n_mels + 2);
    const double val = 1.0 / (n_fft * (1.0 / sr));          // np.fft.rfftfreq(n, d=1/sr)
    for (int k = 0; k < nb; ++k) fftfreqs[k] = k * val;
    const double m0 = hz_to_mel(fmin), m1 = hz_to_mel(fmax);
    const double step = (m1 - m0) / (n_mels + 1);             // np.linspace
    for (int i = 0; i < n_mels + 2; ++i) mel_f[i] = mel_to_hz(i == n_mels + 1 ? m1 : m0 + i * step);
    for (int i = 0; i < n_mels; ++i) {
        const double fd0 = mel_f[i + 1] - mel_f[i], fd1 = mel_f[i + 2] - mel_f[i + 1];
        const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
        for (int k = 0; k < nb; ++k) {
            const double lower = -(mel_f[i] - fftfreqs[k]) / fd0;
            const double upper = (mel_f[i + 2] - fftfreqs[k]) / fd1;
            const float tri = static_cast<float>(std::max(0.0, std::min(lower, upper)));
            w[static_cast<size_t>(i) * nb + k] = static_cast<float>(static_cast<double>(tri) * enorm);
        }
    }
}

// pinv(A) for A [m x n] (m <= n) by one-sided Jacobi SVD of G = A^T in float64.
static void pinv_jacobi(const std::vector<float>& A, int m, int n, std::vector<float>& P /*[n x m]*/) {
    std::vector<double> G(static_cast<size_t>(n) * m), V(static_cast<size_t>(m) * m, 0.0);
    for (int i = 0; i < m; ++i) {
        V[static_cast<size_t>(i) * m + i] = 1.0;
        for (int k = 0; k < n; ++k) G[static_cast<size_t>(k) * m + i] = A[static_cast<size_t>(i) * n + k];
    }
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < m - 1; ++p)
            for (int q = p + 1; q < m; ++q) {
                double a = 0, b = 0, c = 0;
                for (int k = 0; k < n; ++k) {
                    const double gp = G[static_cast<size_t>(k) * m + p], gq = G[static_cast<size_t>(k) * m + q];
                    a += gp * gp; b += gq * gq; c += gp * gq;
                }
                if (std::fabs(c) <= 1e-300 || std::fabs(c) <= 1e-17 * std::sqrt(a * b)) continue;
                off = std::max(off, std::fabs(c) / std::sqrt(a * b));
                const double zeta = (b - a) / (2.0 * c);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
                const double cs = 1.0 / std::sqrt(1.0 + t * t), sn = cs * t;
                for (int k = 0; k < n; ++k) {
                    double& gp = G[static_cast<size_t>(k) * m + p];
                    double& gq = G[static_cast<size_t>(k) * m + q];
                    const double x = gp, y = gq;
                    gp = cs * x - sn * y; gq = sn * x + cs * y;
                }
                for (int k = 0; k < m; ++k) {
                    double& vp = V[static_cast<size_t>(k) * m + p];
                    double& vq = V[static_cast<size_t>(k) * m + q];
                    const double x = vp, y = vq;
                    vp = cs * x - sn * y; vq = sn * x + cs * y;
                }
            }
        if (off < 1e-15) break;
    }
    std::vector<double> s2(m);
    double smax2 = 0;
    for (int j = 0; j < m; ++j) {
        double a = 0;
        for (int k = 0; k < n; ++k) a += G[static_cast<size_t>(k) * m + j] * G[static_cast<size_t>(k) * m + j];
        s2[j] = a; smax2 = std::max(smax2, a);
    }
    const double rcond = 1e-15;   // numpy.linalg.pinv default
    P.assign(static_cast<size_t>(n) * m, 0.f);
    std::vector<double> acc(static_cast<size_t>(n) * m, 0.0);
    for (int j = 0; j < m; ++j) {
        if (std::sqrt(s2[j]) <= rcond * std::sqrt(smax2)) continue;
        const double inv = 1.0 / s2[j];
        for (int k = 0; k < n; ++k) {
            const double g = G[static_cast<size_t>(k) * m + j] * inv;
            for (int i = 0; i < m; ++i) acc[static_cast<size_t>(k) * m + i] += g * V[static_cast<size_t>(i) * m + j];
        }
    }
    for (size_t i = 0; i < acc.size(); ++i) P[i] = static_cast<float>(acc[i]);
}

template <class T>
static int upload(T** dst, const std::vector<T>& src) {
    SPEV_CUDA(cudaMalloc(reinterpret_cast<void**>(dst), std::max<size_t>(1, src.size()) * sizeof(T)));
    if (!src.empty())
        SPEV_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SPEV_OK;
}

static float tf32_trunc(float x) {
    uint32_t u;
    std::memcpy(&u, &x, 4);
    u &= 0xFFFFE000u;
    std::memcpy(&x, &u, 4);
    return x;
}

// Entry points that take a ctx run on the ctx's device and leave the caller's current device as they found it.
struct DeviceGuard {
    int prev = -1, rc = SPEV_OK;
    explicit DeviceGuard(const spev_ctx* c) {
        if (!c) { set_error("ctx is null"); rc = SPEV_E_INVALID; return; }
        cudaError_t e = cudaGetDevice(&prev);
        if (e == cudaSuccess && prev != c->device) e = cudaSetDevice(c->device); else if (e == cudaSuccess) prev = -1;
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaSetDevice(ctx->device)"); prev = -1; }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define SPEV_ON_CTX_DEVICE(c)      \
    DeviceGuard _guard(c);         \
    if (_guard.rc) return _guard.rc

}  // namespace spev

using namespace spev;

extern "C" {

int spev_abi_version(void) { return SPEV_ABI_VERSION; }
const char* spev_last_error(void) { return g_err.c_str(); }

int spev_create(spev_ctx** out, int device, int sr, int n_fft, int hop, int win, int n_mels,
                float fmin, float fmax) {
    SPEV_REQUIRE(out, SPEV_E_INVALID, "spev_create: out is null");
    *out = nullptr;
    SPEV_REQUIRE(n_fft == kNfft && hop == kHop && (win == kNfft || win <= 0), SPEV_E_UNSUPPORTED,
                 "spev_create: only n_fft=1024, hop=256, win=1024 are implemented (got %d/%d/%d)", n_fft, hop, win);
    SPEV_REQUIRE(sr > 0 && n_mels > 0 && n_mels <= 256, SPEV_E_INVALID, "spev_create: bad sr/n_mels");
    if (fmax <= 0.f) fmax = 0.5f * sr;
    SPEV_REQUIRE(fmin >= 0.f && fmin < fmax, SPEV_E_INVALID, "spev_create: need 0 <= fmin < fmax");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("spev_create: no CUDA device (this library has no CPU fallback)");
        return SPEV_E_DEVICE;
    }
    SPEV_REQUIRE(device >= 0 && device < ndev, SPEV_E_DEVICE, "spev_create: device %d out of range", device);
    cudaDeviceProp prop;
    SPEV_CUDA(cudaGetDeviceProperties(&prop, device));
    SPEV_REQUIRE(prop.major == 10 && prop.minor == 0, SPEV_E_DEVICE,
                 "spev_create: device %d is sm_%d%d; this build carries sm_100a code only", device, prop.major, prop.minor);
    int prev_device = -1;
    SPEV_CUDA(cudaGetDevice(&prev_device));
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{prev_device != device ? prev_device : -1};
    SPEV_CUDA(cudaSetDevice(device));

    spev_ctx* c = new spev_ctx();
    c->device = device; c->sr = sr; c->n_fft = n_fft; c->hop = hop; c->win = kNfft; c->n_mels = n_mels;
    c->fmin = fmin; c->fmax = fmax; c->num_sms = c->num_sms_device = prop.multiProcessorCount; c->tma = nullptr; c->use_tc = 1;
    c->d_tw = nullptr; c->d_window = nullptr; c->d_win2048 = nullptr; c->d_tw2048 = nullptr; c->d_basis = c->d_basis_pad = c->d_basis_hi = c->d_basis_lo = nullptr; c->d_nnls_rng = nullptr;
    c->d_pinv_t = c->d_pinv_hi = c->d_pinv_lo = nullptr;
    c->d_prog_w = nullptr; c->d_prog_h = nullptr;

    // periodic Hann, float64 -> float32
    c->h_window.resize(kNfft);
    for (int i = 0; i < kNfft; ++i) c->h_window[i] = static_cast<float>(0.5 - 0.5 * std::cos(2.0 * M_PI * i / kNfft));
    std::vector<float2> tw(1024);
    for (int k1 = 0; k1 < 32; ++k1)
        for (int l = 0; l < 32; ++l) {
            const double a = -2.0 * M_PI * (k1 * l) / 1024.0;
            tw[k1 * 32 + l] = make_float2(static_cast<float>(std::cos(a)), static_cast<float>(std::sin(a)));
        }
    std::vector<float2> win2048(1024), tw2048(512);
    for (int n = 0; n < 1024; ++n) {
        const double w0 = 0.5 - 0.5 * std::cos(2.0 * M_PI * (2 * n) / 2048.0), w1 = 0.5 - 0.5 * std::cos(2.0 * M_PI * (2 * n + 1) / 2048.0);
        win2048[n] = make_float2(0.5f * static_cast<float>(w0), 0.5f * static_cast<float>(w1));
    }
    for (int k = 0; k < 512; ++k) {
        const double a = -2.0 * M_PI * k / 2048.0;
        tw2048[k] = make_float2(static_cast<float>(std::cos(a)), static_cast<float>(std::sin(a)));
    }
    build_mel_basis(sr, n_fft, n_mels, fmin, fmax, c->h_basis);
    pinv_jacobi(c->h_basis, n_mels, kBins, c->h_pinv);

    // mel program of the fused kernel (see MelProgram): float4 groups, LPT-balanced over 16 warps
    std::vector<int> bstart(n_mels), bn4(n_mels);
    c->band_max_len = 0; c->band_nnz = 0;
    for (int m = 0; m < n_mels; ++m) {
        int lo = kBins, hi = -1;
        for (int k = 0; k < kBins; ++k)
            if (c->h_basis[static_cast<size_t>(m) * kBins + k] != 0.f) { lo = std::min(lo, k); hi = std::max(hi, k); ++c->band_nnz; }
        bstart[m] = hi >= lo ? (lo / 4) * 4 : 0;
        bn4[m] = hi >= lo ? (hi - bstart[m] + 4) / 4 : 1;   // an empty filter still emits (a zero)
        c->band_max_len = std::max(c->band_max_len, hi >= lo ? hi - lo + 1 : 0);
    }
    // Bands are dealt to the 16 warps, at most nb = ceil(n_mels / 16) each, longest first onto the least-loaded warp
    // (LPT).  A warp's weights are stored band after band as float4 groups of consecutive bins, so a band is fully
    // described by one header: (first group, first bin, group count, mel index).
    const int nb = (n_mels + kWarps - 1) / kWarps;
    std::vector<std::vector<int>> warp_bands(kWarps);
    {
        std::vector<int> by_len(n_mels), load(kWarps, 0);
        for (int m = 0; m < n_mels; ++m) by_len[m] = m;
        std::stable_sort(by_len.begin(), by_len.end(), [&](int a, int b) { return bn4[a] > bn4[b]; });
        for (int m : by_len) {
            int w = -1;
            for (int q = 0; q < kWarps; ++q)
                if (static_cast<int>(warp_bands[q].size()) < nb && (w < 0 || load[q] < load[w])) w = q;
            warp_bands[w].push_back(m);
            load[w] += bn4[m] + 1;   // +1: emit cost
        }
    }
    std::vector<float4> prog_w;
    std::vector<int4> prog_h(static_cast<size_t>(kWarps) * nb, make_int4(0, 0, 0, -1));
    int gmax = 1;
    for (int w = 0; w < kWarps; ++w) {
        int gw = 0;
        for (size_t q = 0; q < warp_bands[w].size(); ++q) {
            const int m = warp_bands[w][q];
            prog_h[static_cast<size_t>(w) * nb + q] = make_int4(static_cast<int>(prog_w.size()), bstart[m], bn4[m], m);
            for (int j = 0; j < bn4[m]; ++j) {
                float wv[4];
                for (int t = 0; t < 4; ++t) {
                    const int bin = bstart[m] + 4 * j + t;   // bins 513..515 of a slot are kept at zero
                    wv[t] = bin < kBins ? c->h_basis[static_cast<size_t>(m) * kBins + bin] : 0.f;
                }
                prog_w.push_back(make_float4(wv[0], wv[1], wv[2], wv[3]));
            }
            gw += bn4[m];
        }
        gmax = std::max(gmax, gw);
    }
    c->prog_gmax = gmax;
    c->prog_nb = nb;
    c->prog_groups = static_cast<int>(prog_w.size());

    // padded / split operands for the tensor-core GEMMs
    std::vector<float> basis_pad(static_cast<size_t>(n_mels) * kSpecLd, 0.f), b_hi(basis_pad.size()), b_lo(basis_pad.size());
    std::vector<float> pinv_t(static_cast<size_t>(n_mels) * kSpecLd, 0.f);
    for (int m = 0; m < n_mels; ++m)
        for (int k = 0; k < kBins; ++k) {
            basis_pad[static_cast<size_t>(m) * kSpecLd + k] = c->h_basis[static_cast<size_t>(m) * kBins + k];
            pinv_t[static_cast<size_t>(m) * kSpecLd + k] = c->h_pinv[static_cast<size_t>(k) * n_mels + m];
        }
    for (size_t i = 0; i < basis_pad.size(); ++i) { b_hi[i] = tf32_trunc(basis_pad[i]); b_lo[i] = basis_pad[i] - b_hi[i]; }

    // d_window = [1024] Hann followed by [256] 1 / sum_q w[768 - 256 q + s]^2: the window-sum-square of interior ISTFT
    // chunks, accumulated with the same ascending-frame fmaf chain k_istft uses in the kernel (IEEE: same bits)
    std::vector<float> win_iw(c->h_window);
    for (int s = 0; s < kHop; ++s) {
        float wss = 0.f;
        for (int q = 0; q < 4; ++q) { const float w = c->h_window[768 - 256 * q + s]; wss = std::fmaf(w, w, wss); }
        win_iw.push_back(1.0f / wss);
    }
    // banded view of the basis (NNLS screening kernel): per band its run of non-zero bins, per bin the bands that cover it
    std::vector<int> nnls_rng(2 * static_cast<size_t>(n_mels) + 2 * kBins);
    for (int m = 0; m < n_mels; ++m) {
        int lo = kBins, hi = -1;
        for (int k = 0; k < kBins; ++k)
            if (c->h_basis[static_cast<size_t>(m) * kBins + k] != 0.f) { lo = std::min(lo, k); hi = std::max(hi, k); }
        nnls_rng[2 * m] = hi >= lo ? lo : 0;
        nnls_rng[2 * m + 1] = hi >= lo ? hi - lo + 1 : 0;
    }
    for (int k = 0; k < kBins; ++k) {
        int lo = n_mels, hi = -1;
        for (int m = 0; m < n_mels; ++m)
            if (c->h_basis[static_cast<size_t>(m) * kBins + k] != 0.f) { lo = std::min(lo, m); hi = std::max(hi, m); }
        nnls_rng[2 * n_mels + 2 * k] = hi >= lo ? lo : 0;
        nnls_rng[2 * n_mels + 2 * k + 1] = hi >= lo ? hi : -1;
    }
    int rc = SPEV_OK;
    if ((rc = upload(&c->d_tw, tw)) || (rc = upload(&c->d_window, win_iw)) ||
        (rc = upload(&c->d_win2048, win2048)) || (rc = upload(&c->d_tw2048, tw2048)) ||
        (rc = upload(&c->d_basis, c->h_basis)) || (rc = upload(&c->d_nnls_rng, nnls_rng)) || (rc = upload(&c->d_basis_pad, basis_pad)) || (rc = upload(&c->d_basis_hi, b_hi)) ||
        (rc = upload(&c->d_basis_lo, b_lo)) || (rc = upload(&c->d_pinv_t, pinv_t)) ||
        (rc = upload(&c->d_prog_w, prog_w)) || (rc = upload(&c->d_prog_h, prog_h)) ||
        (rc = gemm_tc_init(c)) || (rc = spectral_init(c))) {
        spev_destroy(c);
        return rc;
    }
    *out = c;
    return SPEV_OK;
}

void spev_destroy(spev_ctx* c) {
    if (!c) return;
    DeviceGuard guard(c);
    gemm_tc_destroy(c);
    cudaFree(c->d_tw); cudaFree(c->d_window); cudaFree(c->d_win2048); cudaFree(c->d_tw2048); cudaFree(c->d_basis); cudaFree(c->d_nnls_rng); cudaFree(c->d_basis_pad); cudaFree(c->d_basis_hi);
    cudaFree(c->d_basis_lo); cudaFree(c->d_pinv_t); cudaFree(c->d_pinv_hi); cudaFree(c->d_pinv_lo);
    cudaFree(c->d_prog_w); cudaFree(c->d_prog_h);
    delete c;
}

int spev_get_mel_basis(const spev_ctx* c, float* dst) {
    SPEV_REQUIRE(c && dst, SPEV_E_INVALID, "null argument");
    std::memcpy(dst, c->h_basis.data(), c->h_basis.size() * sizeof(float));
    return SPEV_OK;
}
int spev_get_mel_pinv(const spev_ctx* c, float* dst) {
    SPEV_REQUIRE(c && dst, SPEV_E_INVALID, "null argument");
    std::memcpy(dst, c->h_pinv.data(), c->h_pinv.size() * sizeof(float));
    return SPEV_OK;
}
int spev_get_window(const spev_ctx* c, float* dst) {
    SPEV_REQUIRE(c && dst, SPEV_E_INVALID, "null argument");
    std::memcpy(dst, c->h_window.data(), c->h_window.size() * sizeof(float));
    return SPEV_OK;
}

int spev_host_mel_basis(int sr, int n_fft, int n_mels, float fmin, float fmax, float* basis) {
    SPEV_REQUIRE(basis && sr > 0 && n_fft > 0 && n_mels > 0, SPEV_E_INVALID, "spev_host_mel_basis: bad argument");
    if (fmax <= 0.f) fmax = 0.5f * sr;
    std::vector<float> w;
    build_mel_basis(sr, n_fft, n_mels, fmin, fmax, w);
    std::memcpy(basis, w.data(), w.size() * sizeof(float));
    return SPEV_OK;
}

int spev_host_pinv(const float* a, int m, int n, float* pinv) {
    SPEV_REQUIRE(a && pinv && m > 0 && n >= m, SPEV_E_INVALID, "spev_host_pinv: need m <= n");
    std::vector<float> A(a, a + static_cast<size_t>(m) * n), P;
    pinv_jacobi(A, m, n, P);
    std::memcpy(pinv, P.data(), P.size() * sizeof(float));
    return SPEV_OK;
}

int spev_set_tensor_core(spev_ctx* c, int enable) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "ctx is null");
    c->use_tc = enable ? 1 : 0;
    return SPEV_OK;
}

int spev_tile_frames(void) { return kTileFrames; }
int spev_tile_chunks(void) { return kTileChunks; }

int64_t spev_plan_frame_tiles(const int64_t* frames, const int64_t* sample_lo, const int64_t* n_samples,
                              int n_items, spev_tile* out) {
    SPEV_REQUIRE(frames && n_items >= 0, SPEV_E_INVALID, "spev_plan_frame_tiles: frames is null or n_items < 0");
    SPEV_REQUIRE(sample_lo && n_samples, SPEV_E_INVALID, "spev_plan_frame_tiles: sample_lo or n_samples is null");
    for (int i = 0; i < n_items; ++i)
        SPEV_REQUIRE(n_samples[i] >= 0, SPEV_E_INVALID, "spev_plan_frame_tiles: n_samples[%d] = %lld < 0", i,
                     static_cast<long long>(n_samples[i]));
    int64_t nt = 0, fo = 0;
    for (int i = 0; i < n_items; ++i) {
        const int64_t T = frames[i], lo = sample_lo[i], hi = lo + n_samples[i];
        for (int64_t t0 = 0; t0 < T; t0 += kTileFrames, ++nt) {
            if (!out) continue;
            spev_tile& d = out[nt];
            d.src0 = lo + kHop * t0 - kNfft / 2; d.lo = lo; d.hi = hi; d.row0 = fo + t0;
            d.n = static_cast<int32_t>(std::min<int64_t>(kTileFrames, T - t0));
            d.t0 = static_cast<int32_t>(t0); d.T = static_cast<int32_t>(T); d.item = i;
        }
        fo += T;
    }
    return nt;
}

int64_t spev_plan_chunk_tiles(const int64_t* frames, const int64_t* out_off, const int64_t* out_len, int n_items,
                              spev_tile* out) {
    SPEV_REQUIRE(frames && n_items >= 0, SPEV_E_INVALID, "spev_plan_chunk_tiles: frames is null or n_items < 0");
    SPEV_REQUIRE(out_off && out_len, SPEV_E_INVALID, "spev_plan_chunk_tiles: out_off or out_len is null");
    for (int i = 0; i < n_items; ++i)
        SPEV_REQUIRE(out_len[i] >= 0, SPEV_E_INVALID, "spev_plan_chunk_tiles: out_len[%d] = %lld < 0", i,
                     static_cast<long long>(out_len[i]));
    // Full tiles first, then the (at most one per item) partial tiles: the persistent kernels hand tile j to CTA
    // j mod grid, so the cheap tiles land in the last, incomplete round (cfg3: 448 tiles on 148 SMs).
    int64_t nt = 0;
    for (int pass = 0; pass < 2; ++pass) {
        int64_t fo = 0;
        for (int i = 0; i < n_items; ++i) {
            // ceil(out_len/hop) chunks at out_off, bounded by [lo, hi)
            const int64_t T = frames[i], lo = out_off[i], hi = lo + out_len[i];
            const int64_t nc = (out_len[i] + kHop - 1) / kHop;
            for (int64_t c0 = 0; c0 < nc; c0 += kTileChunks) {
                const int64_t n = std::min<int64_t>(kTileChunks, nc - c0);
                if ((n == kTileChunks) != (pass == 0)) continue;
                if (out) {
                    spev_tile& d = out[nt];
                    d.src0 = lo + kHop * c0; d.lo = lo; d.hi = hi; d.row0 = fo + c0 - 1;
                    d.n = static_cast<int32_t>(n);
                    d.t0 = static_cast<int32_t>(c0); d.T = static_cast<int32_t>(T); d.item = i;
                }
                ++nt;
            }
            fo += T;
        }
    }
    return nt;
}


int spev_logmel(spev_ctx* c, const spev_batch* b, const float* samples, float* out, int mode,
                float floor_v, float lo, float hi, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(mode == 0 || mode == 1, SPEV_E_INVALID, "spev_logmel: mode must be 0 or 1");
    return launch_stft_mel(c, b, samples, out, false, mode, floor_v, lo, hi, static_cast<cudaStream_t>(stream));
}

int spev_stft_power(spev_ctx* c, const spev_batch* b, const float* samples, float* power, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    return launch_stft_mel(c, b, samples, power, true, 0, 0.f, 0.f, 0.f, static_cast<cudaStream_t>(stream));
}

int spev_mel_project(spev_ctx* c, const float* power, int64_t n_frames, float* out, int mode,
                     float floor_v, float lo, float hi, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(mode == 0 || mode == 1, SPEV_E_INVALID, "spev_mel_project: mode must be 0 or 1");
    return launch_mel_project_tc(c, power, n_frames, out, mode, floor_v, lo, hi, static_cast<cudaStream_t>(stream));
}

int spev_mel_to_mag(spev_ctx* c, const spev_batch* b, const float* mel, int layout, int is_log,
                    float* S, int64_t ld_s, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(b, SPEV_E_INVALID, "spev_mel_to_mag: batch is null");
    // frame-major input: TMA-staged tcgen05 (3xTF32) GEMM; [n_mels, T] items: FFMA kernel
    const bool tc_ok = c->use_tc && layout == 0 && c->n_mels % 4 == 0 && ld_s % 4 == 0 && b->n_frames > 0 &&
                       (reinterpret_cast<uintptr_t>(mel) & 15) == 0 && (reinterpret_cast<uintptr_t>(S) & 15) == 0 &&
                       ld_s >= kSpecLd;
    if (tc_ok) return launch_mel_to_mag_tc(c, mel, b->n_frames, is_log, S, ld_s, static_cast<cudaStream_t>(stream));
    return launch_mel_to_mag(c, b, mel, layout, is_log, S, ld_s, static_cast<cudaStream_t>(stream));
}

int spev_nnls_objective(spev_ctx* c, const void* x, int x_mode, int64_t ld_x, const float* mel, int is_log, int L, int64_t T,
                        int64_t t0, int tb, int size_cols, double* value_parts, double* grad, double* pg_max, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(x_mode >= 0 && x_mode <= 2, SPEV_E_INVALID, "spev_nnls_objective: x_mode must be 0, 1 or 2");
    return launch_nnls_objective(c, x, x_mode, ld_x, mel, is_log, L, T, t0, tb, size_cols, value_parts, grad, pg_max,
                                 static_cast<cudaStream_t>(stream));
}

int spev_istft(spev_ctx* c, const spev_batch* b, const void* spec, int64_t ld, float* y, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    return launch_istft(c, b, spec, ld, y, static_cast<cudaStream_t>(stream));
}

int spev_stft(spev_ctx* c, const spev_batch* b, const float* y, void* spec, int64_t ld, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    return launch_stft_phase(c, b, y, nullptr, 0, spec, nullptr, ld, 0.f, 0, false, static_cast<cudaStream_t>(stream));
}

int spev_gl_phase_update(spev_ctx* c, const spev_batch* b, const float* y, const float* S, int64_t ld_s,
                         void* ang, void* tprev, int64_t ld, float alpha, int has_prev, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    return launch_stft_phase(c, b, y, S, ld_s, ang, tprev, ld, alpha, has_prev, true, static_cast<cudaStream_t>(stream));
}

size_t spev_griffinlim_workspace_bytes(int64_t n_frames) {
    if (n_frames < 0) return 0;
    return static_cast<size_t>(n_frames) * kSpecLd * 2 * sizeof(float2) + 256 /* alignment */ + 256 /* ticket counters */;
}

int spev_griffinlim(spev_ctx* c, const spev_batch* b, const float* S, int64_t ld_s, const float* init_phase,
                    uint64_t seed, int n_iter, float momentum, float* y, void* workspace,
                    size_t workspace_bytes, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(b, SPEV_E_INVALID, "spev_griffinlim: batch is null");
    SPEV_REQUIRE(n_iter >= 0 && momentum >= 0.f, SPEV_E_INVALID, "spev_griffinlim: need n_iter >= 0, momentum >= 0");
    if (b->n_frames == 0) return SPEV_OK;
    SPEV_REQUIRE(S && ld_s >= kBins, SPEV_E_INVALID, "spev_griffinlim: null S or ld_s < 513");
    SPEV_REQUIRE(y || b->n_ctiles == 0, SPEV_E_INVALID, "spev_griffinlim: y is null");
    SPEV_REQUIRE(workspace && workspace_bytes >= spev_griffinlim_workspace_bytes(b->n_frames), SPEV_E_WORKSPACE,
                 "spev_griffinlim: workspace too small (%zu < %zu)", workspace_bytes,
                 spev_griffinlim_workspace_bytes(b->n_frames));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~static_cast<uintptr_t>(255);
    float2* ang = reinterpret_cast<float2*>(base);
    float2* tprev = ang + b->n_frames * kSpecLd;
    // ticket counter of the dynamic pair scheduler: word 32 of the 256-byte counter block (a cache line of its own);
    // it only grows during a call -- launch j starts at base j * (work + workers), see draw_ticket()
    unsigned* counters = reinterpret_cast<unsigned*>(tprev + b->n_frames * kSpecLd);
    SPEV_CUDA(cudaMemsetAsync(counters, 0, 256, st));
    const unsigned per_phase = static_cast<unsigned>(static_cast<int64_t>(b->n_ftiles) * kWarps +
                                                     static_cast<int64_t>(fft_grid(c, b->n_ftiles)) * kWarps);
    // librosa: (momentum / (1 + momentum)) is a Python float applied to a complex64 array
    const float alpha = static_cast<float>(static_cast<double>(momentum) / (1.0 + static_cast<double>(momentum)));
    int rc = SPEV_OK;
    if ((rc = launch_gl_init(c, S, ld_s, init_phase, seed, ang, kSpecLd, b->n_frames, st))) return rc;
    // Fused iteration: y = istft(ang) once, then n_iter x { STFT + phase update + inverse transform of the new spectra
    // in registers -> pair segments (in the `ang` buffer, which nothing else reads any more); overlap-add of the
    // segments -> y }.  The new spectra never travel through HBM: 17.3 instead of 20.5 KB per frame and iteration,
    // every FFT in the barrier-free warp-independent kernel, no halo recomputation.
    if ((rc = launch_istft(c, b, ang, kSpecLd, y, st))) return rc;
    for (int it = 0; it < n_iter; ++it) {
        if ((rc = launch_stft_phase(c, b, y, S, ld_s, ang, tprev, kSpecLd, alpha, it > 0, true, st, counters + 32,
                                    per_phase * static_cast<unsigned>(it), true))) return rc;
        if ((rc = launch_ola_pairs(c, b, ang, kSpecLd, y, st))) return rc;
    }
    return SPEV_OK;
}

int spev_frame_features(spev_ctx* c, const spev_batch* b, const float* samples, float* rms, float* centroid, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    return launch_frame_features(c, b, samples, rms, centroid, static_cast<cudaStream_t>(stream));
}

int spev_segment_pool(const float* curve, const int64_t* frame_off, const int64_t* durs, const int64_t* phone_off,
                      int n_items, float mu, float sigma, float lo, float hi, float* out, void* stream) {
    return launch_segment_pool(curve, frame_off, durs, phone_off, n_items, mu, sigma, lo, hi, 0, 0.f, out,
                               static_cast<cudaStream_t>(stream));
}

int spev_segment_pool_log(const float* curve, float log_eps, const int64_t* frame_off, const int64_t* durs,
                          const int64_t* phone_off, int n_items, float mu, float sigma, float lo, float hi, float* out,
                          void* stream) {
    return launch_segment_pool(curve, frame_off, durs, phone_off, n_items, mu, sigma, lo, hi, 1, log_eps, out,
                               static_cast<cudaStream_t>(stream));
}

int spev_collate(const spev_pad_array* arrays, int n_arrays, const int64_t* frame_off, const int64_t* phone_off,
                 const int64_t* sel, int B, int64_t t_max, int64_t p_max, void* stream) {
    return launch_collate(arrays, n_arrays, frame_off, phone_off, sel, B, t_max, p_max, static_cast<cudaStream_t>(stream));
}

int spev_transpose_batched(const void* src, void* dst, int elem_bytes, int64_t batches, int rows, int cols, int64_t src_pitch,
                           int64_t src_batch, int64_t dst_pitch, int64_t dst_batch, void* stream) {
    return launch_transpose(src, dst, elem_bytes, batches, rows, cols, src_pitch, src_batch, dst_pitch, dst_batch,
                            static_cast<cudaStream_t>(stream));
}

int spev_copy_segments_piece_bytes(void) { return 256 * 16 * 4; }

int spev_copy_segments(const void* src, void* dst, const int64_t* src_off, const int64_t* dst_off, const int64_t* nbytes,
                       const int64_t* piece_off, int n_segments, int64_t n_pieces, void* stream) {
    return launch_copy_segments(src, dst, src_off, dst_off, nbytes, piece_off, n_segments, n_pieces,
                                static_cast<cudaStream_t>(stream));
}

int spev_set_sm_limit(spev_ctx* c, int max_ctas) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "ctx is null");
    SPEV_REQUIRE(max_ctas >= 0, SPEV_E_INVALID, "spev_set_sm_limit: negative limit");
    c->num_sms = (max_ctas == 0 || max_ctas > c->num_sms_device) ? c->num_sms_device : max_ctas;
    return SPEV_OK;
}

int spev_lr_plan(const void* dur, int dur_dtype, int B, int T, int32_t* cumsum, int64_t* mel_lens,
                 int64_t* max_len_dev, int64_t* max_len_host, void* stream) {
    return launch_lr_plan(dur, dur_dtype, B, T, cumsum, mel_lens, max_len_dev, max_len_host,
                          static_cast<cudaStream_t>(stream));
}

int spev_lr_expand(const void* x, int64_t row_bytes, const int32_t* cumsum, int B, int T, void* out,
                   int64_t max_len, void* stream) {
    SPEV_REQUIRE(x && out, SPEV_E_INVALID, "spev_lr_expand: null x/out");
    return launch_lr_expand(x, row_bytes, nullptr, 0, nullptr, nullptr, cumsum, B, T, out, nullptr, max_len,
                            static_cast<cudaStream_t>(stream));
}

int spev_lr_expand_fused(const void* x, int64_t row_bytes, const float* feats, int n_feat,
                         const float* clamp_lo_host, const float* clamp_hi_host, const int32_t* cumsum,
                         int B, int T, void* out, float* feats_out, int64_t max_len, void* stream) {
    return launch_lr_expand(x, row_bytes, feats, n_feat, clamp_lo_host, clamp_hi_host, cumsum, B, T, out,
                            feats_out, max_len, static_cast<cudaStream_t>(stream));
}

int spev_pcm16_to_f32(const int16_t* pcm, int64_t n, float* out, void* stream) {
    return launch_pcm16_to_f32(pcm, n, out, static_cast<cudaStream_t>(stream));
}

int spev_variance_fuse(const float* x, const float* feats, int n_feat, const float* clamp_lo_host, const float* clamp_hi_host,
                       const float* conv_w, const float* conv_b, const int32_t* cumsum, int B, int T, int H, float* out,
                       float* feats_out, int64_t max_len, void* stream) {
    return launch_variance_fuse(x, feats, n_feat, clamp_lo_host, clamp_hi_host, conv_w, conv_b, cumsum, B, T, H, out,
                                feats_out, max_len, static_cast<cudaStream_t>(stream));
}

int spev_lr_expand_backward(const void* grad_out, int dtype, int H, const float* grad_feats_out, int n_feat,
                            const float* feats, const float* clamp_lo_host, const float* clamp_hi_host,
                            const int32_t* cumsum, int B, int T, int64_t max_len, void* grad_x, float* grad_feats,
                            void* stream) {
    return launch_lr_expand_backward(grad_out, dtype, H, grad_feats_out, n_feat, feats, clamp_lo_host, clamp_hi_host, cumsum,
                                     B, T, max_len, grad_x, grad_feats, static_cast<cudaStream_t>(stream));
}

size_t spev_variance_fuse_backward_workspace_bytes(int n_feat, int B, int H, int64_t max_len) {
    return variance_fuse_backward_workspace_bytes(n_feat, B, H, max_len);
}

int spev_variance_fuse_backward(const float* grad_out, const float* feats, int n_feat, const float* clamp_lo_host,
                                const float* clamp_hi_host, const float* conv_w, const int32_t* cumsum, int B, int T,
                                int H, int64_t max_len, float* grad_x, float* grad_feats, float* grad_w, float* grad_b,
                                void* workspace, size_t workspace_bytes, void* stream) {
    return launch_variance_fuse_backward(grad_out, feats, n_feat, clamp_lo_host, clamp_hi_host, conv_w, cumsum, B, T, H,
                                         max_len, grad_x, grad_feats, grad_w, grad_b, workspace, workspace_bytes,
                                         static_cast<cudaStream_t>(stream));
}

int spev_duration_rule(const float* log_dur, int64_t n, float d_control, int64_t* dur, void* stream) {
    return launch_duration_rule(log_dur, n, d_control, dur, static_cast<cudaStream_t>(stream));
}

int spev_bucketize_embed(const float* v, int64_t n, const float* boundaries, int n_boundaries, int right,
                         const float* table, int H, int64_t* idx_out, float* out, int accumulate, void* stream) {
    return launch_bucketize_embed(v, n, boundaries, n_boundaries, right, table, H, idx_out, out, accumulate,
                                  static_cast<cudaStream_t>(stream));
}

}  // extern "C"
