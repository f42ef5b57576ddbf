// abi.cu -- ctx construction, host constants and tile planners of the C ABI (include/spev_b200.h); every other
// entry point is defined beside its kernels.
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

    spev_ctx* c = new spev_ctx();   // value-initialised: every device pointer starts out null
    c->device = device; c->sr = sr; c->n_fft = n_fft; c->hop = hop; c->win = kNfft; c->n_mels = n_mels;
    c->fmin = fmin; c->fmax = fmax; c->num_sms = c->num_sms_device = prop.multiProcessorCount; c->use_tc = 1;

    // periodic Hann, float64 -> float32
    c->h_window.resize(kNfft);
    for (int i = 0; i < kNfft; ++i) c->h_window[i] = static_cast<float>(0.5 - 0.5 * std::cos(2.0 * M_PI * i / kNfft));
    std::vector<float2> tw(1024);
    for (int k1 = 0; k1 < 32; ++k1)
        for (int l = 0; l < 32; ++l) {
            const double a = -2.0 * M_PI * (k1 * l) / 1024.0;
            tw[k1 * 32 + l] = make_float2(static_cast<float>(std::cos(a)), static_cast<float>(std::sin(a)));
        }
    build_mel_basis(sr, n_fft, n_mels, fmin, fmax, c->h_basis);
    pinv_jacobi(c->h_basis, n_mels, kBins, c->h_pinv);
    int rc = SPEV_OK;
    if ((rc = upload(&c->d_tw, tw)) || (rc = spectral_init(c)) || (rc = gemm_tc_init(c)) || (rc = nnls_init(c)) ||
        (rc = features_init(c))) {
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
    cudaFree(c->d_tw); cudaFree(c->d_window); cudaFree(c->d_win2048); cudaFree(c->d_tw2048); cudaFree(c->d_basis); cudaFree(c->d_nnls_rng); cudaFree(c->d_basis_hi);
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

int spev_set_sm_limit(spev_ctx* c, int max_ctas) {
    SPEV_REQUIRE(c, SPEV_E_INVALID, "ctx is null");
    SPEV_REQUIRE(max_ctas >= 0, SPEV_E_INVALID, "spev_set_sm_limit: negative limit");
    c->num_sms = (max_ctas == 0 || max_ctas > c->num_sms_device) ? c->num_sms_device : max_ctas;
    return SPEV_OK;
}

}  // extern "C"
