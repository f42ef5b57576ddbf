// features.cu -- frame-level energy / brightness features and per-phoneme pooling (SURVEY 8(f)
// "next" row 1; reference: /root/reference/spev_real_metrics.py:370-371 and :400-417).
//
// K9  k_frame_features : per frame t (hop 256) of the centre-padded 2048-sample window
//        rms[t]      = sqrt(mean(x^2))                       (librosa.feature.rms, :370)
//        centroid[t] = sum_k f_k |X_k| / sum_k |X_k|          (librosa.feature.spectral_centroid, :371)
//     with X = rFFT-2048(hann-2048 * x).  One warp per frame: the 2048 real samples are packed as
//     1024 complex points (z[n] = x[2n] + i x[2n+1]), transformed with the same 32x32 warp FFT as
//     the STFT kernels, and split with the w2048^k post-twiddle; the pair (k, 1024-k) comes from one
//     __shfl_sync (fetch_mirror).  Only two scalars per frame leave the SM.
// K10 k_segment_pool   : per phoneme p with duration d_p (frames): clip((mean(curve[seg_p]) - mu) /
//     sigma, lo, hi) -- the e / bri (and, with mu=1, sigma=-1, the br) lines of :400-417.  One warp
//     per utterance: warp-scan of the durations, then one lane per phoneme.  The mean covers the
//     phone's frames inside the item (numpy's slice); a phone with none gives NaN.  Negative
//     durations count as 0.
#include <algorithm>
#include <cmath>
#include "spev_internal.cuh"
#include "tile_pipe.cuh"

namespace spev {

constexpr int kFeatFft = 2048;
constexpr int kFeatStage = (kTileFrames - 1) * kHop + kFeatFft;   // 9984 samples per 32-frame tile

__global__ void __launch_bounds__(kThreads, 1)
k_frame_features(BatchView bv, const float* __restrict__ samples, float* __restrict__ rms_out,
                 float* __restrict__ cent_out, const float2* __restrict__ g_tw, const float2* __restrict__ g_win2,
                 const float2* __restrict__ g_tw2, float freq_step) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_tw = reinterpret_cast<float2*>(smem_raw);          // [1024] inter-stage twiddles
    float2* s_win2 = s_tw + 1024;                                // [1024] 0.5 * hann2048 as (w[2n], w[2n+1])
    float2* s_tw2 = s_win2 + 1024;                               // [512]  w2048^k
    spev_tile* s_ring = reinterpret_cast<spev_tile*>(s_tw2 + 512);
    float* s_stage = reinterpret_cast<float*>(s_ring + kRing);   // [9984]
    float* s_x = s_stage + kFeatStage;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) { s_tw[i] = g_tw[i]; s_win2[i] = g_win2[i]; }
    for (int i = threadIdx.x; i < 512; i += blockDim.x) s_tw2[i] = g_tw2[i];
    float2* xw = reinterpret_cast<float2*>(s_x + warp * kWarpRegionWords);

    const int stride = gridDim.x;
    const int my_n = ring_prologue(s_ring, bv.ftiles, bv.n_ftiles);
    for (int i = 0; i < my_n; ++i) {
        __syncthreads();   // previous tile done with the staging buffer; descriptor i visible
        const spev_tile d = s_ring[i & 3];
        if (i + 3 < my_n) fetch_desc(s_ring + ((i + 3) & 3), bv.ftiles + blockIdx.x + (i + 3) * stride);
        {   // stage [src0 - 512, +count): the 2048-window reaches 1024 samples left of the frame centre
            const int count = (d.n - 1) * kHop + kFeatFft;
            const int64_t first = d.src0 - 512;
            const int i_lo = static_cast<int>(max(static_cast<int64_t>(0), d.lo - first));
            const int i_hi = static_cast<int>(min(static_cast<int64_t>(count), d.hi - first));
            const float* xs = samples + first;
            const bool vec_ok = ((reinterpret_cast<uintptr_t>(samples) & 15) == 0) && ((d.lo & 3) == 0);
            if (vec_ok) {
                for (int j = threadIdx.x * 4; j < count; j += blockDim.x * 4) {
                    int nb = j >= i_lo ? (i_hi - j) * 4 : 0;
                    nb = max(0, min(16, nb));
                    cp_async16(s_stage + j, nb > 0 ? xs + j : samples, nb);
                }
            } else {
                for (int j = threadIdx.x; j < count; j += blockDim.x) {
                    const bool ok = j >= i_lo && j < i_hi;
                    cp_async4(s_stage + j, ok ? xs + j : samples, ok ? 4 : 0);
                }
            }
        }
        cp_async_commit();
        cp_async_wait_all();
        __syncthreads();
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            const int f = 2 * warp + r;
            if (f >= d.n) break;
            const float2* px = reinterpret_cast<const float2*>(s_stage + f * kHop) + lane;
            float2 v[32];
            float sumsq = 0.f;
            static_for<0, 32>([&](auto jc) {
                constexpr int j = decltype(jc)::value;
                const float2 x = px[32 * j];
                const float2 w = s_win2[32 * j + lane];
                sumsq = fmaf(x.x, x.x, sumsq);
                sumsq = fmaf(x.y, x.y, sumsq);
                v[j] = make_float2(w.x * x.x, w.y * x.y);
            });
            warp_fft1024<-1>(v, xw, s_tw, lane);
            float2 p[16];
            fetch_mirror(v, p, lane);
            float s_mag = 0.f, s_fmag = 0.f;
            static_for<0, 16>([&](auto kc) {
                constexpr int k2 = decltype(kc)::value;
                const int k = lane + 32 * k2;
                const float2 z = v[k2], zm = p[k2];
                const float er = z.x + zm.x, ei = z.y - zm.y;          // E = Z + conj(Zm)   (1/2 folded into the window)
                const float or_ = z.x - zm.x, oi = z.y + zm.y;         // O = Z - conj(Zm)
                const float2 w = s_tw2[k];                             // w2048^k
                const float tr = fmaf(w.x, or_, -w.y * oi), ti = fmaf(w.x, oi, w.y * or_);   // T = w * O
                const float ar = er + ti, ai = ei - tr;                // X[k]      = E - iT
                const float br = er - ti, bi = ei + tr;                // X[1024-k] = conj(E) - i conj(T)  (same modulus as (br, bi))
                const float m1 = sqrtf(fmaf(ar, ar, ai * ai));
                const float m2 = sqrtf(fmaf(br, br, bi * bi));
                s_mag += m1 + m2;
                s_fmag = fmaf(static_cast<float>(k), m1, s_fmag);
                s_fmag = fmaf(static_cast<float>(1024 - k), m2, s_fmag);
            });
            if (lane == 0) {   // bin 512 pairs with itself: |X[512]| = |Z[512]|  (window carries 1/2 -> x2)
                const float m = 2.f * sqrtf(fmaf(v[16].x, v[16].x, v[16].y * v[16].y));
                s_mag += m;
                s_fmag = fmaf(512.f, m, s_fmag);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s_mag += __shfl_xor_sync(0xffffffffu, s_mag, o);
                s_fmag += __shfl_xor_sync(0xffffffffu, s_fmag, o);
                sumsq += __shfl_xor_sync(0xffffffffu, sumsq, o);
            }
            if (lane == 0) {
                const int64_t row = d.row0 + f;
                rms_out[row] = sqrtf(sumsq * (1.0f / kFeatFft));
                // librosa.util.normalize(norm=1): columns whose l1 norm is below tiny are left unscaled
                const float len = s_mag < kTiny ? 1.0f : s_mag;
                cent_out[row] = freq_step * s_fmag / len;
            }
            __syncwarp();
        }
    }
}

// ---- per-phoneme pooling -----------------------------------------------------------------------
// LOG: pool log(curve + log_eps) instead of the curve itself (the reference takes the log of rms / centroid per
// frame before the per-phone mean, spev_real_metrics.py:370, :397)
template <bool LOG>
__global__ void k_segment_pool(const float* __restrict__ curve, const int64_t* __restrict__ frame_off,
                               const long long* __restrict__ durs, const int64_t* __restrict__ phone_off, int U,
                               float mu, float sigma, float lo, float hi, float log_eps, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    for (int u = blockIdx.x * wpb + (threadIdx.x >> 5); u < U; u += gridDim.x * wpb) {
        const int64_t p0 = phone_off[u], p1 = phone_off[u + 1];
        const float* c = curve + frame_off[u];
        const int64_t T = frame_off[u + 1] - frame_off[u];
        long long carry = 0;
        for (int64_t pb = p0; pb < p1; pb += 32) {
            const int64_t p = pb + lane;
            long long dd = p < p1 ? durs[p] : 0;
            if (dd < 0) dd = 0;
            long long incl = dd;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const long long start = carry + incl - dd;
            if (p < p1) {
                float acc = 0.f;
                const long long end = min(static_cast<long long>(T), start + dd);
                const long long n = max(0LL, end - start);   // frames of the phone inside the item
                for (long long t = start; t < end; ++t) acc += LOG ? logf(c[t] + log_eps) : c[t];
                // numpy: the mean of a slice cut at the item's end; the mean of an empty slice is NaN
                const float m = n > 0 ? acc / static_cast<float>(n) : __int_as_float(0x7fc00000);
                // np.clip propagates the NaN of an empty phone; fminf/fmaxf would swallow it
                out[p] = n > 0 ? fminf(fmaxf((m - mu) / sigma, lo), hi) : m;
            }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

// ---- host side ---------------------------------------------------------------------------------
// 0.5 * periodic Hann-2048 as (w[2n], w[2n+1]) pairs and the post-twiddles w2048^k, float64 -> float32
int features_init(spev_ctx* c) {
    std::vector<float2> win2048(1024), tw2048(512);
    for (int n = 0; n < 1024; ++n) {
        const double w0 = 0.5 - 0.5 * std::cos(2.0 * M_PI * (2 * n) / 2048.0), w1 = 0.5 - 0.5 * std::cos(2.0 * M_PI * (2 * n + 1) / 2048.0);
        win2048[n] = make_float2(0.5f * static_cast<float>(w0), 0.5f * static_cast<float>(w1));
    }
    for (int k = 0; k < 512; ++k) {
        const double a = -2.0 * M_PI * k / 2048.0;
        tw2048[k] = make_float2(static_cast<float>(std::cos(a)), static_cast<float>(std::sin(a)));
    }
    int rc = upload(&c->d_win2048, win2048);
    return rc ? rc : upload(&c->d_tw2048, tw2048);
}

template <bool LOG>
static int segment_pool(const float* curve, const int64_t* frame_off, const int64_t* durs, const int64_t* phone_off,
                        int U, float mu, float sigma, float lo, float hi, float log_eps, float* out, cudaStream_t st) {
    SPEV_REQUIRE(U >= 0, SPEV_E_INVALID, "segment_pool: U < 0");
    if (U == 0) return SPEV_OK;
    SPEV_REQUIRE(curve && frame_off && durs && phone_off && out, SPEV_E_INVALID, "segment_pool: null buffer");
    SPEV_REQUIRE(sigma != 0.f, SPEV_E_INVALID, "segment_pool: sigma == 0");
    const int wpb = 4;
    const int grid = std::min((U + wpb - 1) / wpb, 148 * 16);
    k_segment_pool<LOG><<<grid, wpb * 32, 0, st>>>(curve, frame_off, reinterpret_cast<const long long*>(durs), phone_off,
                                                   U, mu, sigma, lo, hi, log_eps, out);
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

}  // namespace spev

using namespace spev;

extern "C" {

int spev_frame_features(spev_ctx* c, const spev_batch* b, const float* samples, float* rms, float* centroid, void* stream) {
    SPEV_ON_CTX_DEVICE(c);
    SPEV_REQUIRE(b, SPEV_E_INVALID, "null ctx or batch");
    if (b->n_ftiles == 0) return SPEV_OK;
    SPEV_REQUIRE(samples && rms && centroid && b->ftiles, SPEV_E_INVALID, "frame_features: null buffer");
    const size_t smem = sizeof(float2) * (1024 + 1024 + 512) + sizeof(spev_tile) * kRing + sizeof(float) * kFeatStage +
                        sizeof(float) * kWarps * kWarpRegionWords;
    SPEV_CUDA(cudaFuncSetAttribute(k_frame_features, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int grid = std::min<int64_t>(b->n_ftiles, c->num_sms);
    k_frame_features<<<grid, kThreads, smem, static_cast<cudaStream_t>(stream)>>>(
        view_of(b), samples, rms, centroid, c->d_tw, c->d_win2048, c->d_tw2048, static_cast<float>(static_cast<double>(c->sr) / kFeatFft));
    SPEV_CUDA(cudaGetLastError());
    return SPEV_OK;
}

int spev_segment_pool(const float* curve, const int64_t* frame_off, const int64_t* durs, const int64_t* phone_off,
                      int n_items, float mu, float sigma, float lo, float hi, float* out, void* stream) {
    return segment_pool<false>(curve, frame_off, durs, phone_off, n_items, mu, sigma, lo, hi, 0.f, out,
                               static_cast<cudaStream_t>(stream));
}

int spev_segment_pool_log(const float* curve, float log_eps, const int64_t* frame_off, const int64_t* durs,
                          const int64_t* phone_off, int n_items, float mu, float sigma, float lo, float hi, float* out,
                          void* stream) {
    return segment_pool<true>(curve, frame_off, durs, phone_off, n_items, mu, sigma, lo, hi, log_eps, out,
                              static_cast<cudaStream_t>(stream));
}

}  // extern "C"
